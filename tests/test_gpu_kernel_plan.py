"""The build check (imx_jit_compile_check) compiles exactly the specialisations a handle loads: after a handle has built every
module it can use into a fresh cubin cache, checking each of those variants adds no file to the cache.  The check assumes the
B200's 126 MB L2 while a handle reads the device's, so the batch (65 536 envs) sits far from the L2-priority thresholds."""
import ctypes
import os
import subprocess
import sys

import pytest

from marl_for_im_b200 import _lib, presets
from marl_for_im_b200.envs import ENV_CLASSES

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = 65536
ALL_MODULES = 1 | 2 | 4 | 8 | 16 | _lib.PREPARE_EPISODE

# a new process: the library's in-memory module cache would otherwise serve a specialisation an earlier test loaded,
# without touching the fresh disk cache
CREATE = """
import ctypes, sys
sys.path.insert(0, {root!r})
from marl_for_im_b200 import _lib, presets
from marl_for_im_b200.envs import ENV_CLASSES
lib = _lib.load()
c = ENV_CLASSES[{kind!r}](dict(presets.PRESETS[{preset!r}](), num_envs={n}, _config_only=True)).imx_config
h = ctypes.c_void_p()
_lib.check(lib.imx_create(ctypes.byref(c), ctypes.byref(h)))
_lib.check(lib.imx_prepare(h, {flags}))
_lib.check(lib.imx_destroy(h))
"""


def _cubins(d):
    return {f for f in os.listdir(d) if f.endswith("_sm100a.cubin")}


@pytest.mark.parametrize("switch", [None, ("IMX_PIPE", "0"), ("IMX_PIPE_STAGES", "2")], ids=["default", "pipe0", "stages2"])
@pytest.mark.parametrize("kind,preset", [("MAIM", "serial4"), ("MAIM_div", "div1"), ("MAIM_div", "div2")])
def test_check_builds_what_a_handle_loads(kind, preset, switch, tmp_path, monkeypatch):
    monkeypatch.setenv("IMX_CACHE_DIR", str(tmp_path))
    monkeypatch.setenv("IMX_JIT", "1")
    if switch:
        monkeypatch.setenv(*switch)
    code = CREATE.format(root=ROOT, kind=kind, preset=preset, n=N, flags=ALL_MODULES)
    subprocess.run([sys.executable, "-c", code], check=True, env=dict(os.environ))
    loaded = _cubins(tmp_path)
    assert len(loaded) == 5, sorted(loaded)            # step, no observations, critic rows, episode with and without observations
    c = ENV_CLASSES[kind](dict(presets.PRESETS[preset](), num_envs=N, _config_only=True)).imx_config
    lib = _lib.load()
    for variant in range(5):
        buf = ctypes.create_string_buffer(4096)
        rc = lib.imx_jit_compile_check(ctypes.byref(c), variant, buf, 4096)
        assert rc > 0, (variant, rc, lib.imx_last_error())
        assert _cubins(tmp_path) == loaded, (variant, sorted(_cubins(tmp_path) - loaded))
