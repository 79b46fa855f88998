"""imx_replay_episode_records without a GPU: the episode kernel with records (variants 5 and 6 of imx_jit_compile_check)
builds for sm_100a for every network preset and observation type; it holds the records' bulk stores and the modules
without records do not; the header and the binding expose the call, the struct and the prepare flag."""
import ctypes
import os
import re
import subprocess

import pytest

from marl_for_im_b200 import _lib, presets
from marl_for_im_b200.envs import ENV_CLASSES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PRESETS = {"serial2": ("MAIM", presets.serial2), "serial4": ("MAIM", presets.serial4), "serial8": ("IM", presets.serial8),
           "div1": ("IM_div", presets.div1), "div2": ("MAIM_div", presets.div2)}
OBS = {"float64": {}, "float32": {"obs_dtype": "float32"}, "bfloat16": {"obs_dtype": "bfloat16", "action_dtype": "float32"}}


def _config(kind, cfg, extra, n=65536):
    return ENV_CLASSES[kind](dict(cfg, num_envs=n, _config_only=True, **extra)).imx_config


def _compile(c, variant, path=None, monkeypatch=None):
    if path is not None:
        monkeypatch.setenv("IMX_JIT_DUMP", str(path))
    buf = ctypes.create_string_buffer(1 << 14)
    n = _lib.load().imx_jit_compile_check(ctypes.byref(c), variant, buf, 1 << 14)
    assert n > 10000, (variant, n, buf.value.decode()[:600], _lib.load().imx_last_error())
    return n


@pytest.mark.parametrize("variant", [5, 6])
@pytest.mark.parametrize("obs", sorted(OBS))
@pytest.mark.parametrize("preset", sorted(PRESETS))
def test_records_kernel_compiles_for_sm100a(preset, obs, variant):
    kind, cfg = PRESETS[preset]
    _compile(_config(kind, cfg(), OBS[obs]), variant)


def test_records_kernel_with_noisy_delays_compiles():
    c = _config("MAIM_div", presets.div2(), {"noisy_delay": True, "noisy_delay_threshold": 0.3})
    c.noisy_delay = 1
    for variant in (5, 6):
        _compile(c, variant)


def _bulk_stores(cubin):
    sass = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", str(cubin)], capture_output=True, text=True, check=True).stdout
    return len(re.findall(r"\bUBLKCP\.G\.S\b", sass))


@pytest.mark.skipif(not os.path.exists("/usr/local/cuda/bin/cuobjdump"), reason="needs cuobjdump")
def test_records_add_bulk_stores_only_to_the_records_module(tmp_path, monkeypatch):
    """The records module has the record stores (row 0 of three state fields, five per-period fields, three state rows);
    the episode module without records is the build it was (the flag is a literal, not a uniform branch)."""
    monkeypatch.setenv("IMX_CACHE_DIR", str(tmp_path / "cache"))
    c = _config("MAIM", presets.serial4(), {})
    counts = {}
    for variant in (3, 5):
        path = tmp_path / f"v{variant}.cubin"
        _compile(c, variant, path, monkeypatch)
        counts[variant] = _bulk_stores(path)
    assert counts[5] >= counts[3] + 11, counts


def test_records_layout_beyond_shared_memory_is_refused_not_compiled():
    c = _config("MAIM_div", dict(presets.div2(), num_periods=4000), {})
    buf = ctypes.create_string_buffer(1024)
    assert _lib.load().imx_jit_compile_check(ctypes.byref(c), 5, buf, 1024) < 0
    assert b"200 KB" in _lib.load().imx_last_error()
    assert _lib.load().imx_jit_compile_check(ctypes.byref(c), 7, buf, 1024) < 0


def test_header_and_binding_expose_the_records_call():
    header = open(os.path.join(ROOT, "include", "imx_b200.h")).read()
    assert re.search(r"int imx_replay_episode_records\(imx_env\* env, const int32_t\* demand_dev, const uint8_t\* delay_mask_dev, "
                     r"int noisy, uint64_t episode,\s+const double\* actions_dev, void\* obs_dev, double\* reward_dev, "
                     r"double\* return_dev,\s+double\* stats_dev, int accumulate, double\* eval_acc_dev, "
                     r"const imx_records_out\* records,\s+void\* stream\);", header)
    assert re.search(r"IMX_PREPARE_RECORDS = 64\b", header)
    fields = re.search(r"typedef struct imx_records_out \{(.*?)\} imx_records_out;", header, re.S).group(1)
    names = re.findall(r"\*\s*(\w+_dev);", fields)
    assert names == [f for f, _ in _lib.ImxRecordsOut._fields_]
    lib = _lib.load()
    fn = lib.imx_replay_episode_records
    assert fn.restype is ctypes.c_int and len(fn.argtypes) == 14
    assert _lib.PREPARE_RECORDS == 64 and ctypes.sizeof(_lib.ImxRecordsOut) == 64
    assert set(ENV_CLASSES["MAIM"].RECORD_FIELDS) == {"inv", "backlog", "order_u", "demand", "ship", "acquisition", "order_r", "profit"}
