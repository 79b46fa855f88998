"""imx_step_eval without a GPU: its modules (variants 8 and 9 of imx_jit_compile_check) build for sm_100a for every network
preset, kind and observation type; their step kernels use no local memory; they hold only the one-period kernels; the header and
the binding expose the call and the prepare flag."""
import ctypes
import os
import re
import subprocess

import pytest

from marl_for_im_b200 import _lib, presets
from marl_for_im_b200.envs import ENV_CLASSES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"

KINDS = {"serial2": ("IM", "MAIM"), "serial4": ("IM", "MAIM"), "serial4_dfo": ("IM",), "serial8": ("IM", "MAIM"),
         "div1": ("IM_div", "MAIM_div"), "div2": ("IM_div", "MAIM_div")}
OBS = {"float64": {}, "float32": {"obs_dtype": "float32", "action_dtype": "float32"},
       "bfloat16": {"obs_dtype": "bfloat16", "action_dtype": "float32"}}


def _config(kind, cfg, extra, n=65536):
    return ENV_CLASSES[kind](dict(cfg, num_envs=n, _config_only=True, **extra)).imx_config


def _compile(c, variant, path=None, monkeypatch=None):
    if path is not None:
        monkeypatch.setenv("IMX_JIT_DUMP", str(path))
    buf = ctypes.create_string_buffer(1 << 14)
    n = _lib.load().imx_jit_compile_check(ctypes.byref(c), variant, buf, 1 << 14)
    assert n > 10000, (variant, n, buf.value.decode()[:600], _lib.load().imx_last_error())
    return n


@pytest.mark.parametrize("variant", [8, 9])
@pytest.mark.parametrize("obs", sorted(OBS))
@pytest.mark.parametrize("preset,kind", [(p, k) for p in sorted(KINDS) for k in KINDS[p]])
def test_step_eval_modules_compile_for_sm100a(preset, kind, obs, variant):
    _compile(_config(kind, presets.PRESETS[preset](), OBS[obs]), variant)


@pytest.mark.parametrize("switch", [{"IMX_STEP_ET": "0"}, {"IMX_STEP_ET": "1"}, {"IMX_L2_HINTS": "1"}, {"IMX_PIPE": "0"}])
def test_step_eval_modules_compile_under_the_tuning_switches(switch, monkeypatch):
    for k, v in switch.items():
        monkeypatch.setenv(k, v)
    c = _config("MAIM_div", presets.div2(), {"noisy_delay": True, "noisy_delay_threshold": 0.3})
    c.noisy_delay = 1
    for variant in (8, 9):
        _compile(c, variant)


def _sass(cubin):
    return subprocess.run([CUOBJDUMP, "-sass", str(cubin)], capture_output=True, text=True, check=True).stdout


def _res_usage(cubin):
    out = subprocess.run([CUOBJDUMP, "-res-usage", str(cubin)], capture_output=True, text=True, check=True).stdout
    return re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", out)


@pytest.mark.skipif(not os.path.exists(CUOBJDUMP), reason="needs cuobjdump")
@pytest.mark.parametrize("kind,preset", [("MAIM", "serial4"), ("IM", "serial8"), ("IM_div", "div1"), ("MAIM_div", "div2")])
def test_step_eval_modules_hold_only_the_step_kernels_and_use_no_local_memory(kind, preset, tmp_path, monkeypatch):
    monkeypatch.setenv("IMX_CACHE_DIR", str(tmp_path / "cache"))
    c = _config(kind, presets.PRESETS[preset](), {})
    for variant in (8, 9):
        path = tmp_path / f"v{variant}.cubin"
        _compile(c, variant, path, monkeypatch)
        funcs = _res_usage(path)
        names = sorted(f for f, _, _, _ in funcs)
        assert names and all("step_kernel_tma" in f or "step_kernel_pipe" in f for f in names), names
        assert not any("many" in f or "episode" in f or "rollout" in f for f in names), names
        for f, _, _, local in funcs:                          # (a small call-stack frame, as the plain divergent kernels have, is not a spill)
            assert int(local) == 0, (variant, f, local)


@pytest.mark.skipif(not os.path.exists(CUOBJDUMP), reason="needs cuobjdump")
def test_step_eval_adds_bulk_copies_only_to_its_modules(tmp_path, monkeypatch):
    """The bookkeeping tiles move by bulk copy (returns, accumulators, five diagnostics); the plain step module is the build
    it was (the flag is a literal, not a uniform branch)."""
    monkeypatch.setenv("IMX_CACHE_DIR", str(tmp_path / "cache"))
    c = _config("MAIM", presets.serial4(), {})
    counts = {}
    for variant in (0, 8):
        path = tmp_path / f"v{variant}.cubin"
        _compile(c, variant, path, monkeypatch)
        counts[variant] = len(re.findall(r"\bUBLKCP\.G\.S\b", _sass(path)))
    assert counts[8] >= counts[0] + 7, counts


@pytest.mark.parametrize("variant", [-1, 7, 10])
def test_unassigned_variant_numbers_are_refused(variant):
    """Variants 8 / 9 are imx_step_eval's modules; 7 is not assigned and, like any number past the table, is refused."""
    c = _config("MAIM", presets.serial4(), {})
    buf = ctypes.create_string_buffer(1024)
    assert _lib.load().imx_jit_compile_check(ctypes.byref(c), variant, buf, 1024) < 0
    assert b"variant must be" in _lib.load().imx_last_error()


def test_header_and_binding_expose_step_eval():
    header = open(os.path.join(ROOT, "include", "imx_b200.h")).read()
    assert re.search(r"int imx_step_eval\(imx_env\* env, const void\* actions_dev, void\* obs_dev, double\* reward_dev, "
                     r"const imx_info_out\* info,\s+double\* return_dev, double\* eval_acc_dev, void\* stream\);", header)
    assert re.search(r"IMX_PREPARE_EVAL = 128\b", header)
    assert re.search(r"#define IMX_ABI_VERSION 3\b", header)
    fn = _lib.load().imx_step_eval
    assert fn.restype is ctypes.c_int and len(fn.argtypes) == 8
    assert _lib.PREPARE_EVAL == 128
    assert list(ENV_CLASSES["MAIM"].INFO_FIELDS) == ["demand", "ship", "acquisition", "actual order", "profit"]
