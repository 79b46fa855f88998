"""imx_replay_episode without a GPU: the episode kernel (with and without observations) builds for sm_100a through the
runtime specialisation for every network family and observation mode, and the header / binding expose the new call."""
import ctypes
import os
import re

import pytest

from marl_for_im_b200 import _lib, presets
from marl_for_im_b200.envs import ENV_CLASSES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CASES = {
    "serial2_cc5": ("MAIM", presets.serial2(), {}),
    "serial4": ("MAIM", presets.serial4(), {}),
    "serial8": ("IM", presets.serial8(), {}),
    "div1": ("IM_div", presets.div1(), {}),
    "div2": ("MAIM_div", presets.div2(), {}),
    "serial4_obs_f32": ("MAIM", presets.serial4(), {"obs_dtype": "float32"}),
    "serial8_noisy_delay": ("MAIM", presets.serial8(), {"noisy_delay": True, "noisy_delay_threshold": 0.3}),
    "div2_noisy_delay_and_demand": ("MAIM_div", presets.div2(), {"noisy_delay": True, "noisy_delay_threshold": 0.3,
                                                                  "noisy_demand": True, "noisy_demand_threshold": 0.1}),
}


def _config(kind, cfg, extra, n=65536):
    return ENV_CLASSES[kind](dict(cfg, num_envs=n, _config_only=True, **extra)).imx_config


@pytest.mark.parametrize("variant", [3, 4])
@pytest.mark.parametrize("case", sorted(CASES))
def test_episode_kernel_compiles_for_sm100a(case, variant):
    kind, cfg, extra = CASES[case]
    c = _config(kind, cfg, extra)
    if extra.get("noisy_delay"):
        c.noisy_delay = 1                    # the handle a noisy episode runs on carries the delayed goods
    lib = _lib.load()
    buf = ctypes.create_string_buffer(8192)
    n = lib.imx_jit_compile_check(ctypes.byref(c), variant, buf, 8192)
    assert n > 10000, (case, variant, n, buf.value.decode()[:600], lib.imx_last_error())


def test_episode_layout_beyond_shared_memory_is_refused_not_compiled():
    """A trace that cannot be resident (here 4000 periods of a divergent network) has no episode kernel: the call falls back
    to the composition, and the build check says why instead of compiling."""
    c = _config("MAIM_div", dict(presets.div2(), num_periods=4000), {})
    lib = _lib.load()
    buf = ctypes.create_string_buffer(1024)
    assert lib.imx_jit_compile_check(ctypes.byref(c), 3, buf, 1024) < 0
    assert b"200 KB" in lib.imx_last_error()


def test_header_declares_the_episode_call_and_prepare_flag():
    header = open(os.path.join(ROOT, "include", "imx_b200.h")).read()
    assert re.search(r"int imx_replay_episode\(imx_env\* env, const int32_t\* demand_dev, const uint8_t\* delay_mask_dev, int noisy, "
                     r"uint64_t episode,\s+const double\* actions_dev, void\* obs_dev, double\* reward_dev, double\* return_dev,\s+"
                     r"double\* stats_dev, int accumulate, double\* eval_acc_dev, void\* stream\);", header)
    assert re.search(r"IMX_PREPARE_EPISODE = 32\b", header)
    assert "#define IMX_ABI_VERSION 3 " in header


def test_binding_exposes_the_episode_call():
    lib = _lib.load()
    fn = lib.imx_replay_episode
    assert fn.restype is ctypes.c_int and len(fn.argtypes) == 13
    assert _lib.PREPARE_EPISODE == 32
    for cls in ENV_CLASSES.values():
        assert callable(getattr(cls, "replay_episode"))
