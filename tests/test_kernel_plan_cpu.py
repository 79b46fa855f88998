"""The build check (imx_jit_compile_check) plans a specialisation as a handle does, switches included, without a GPU.

A handle and the check derive the kernel plan in one function, so the check compiles the module a handle with the same
config and switches loads: with IMX_PIPE=0 that module has no pipelined kernel, and IMX_PIPE_STAGES sets its ring depth."""
import ctypes
import os

import pytest

from marl_for_im_b200 import _lib, presets
from marl_for_im_b200.envs import ENV_CLASSES


def _config(kind="MAIM", preset="serial4", n=65536):
    return ENV_CLASSES[kind](dict(presets.PRESETS[preset](), num_envs=n, _config_only=True)).imx_config


def _check(c, variant):
    lib = _lib.load()
    buf = ctypes.create_string_buffer(8192)
    n = lib.imx_jit_compile_check(ctypes.byref(c), variant, buf, 8192)
    assert n > 10000, (variant, n, buf.value.decode()[:500], lib.imx_last_error())


def _cubin(c, variant, path, monkeypatch):
    monkeypatch.setenv("IMX_JIT_DUMP", str(path))
    _check(c, variant)
    monkeypatch.delenv("IMX_JIT_DUMP")
    return path.read_bytes()


@pytest.mark.parametrize("variant", [0, 1, 2])
def test_pipe_off_builds_no_pipelined_kernel(variant, tmp_path, monkeypatch):
    monkeypatch.setenv("IMX_JIT_CACHE", "0")
    c = _config()
    assert b"step_kernel_pipe" in _cubin(c, variant, tmp_path / "default.cubin", monkeypatch)
    monkeypatch.setenv("IMX_PIPE", "0")
    cubin = _cubin(c, variant, tmp_path / "pipe0.cubin", monkeypatch)
    assert b"step_kernel_pipe" not in cubin
    assert b"step_kernel_tma" in cubin


def test_pipe_stages_switch_changes_the_specialisation(tmp_path, monkeypatch):
    """serial4's default ring has four stages: IMX_PIPE_STAGES=4 hits the default's cache entry, 2 builds another one."""
    monkeypatch.setenv("IMX_CACHE_DIR", str(tmp_path))
    c = _config()
    files = lambda: {f for f in os.listdir(tmp_path) if f.endswith("_sm100a.cubin")}  # noqa: E731
    _check(c, 0)
    default = files()
    assert len(default) == 1
    monkeypatch.setenv("IMX_PIPE_STAGES", "4")
    _check(c, 0)
    assert files() == default
    monkeypatch.setenv("IMX_PIPE_STAGES", "2")
    _check(c, 0)
    assert len(files() - default) == 1
