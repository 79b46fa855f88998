"""bfloat16 observations and float32 actions (``imx_config.io_flags``) without a GPU: the specialised kernels build for sm_100a
with the new element types, the float64 / float32 specialisations keep their register and spill counts, the config is
validated, and the host's float32 -> bfloat16 rounding (the bfloat16 copy of the rescale tables) is torch's, bit for bit."""
import ctypes
import json
import os
import re
import shutil
import struct
import subprocess

import numpy as np
import pytest
import torch

from marl_for_im_b200 import _lib, presets
from marl_for_im_b200.envs import ENV_CLASSES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"

# the network families of the shipped configs: serial2 in CC_5 mode, serial4, serial8 (64-byte float64 rows), div1, div2
CASES = {"serial2_cc5": ("MAIM", "serial2"), "serial4": ("MAIM", "serial4"), "serial8": ("IM", "serial8"),
         "div1": ("IM_div", "div1"), "div2": ("MAIM_div", "div2")}
FLAGS = {"obs_bf16": _lib.IO_OBS_BF16, "act_f32": _lib.IO_ACTIONS_F32, "both": _lib.IO_OBS_BF16 | _lib.IO_ACTIONS_F32}


def _config(case, obs_dtype="float64", io_flags=0):
    kind, preset = CASES[case]
    c = ENV_CLASSES[kind](dict(presets.PRESETS[preset](), num_envs=65536, obs_dtype=obs_dtype, _config_only=True)).imx_config
    c.io_flags = io_flags
    return c


def _compile(c, variant, tmp_path, name="k.cubin"):
    """cubin of one specialisation (the on-disk cache is bypassed so the cubin is this build's)."""
    path = str(tmp_path / name)
    os.environ["IMX_JIT_DUMP"] = path
    try:
        buf = ctypes.create_string_buffer(1 << 14)
        n = _lib.load().imx_jit_compile_check(ctypes.byref(c), variant, buf, 1 << 14)
    finally:
        del os.environ["IMX_JIT_DUMP"]
    assert n > 10000, (variant, n, buf.value.decode()[:500], _lib.load().imx_last_error())
    return path


def _variants(case):
    return (0, 1, 2, 3, 4) if CASES[case][0].startswith("MAIM") else (0, 1, 3, 4)


@pytest.mark.parametrize("flags", sorted(FLAGS))
@pytest.mark.parametrize("case", sorted(CASES))
def test_new_specialisations_compile_for_sm100a(case, flags, tmp_path, monkeypatch):
    monkeypatch.setenv("IMX_JIT_CACHE", "0")
    for variant in _variants(case):
        _compile(_config(case, io_flags=FLAGS[flags]), variant, tmp_path)


def _res_usage(path):
    out = subprocess.run([CUOBJDUMP, "-res-usage", path], capture_output=True, text=True, check=True).stdout
    res, fn = {}, None
    for line in out.splitlines():
        m = re.search(r"Function ([^:]+):", line)
        if m:
            fn = m.group(1)
            continue
        m = re.search(r"REG:(\d+) STACK:\d+ SHARED:\d+ LOCAL:(\d+)", line)
        if m and fn:
            res[fn] = [int(m.group(1)), int(m.group(2))]
    return res


@pytest.mark.parametrize("case", sorted(CASES))
def test_existing_specialisations_keep_their_registers_and_spills(case, tmp_path, monkeypatch):
    """The float64 and float32 observation kernels fold the new element-type branches away: per kernel, the register count
    and the local-memory (spill) bytes equal those of the build before the element types became a code."""
    monkeypatch.setenv("IMX_JIT_CACHE", "0")
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "jit_res_usage.json")))
    for obs in ("float64", "float32"):
        for variant in _variants(case):
            got = _res_usage(_compile(_config(case, obs), variant, tmp_path))
            assert got == golden[f"{case}|{obs}|{variant}"], (case, obs, variant)


def _pipe_sass(c, tmp_path):
    path = _compile(c, 0, tmp_path)
    sass = subprocess.run([CUOBJDUMP, "-sass", path], capture_output=True, text=True, check=True).stdout
    for f in re.split(r"\n\s+Function : ", sass)[1:]:
        if f.startswith("_ZN3imx16step_kernel_pipe"):
            return re.findall(r"/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\w+\s+)?([A-Z0-9_.]+)", f)
    raise AssertionError("no pipelined kernel in the module")


@pytest.mark.parametrize("flags", ["obs_bf16", "both"])
def test_pipelined_kernel_loads_the_bf16_table_and_converts_no_observation(flags, tmp_path, monkeypatch):
    """Config 2's pipelined kernel stores bfloat16 observations as 2-byte table loads (LDG.E.U16): no float64 -> float32
    conversion and no bfloat16 packing on the observation path (the only F2F left is float32 actions widened to float64)."""
    monkeypatch.setenv("IMX_JIT_CACHE", "0")
    ops = _pipe_sass(_config("serial4", io_flags=FLAGS[flags]), tmp_path)
    assert "LDG.E.U16.CONSTANT" in ops
    assert not [o for o in ops if o.startswith("F2F.F32.F64") or o.startswith("F2FP")], sorted(set(ops))
    widen = [o for o in ops if o.startswith("F2F")]
    assert all(o == "F2F.F64.F32" for o in widen) and (bool(widen) == (flags == "both"))


def test_config_layout_and_validation():
    lib = _lib.load()
    assert lib.imx_config_size() == ctypes.sizeof(_lib.ImxConfig) == 2832     # the size of ABI 3 before io_flags
    assert _lib.ImxConfig.io_flags.offset == _lib.ImxConfig.obs_f32.offset + 4
    c = _config("serial4")
    h = ctypes.c_void_p()
    for flags, msg in ((4, b"unknown bits"), (_lib.IO_OBS_BF16 | 8, b"unknown bits")):
        c.io_flags = flags
        assert lib.imx_create(ctypes.byref(c), ctypes.byref(h)) == -1
        assert msg in lib.imx_last_error(), lib.imx_last_error()
        assert lib.imx_jit_compile_check(ctypes.byref(c), 0, None, 0) == -1
    c.io_flags, c.obs_f32 = _lib.IO_OBS_BF16, 1
    assert lib.imx_create(ctypes.byref(c), ctypes.byref(h)) == -1
    assert b"obs_f32 and IMX_IO_OBS_BF16" in lib.imx_last_error()


def test_io_flags_offset_agrees_with_the_c_header(tmp_path):
    gcc = shutil.which("gcc") or shutil.which("cc")
    if gcc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "off.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "imx_b200.h"\n'
                   'int main(void) { printf("%d %d %d %d\\n", (int)offsetof(imx_config, io_flags), (int)sizeof(imx_config), '
                   'IMX_IO_OBS_BF16, IMX_IO_ACTIONS_F32); return 0; }\n')
    exe = tmp_path / "off"
    subprocess.run([gcc, "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    off, size, bf16, f32 = map(int, subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split())
    assert (off, size) == (_lib.ImxConfig.io_flags.offset, ctypes.sizeof(_lib.ImxConfig))
    assert (bf16, f32) == (_lib.IO_OBS_BF16, _lib.IO_ACTIONS_F32)


def test_batched_options_are_refused_in_drop_in_mode():
    for kw in ({"obs_dtype": "bfloat16"}, {"action_dtype": "float32"}):
        with pytest.raises(ValueError, match="batched-mode"):
            ENV_CLASSES["MAIM"](dict(presets.serial4(), _config_only=True, **kw))
    c = ENV_CLASSES["MAIM"](dict(presets.serial4(), num_envs=8, obs_dtype=torch.bfloat16, action_dtype="float32", _config_only=True)).imx_config
    assert c.io_flags == _lib.IO_OBS_BF16 | _lib.IO_ACTIONS_F32 and c.obs_f32 == 0


def _round_host(x32):
    x32 = np.ascontiguousarray(x32, dtype=np.float32)
    out = np.empty(x32.shape, dtype=np.uint16)
    assert _lib.load().imx_round_bf16(x32.ctypes.data, out.ctypes.data, x32.size) == 0
    return out


def _round_torch(x32):
    return torch.from_numpy(np.ascontiguousarray(x32, dtype=np.float32)).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)


def test_torch_rounds_float64_to_bf16_through_float32():
    """The contract of the bfloat16 observations: torch's float64 -> bfloat16 conversion is the bfloat16 rounding of the
    float32 rounding (1 + 2^-8 + 2^-30 becomes 1.0, not the once-rounded 1.0078125)."""
    x = torch.tensor([1 + 2 ** -8 + 2 ** -30], dtype=torch.float64)
    assert x.to(torch.bfloat16).item() == 1.0
    assert x.to(torch.float32).to(torch.bfloat16).item() == 1.0


def test_host_bf16_rounding_is_torchs_on_every_table_entry():
    """Every entry a + (v (b - a)) / max of the rescale tables (imx_api.cu build_tables), for every preset's interval and
    every maximum up to twice its largest capacity (a superset of the four table rows of each node), rounded to float32 and
    then to bfloat16 on the host, equals torch's rounding bit for bit."""
    for name, make in presets.PRESETS.items():
        cfg = make()
        a, b = float(cfg.get("a", -1)), float(cfg.get("b", 1))
        caps = [int(x) for x in np.concatenate([np.ravel(cfg.get("inv_max", [100])), np.ravel(cfg.get("order_max", [100]))])]
        maxv = 2 * max(caps + [200])
        v = np.arange(0, 2 * maxv + 18, dtype=np.float64)
        vals = [a + (v * (b - a)) / float(mx) for mx in range(1, maxv + 1)]
        x32 = np.concatenate(vals).astype(np.float32)
        np.testing.assert_array_equal(_round_host(x32), _round_torch(x32), err_msg=name)


def test_host_bf16_rounding_edge_values():
    bits = [0x3F808000,             # 1 + 2^-8: a tie, rounds to the even 1.0
            0x3F818000,             # 1 + 3 * 2^-8: a tie, rounds up to the even 1 + 2^-6
            0x3F807FFF, 0x3F808001,  # just below / above the tie
            0x3FFFFFFF,             # rounds up into the next binade (2.0)
            0x7F7FFFFF, 0xFF7FFFFF,  # +-the largest finite float32 (round to +-inf, as torch does)
            0x80000000, 0x00000000,  # -0.0, +0.0
            0x00000001, 0x807FFFFF,  # subnormals
            0x7F800000, 0xFF800000]  # +-inf
    x32 = np.array([struct.unpack("<f", struct.pack("<I", u))[0] for u in bits], dtype=np.float32)
    np.testing.assert_array_equal(_round_host(x32), _round_torch(x32))
    # (observations are never NaN; the host keeps a NaN a NaN, whose payload torch's vectorised and scalar paths disagree on)
    assert (_round_host(np.array([np.nan], dtype=np.float32))[0] & 0x7FC0) == 0x7FC0
    assert list(_round_host(x32[:2])) == [0x3F80, 0x3F82]
    rng = np.random.default_rng(5)
    r = rng.integers(0, 2 ** 32, size=1 << 16, dtype=np.uint64).astype(np.uint32).view(np.float32)
    r = r[~np.isnan(r)]
    np.testing.assert_array_equal(_round_host(r), _round_torch(r))
