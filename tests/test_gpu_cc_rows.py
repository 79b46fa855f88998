"""Centralised-critic rows against a float64 reference, bit for bit, on every path that writes them.

A critic row of agent i is ``[opponent actions (m-1) | opponent observations (m-1)*O | own observation O]``
(models/CC_Model.py:165-214).  imx_step_cc writes the rows in the step kernel's epilogue where the specialised kernels serve
the whole batch (one tile per CTA, or the pipelined kernel), and otherwise runs the step and then the imx_cc_observe gather.
Both are compared here with ``cc_rows_ref``, a vectorised restatement of ``im_oracle.central_critic_flat``, over whole
episodes whose observations, rewards and final state come from the C oracle: serial chains of 1 to 32 stages, the divergent
presets, random trees, the env-per-thread step, three observation / action type pairs, non-finite and out-of-range actions
and five clip intervals, including ``lo == hi`` and ``lo > hi``.

The CPU tests pin the reference to ``central_critic_flat``, the oracle's clip to ``np.clip`` (signed zeros and NaN
included), the tile sizes that decide which cases are fused, and build every fused case's module for sm_100a."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from harness import copy_config, random_tree_config
from marl_for_im_b200 import _lib, presets
from marl_for_im_b200.envs import ENV_CLASSES
from oracle import c_oracle, im_oracle
from test_config_limits_cpu import chain32

DEV = "cuda:0"
SMEM_LIMIT = 200 * 1024                 # the largest tile layout a specialised module is built for
FLT_MAX = float(np.finfo(np.float32).max)
F32_TINY = float(np.nextafter(np.float32(0), np.float32(1)))     # the smallest float32 subnormal
# clip intervals: the default, one-sided, asymmetric, a single point, and lo > hi (np.clip gives hi)
CLIPS = [(-1.0, 1.0), (0.0, 1.0), (-2.5, 0.5), (0.25, 0.25), (0.5, -0.5)]
# observation / action element types
IO = {"f64": ("float64", "float64"), "f32": ("float32", "float64"), "bf16": ("bfloat16", "float32")}
_INT = {torch.float64: torch.int64, torch.float32: torch.int32, torch.bfloat16: torch.int16}


# --------------------------------------------------------------------------------------
# the reference
# --------------------------------------------------------------------------------------
def _opponents(m):
    """[m, m-1]: the opponents of agent i in agent order, skipping i."""
    return np.array([[q + (q >= i) for q in range(m - 1)] for i in range(m)], dtype=np.int64).reshape(m, m - 1)


def cc_rows_ref(obs, actions, lo, hi):
    """obs [N, m, O], actions [N, m] or None -> float64 rows [N, m, W].  The clip takes its operands in the order of
    central_critic_flat's ``min(max(v, lo), hi)``: a NaN stays NaN, -0.0 stays -0.0 against a bound of +0.0, and
    lo > hi gives hi."""
    obs = np.asarray(obs, dtype=np.float64)
    N, m, O = obs.shape
    opp = _opponents(m)
    out = np.zeros((N, m, (m - 1) * (1 + O) + O))
    if actions is not None:
        v = np.asarray(actions, dtype=np.float64)[:, opp]
        with np.errstate(invalid="ignore"):
            t = np.where(lo > v, lo, v)
            out[:, :, :m - 1] = np.where(hi < t, hi, t)
    out[:, :, m - 1:(m - 1) * (1 + O)] = obs[:, opp, :].reshape(N, m, (m - 1) * O)
    out[:, :, (m - 1) * (1 + O):] = obs
    return out


def narrow(x64, dtype):
    """float64 array -> CPU tensor of `dtype`: float32 by numpy, bfloat16 from that float32 by torch (two explicit steps)."""
    x64 = np.ascontiguousarray(x64, dtype=np.float64)
    if dtype == torch.float64:
        return torch.from_numpy(x64)
    f32 = torch.from_numpy(x64.astype(np.float32))
    return f32 if dtype == torch.float32 else f32.to(torch.bfloat16)


def assert_bits(got, want, what):
    """Same bit pattern in every element (assert_array_equal would take -0.0 for 0.0).  A bfloat16 NaN is 0x7FFF, the
    kernels' documented NaN, whatever NaN torch's conversion of the reference gives (rounding defines no NaN encoding); float64
    and float32 NaNs keep their bits, sign included."""
    got, want = got.detach().cpu().contiguous(), want.detach().cpu().contiguous()
    assert got.dtype == want.dtype and got.shape == want.shape, (what, got.dtype, want.dtype, tuple(got.shape), tuple(want.shape))
    if got.dtype in _INT:
        g, w = got.view(_INT[got.dtype]), want.view(_INT[want.dtype])
    else:
        g, w = got, want
    bad = g != w
    if got.dtype == torch.bfloat16:
        bad &= ~(torch.isnan(got) & torch.isnan(want) & (g == 0x7FFF))
    if bool(bad.any()):
        idx = bad.nonzero()[:4].tolist()
        pairs = [(i, hex(int(g[tuple(i)]) & 0xFFFFFFFFFFFFFFFF), hex(int(w[tuple(i)]) & 0xFFFFFFFFFFFFFFFF)) for i in idx]
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements differ; (index, got, want): {pairs}")


# --------------------------------------------------------------------------------------
# networks
# --------------------------------------------------------------------------------------
def chain(m, P=1, td=True, pd=True, pa=False, periods=12):
    """A MAIM chain of m stages with heterogeneous lead times and costs."""
    return {"num_stages": m, "num_periods": periods, "init_inv": 8.0 + np.arange(m) % 4, "inv_target": np.arange(m) % 3 * 1.0,
            "inv_max": np.full(m, 30.0), "price": np.arange(m + 1, 0, -1).astype(float) + 0.25,
            "stock_cost": 0.1 + 0.3 * (np.arange(m) % 4) / 4, "backlog_cost": 0.4 + 0.5 * (np.arange(m) % 3) / 3,
            "delay": 1 + np.arange(m) % 3, "time_dependency": td, "prev_demand": pd, "prev_actions": pa, "prev_length": P,
            "independent": m % 2 == 1, "standardise_state": True, "standardise_actions": True, "a": -1, "b": 1}


def _trees():
    rng = np.random.default_rng(2024)
    big = random_tree_config(rng, 12, 3, periods=12, prev_actions=True, prev_length=2)        # lane-mapped, 16-lane tile
    small = random_tree_config(rng, 7, 3, periods=12)                                        # 7 nodes: env-per-thread plain step
    five = random_tree_config(rng, 5, 2, periods=12, share_network=True)
    return big, small, five


TREE12, TREE7, TREE5 = _trees()
NETS = {
    "chain1": ("MAIM", chain(1)),
    "chain2": ("MAIM", presets.serial2()),
    "chain3": ("MAIM", chain(3, P=2, pa=True)),
    "chain4": ("MAIM", presets.serial4()),
    "chain5": ("MAIM", chain(5, td=False, pa=True)),
    "chain8": ("MAIM", presets.serial8(prev_actions=True, prev_length=2)),
    # the 16-stage chain's float64 critic-row tile: O = 9 fits in 200 KB (its 2-stage ring does not), O = 11 does not
    "chain16_fits": ("MAIM", chain(16, P=3, td=False, pa=True, periods=10)),
    "chain16_over": ("MAIM", chain(16, P=4, td=False, pa=True, periods=10)),
    "chain32": ("MAIM", chain32("MAIM", periods=6)),
    "div1": ("MAIM_div", presets.div1()),
    "div2": ("MAIM_div", presets.div2()),
    "div2_share": ("MAIM_div", presets.div2(share_network=True, prev_actions=True)),
    "tree12": ("MAIM_div", TREE12),
    "tree7": ("MAIM_div", TREE7),
    "tree5": ("MAIM_div", TREE5),
}


def make_env(net, io, n, **extra):
    kind, cfg = NETS[net]
    c = copy_config(cfg)
    c.update(num_envs=n, return_info=False, obs_dtype=IO[io][0], action_dtype=IO[io][1], **extra)
    return ENV_CLASSES[kind](c)


# --------------------------------------------------------------------------------------
# the tile layout of the critic-row module (compute_tile with the critic rows, imx_api.cu), from the imx_config
# --------------------------------------------------------------------------------------
def _derived(c):
    div = c.kind in (_lib.KIND["IM_div"], _lib.KIND["MAIM_div"])
    multi = c.kind in (_lib.KIND["MAIM"], _lib.KIND["MAIM_div"])
    m = c.num_nodes
    delay = [c.delay[i] for i in range(m)]
    D, L = max(delay), sum(delay)
    P = c.prev_length
    std_state = True if c.kind == _lib.KIND["MAIM_div"] else bool(c.standardise_state)
    write_hd = not (multi and c.prev_demand and not c.prev_actions and not c.time_dependency)
    need_hd = bool(c.prev_demand) and write_hd and not (multi and not std_state)
    need_ho = bool(c.prev_actions) and not (multi and not std_state)
    O = 3 + (P if c.prev_demand else 0) + (P if c.prev_actions else 0) + (D if c.time_dependency else 0) + \
        (1 if c.kind == _lib.KIND["MAIM_div"] and c.share_network else 0)
    nch = [c.num_children[i] for i in range(m)] if div else [0] * m
    NB = sum(k for k in nch if k > 1) if div else 0
    R = sum(1 for k in nch if k == 0) if div else 1
    S = 3 * m + L + (m * P if need_hd else 0) + (m * P if need_ho else 0) + (m if c.noisy_delay else 0) + NB
    es = 2 if c.io_flags & _lib.IO_OBS_BF16 else 4 if c.obs_f32 else 8
    ae = 4 if c.io_flags & _lib.IO_ACTIONS_F32 else 8
    m_pad = next(p for p in ((4, 8, 16, 32) if div else (2, 4, 8, 16, 32)) if m <= p)
    return dict(div=div, m=m, D=D, L=L, P=P, need_hd=need_hd, need_ho=need_ho, O=O, NB=NB, R=R, S=S, es=es, ae=ae, m_pad=m_pad,
                carry=bool(c.noisy_delay))


def cc_tile_bytes(c):
    """Bytes of one critic-row tile: compute_tile(e, e->tile_cc, m_pad, true) with choose_tma_threads' default CTA size."""
    d = _derived(c)
    m, N = d["m"], c.num_envs
    per_env = 8 * d["S"] + 4 * d["R"] + m * (d["ae"] + 8 + d["O"] * d["es"])
    small4 = not d["div"] and d["m_pad"] == 4 and N >= 1024 and per_env * N <= (192 << 20)
    big4 = not d["div"] and d["m_pad"] == 4 and N >= (1 << 19)
    threads = 64 if small4 else 256 if (big4 or (d["m_pad"] <= 4 and N >= (1 << 20))) else 128
    E = (threads // 32) * (32 // d["m_pad"])
    W = (m - 1) * (1 + d["O"]) + d["O"]
    off = 0
    for nbytes in (E * m * (12 if d["ae"] == 4 else 8), E * m * 4, E * m * 4, E * m * 4, E * d["L"] * 4,
                   E * m * d["P"] * 4 if d["need_hd"] else 0, E * m * d["P"] * 4 if d["need_ho"] else 0,
                   E * m * 4 if d["carry"] else 0, E * d["NB"] * 4, d["R"] * E * 4, E * m * d["O"] * d["es"], E * m * 8,
                   E * m * W * d["es"]):
        off += (nbytes + 127) & ~127
    return off, E


def config_of(net, io, n, noisy=False):
    """The imx_config of a case's handle; `noisy`: the handle a reset with a delay mask creates (with the carry state)."""
    c = make_env(net, io, n, _config_only=True).imx_config
    c.noisy_delay = int(bool(noisy))
    return c


SMS = 148                               # B200: the pipelined grid of IMX_PIPE_CTAS=1 is one CTA per SM


def pipe_stages(total, switches):
    """pipe_stages_for() of the critic-row layout: 4 stages (or IMX_PIPE_STAGES), fewer while the ring exceeds 200 KB or
    fewer than four CTAs would fit on an SM."""
    s = int(switches.get("IMX_PIPE_STAGES", 0)) or 4
    while s > 2 and (s * total > SMEM_LIMIT or (227 * 1024) // (s * total + 1024) < 4):
        s -= 1
    return s


# --------------------------------------------------------------------------------------
# the GPU matrix: (network, I/O types, N, path, switches, options)
#   path "one": fused, the one-tile kernel (variant 2); "pipe": fused, the pipelined kernel (variant 3);
#   "unfused": the step's launches and one gather.  Options: "mix" interleaves step_cc, step and step_many periods;
#   "noisy" replays a noisy-delay mask; "offset" writes the rows 8 bytes past a 16-byte boundary.
# --------------------------------------------------------------------------------------
ONE = {"IMX_PIPE": "0"}
PIPE = {"IMX_PIPE": "1", "IMX_PIPE_CTAS": "1"}
PIPE2 = {"IMX_PIPE": "1", "IMX_PIPE_CTAS": "1", "IMX_PIPE_STAGES": "2"}
ET = {"IMX_STEP_ET": "1"}
CASES = {
    "chain1-f64-one": ("chain1", "f64", 4096, "one", ONE, ()),
    "chain1-bf16-pipe": ("chain1", "bf16", 98304, "pipe", PIPE, ()),
    "chain2-f64-one": ("chain2", "f64", 4096, "one", ONE, ()),
    "chain2-f32-pipe": ("chain2", "f32", 65536, "pipe", PIPE, ()),
    "chain2-bf16-pipe2": ("chain2", "bf16", 65536, "pipe", PIPE2, ()),
    "chain3-f64-pipe": ("chain3", "f64", 16384, "pipe", PIPE, ()),
    "chain3-f32-one": ("chain3", "f32", 4096, "one", ONE, ()),
    "chain4-f64-one": ("chain4", "f64", 4096, "one", ONE, ()),
    "chain4-bf16-pipe": ("chain4", "bf16", 32768, "pipe", PIPE, ()),
    "chain4-f64-pipe-default-ring": ("chain4", "f64", 16384, "pipe", PIPE, ()),
    "chain4-f32-tail": ("chain4", "f32", 4096 + 4, "unfused", PIPE, ()),
    "chain4-f64-noisy": ("chain4", "f64", 4096, "one", ONE, ("noisy",)),
    "chain4-f64-offset": ("chain4", "f64", 4096, "unfused", ONE, ("offset",)),
    "chain5-f64-pipe2": ("chain5", "f64", 16384, "pipe", PIPE2, ()),
    "chain5-bf16-one": ("chain5", "bf16", 4096, "one", ONE, ()),
    "chain8-f64-one": ("chain8", "f64", 4096, "one", ONE, ()),
    "chain8-f32-pipe": ("chain8", "f32", 8192, "pipe", PIPE, ()),
    "chain8-f64-small": ("chain8", "f64", 512, "unfused", {}, ()),
    "chain16-f64-fits-no-ring": ("chain16_fits", "f64", 1024, "one", PIPE, ()),
    "chain16-bf16-pipe": ("chain16_fits", "bf16", 4096, "pipe", PIPE, ()),
    "chain16-f64-over": ("chain16_over", "f64", 1024, "unfused", PIPE, ()),
    "chain32-f64-over": ("chain32", "f64", 1024, "unfused", PIPE, ()),
    "chain32-bf16-over": ("chain32", "bf16", 1024, "unfused", ONE, ()),
    "div1-f64-one": ("div1", "f64", 4096, "one", ONE, ()),
    "div1-bf16-pipe": ("div1", "bf16", 32768, "pipe", PIPE, ()),
    "div1-et-f64-one": ("div1", "f64", 4096, "one", dict(ONE, **ET), ("mix",)),
    "div1-et-f32-pipe": ("div1", "f32", 16384, "pipe", dict(PIPE, **ET), ("mix",)),
    "div2-f64-one": ("div2", "f64", 4096, "one", ONE, ("mix",)),
    "div2-bf16-pipe": ("div2", "bf16", 32768, "pipe", PIPE, ("mix",)),
    "div2-f32-pipe2": ("div2", "f32", 8192, "pipe", PIPE2, ("mix",)),
    "div2-f32-tail": ("div2", "f32", 4096 + 4, "unfused", PIPE, ("mix",)),
    "div2-bf16-offset": ("div2", "bf16", 4096, "unfused", PIPE, ("offset", "mix")),
    "div2-share-f64-pipe": ("div2_share", "f64", 8192, "pipe", PIPE, ()),
    "div2-share-f32-one": ("div2_share", "f32", 4096, "one", ONE, ()),
    "tree12-f64-one": ("tree12", "f64", 4096, "one", ONE, ()),
    "tree12-bf16-pipe": ("tree12", "bf16", 4096, "pipe", PIPE, ()),
    "tree7-f64-pipe": ("tree7", "f64", 8192, "pipe", PIPE, ("mix",)),
    "tree7-f32-one": ("tree7", "f32", 4096, "one", ONE, ("mix",)),
    "tree7-f64-noisy": ("tree7", "f64", 8192, "pipe", PIPE, ("noisy",)),
    "tree5-bf16-one": ("tree5", "bf16", 4096, "one", ONE, ()),
    "tree5-f64-small": ("tree5", "f64", 768, "unfused", {}, ()),
}


# --------------------------------------------------------------------------------------
# CPU tests
# --------------------------------------------------------------------------------------
def _specials():
    return [0.0, -0.0, math.inf, -math.inf, math.nan, FLT_MAX, -FLT_MAX, 1e300, -1e300, 5e-324, -5e-324, F32_TINY,
            1.0, -1.0, 0.25, 0.5, -0.5, 2.5, -2.5, 1.4, -1.4, 0.999, -1.001]


def test_cc_rows_ref_equals_central_critic_flat():
    rng = np.random.default_rng(0)
    sp = np.array(_specials())
    for m, O in ((1, 3), (2, 1), (3, 5), (5, 2), (8, 7), (13, 4)):
        N = 40
        obs = rng.uniform(-1, 1, size=(N, m, O))
        obs[rng.uniform(size=obs.shape) < 0.2] = -0.0
        obs[rng.uniform(size=obs.shape) < 0.1] = 5e-324
        act = np.where(rng.uniform(size=(N, m)) < 0.6, rng.choice(sp, size=(N, m)), rng.uniform(-3, 3, size=(N, m)))
        for lo, hi in CLIPS + [(-0.0, 0.0), (0.0, -0.0)]:
            for a in (act, None):
                got = cc_rows_ref(obs, a, lo, hi)
                want = np.stack([im_oracle.central_critic_flat(obs[n], None if a is None else a[n], (lo, hi)) for n in range(N)])
                assert_bits(torch.from_numpy(got), torch.from_numpy(want), f"m={m} O={O} clip=({lo}, {hi})")


def test_oracle_clip_matches_np_clip():
    """central_critic_flat clips like np.clip, bit for bit: NaN stays NaN, signed zeros as numpy gives them, lo > hi -> hi."""
    sp = _specials()
    for lo, hi in CLIPS + [(-0.0, 0.0), (0.0, -0.0), (-0.0, 1.0), (-1.0, 0.0), (-1.0, -0.0)]:
        got = np.array([im_oracle.central_critic_flat(np.zeros((2, 1)), [0.0, v], (lo, hi))[0, 0] for v in sp])
        want = np.clip(np.array(sp), lo, hi)
        np.testing.assert_array_equal(got.view(np.int64), want.view(np.int64), err_msg=f"clip=({lo}, {hi})")
    assert math.isnan(im_oracle.central_critic_flat(np.zeros((2, 1)), [0.0, math.nan])[0, 0])


def test_case_layouts_sit_on_the_intended_side_of_the_limit():
    """The 16-stage chain straddles the 200 KB limit in float64 (one side each), its fitting layout has no room for a 2-stage
    ring, and the 32-stage chain is over in float64 and bfloat16: the paths the GPU cases pin follow from these sizes.  Every
    pipelined case has more tiles per CTA than its ring has stages, config 5's shape (the 2-stage chain, float32 rows, 3 stages)
    among them, and the 3- and 4-stage rings are covered."""
    fits, _ = cc_tile_bytes(config_of("chain16_fits", "f64", 1024))
    over, _ = cc_tile_bytes(config_of("chain16_over", "f64", 1024))
    assert fits <= SMEM_LIMIT < 2 * fits and over > SMEM_LIMIT
    bf16, _ = cc_tile_bytes(config_of("chain16_fits", "bf16", 1024))
    assert 2 * bf16 <= SMEM_LIMIT                  # chain16-bf16-pipe has a ring
    for io in ("f64", "bf16"):
        assert cc_tile_bytes(config_of("chain32", io, 1024))[0] > SMEM_LIMIT
    for name, (net, io, n, path, switches, opts) in CASES.items():
        total, E = cc_tile_bytes(config_of(net, io, n, "noisy" in opts))
        if path in ("one", "pipe"):
            assert total <= SMEM_LIMIT and n % E == 0, name
        if path == "pipe":
            assert 2 * total <= SMEM_LIMIT, name
            # one CTA per SM walks its tiles through the ring: more tiles per CTA than stages, so stages are refilled
            assert switches.get("IMX_PIPE_CTAS") == "1" and n // E >= (pipe_stages(total, switches) + 1) * SMS, name


def _fused_builds():
    seen, out = set(), []
    for name, (net, io, n, path, env, opts) in CASES.items():
        key = (net, io, "noisy" in opts, env.get("IMX_PIPE", ""), env.get("IMX_PIPE_STAGES", ""), env.get("IMX_STEP_ET", ""))
        if key in seen or path not in ("one", "pipe"):
            continue
        seen.add(key)
        out.append(name)
    return out


@pytest.mark.parametrize("name", _fused_builds())
def test_critic_row_module_builds_for_sm100a(name, monkeypatch):
    """imx_jit_compile_check(variant 2): the module every fused case loads compiles for sm_100a without a GPU."""
    net, io, n, path, env, opts = CASES[name]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    c = config_of(net, io, n, "noisy" in opts)
    assert cc_tile_bytes(c)[0] <= SMEM_LIMIT
    buf = C.create_string_buffer(8192)
    got = _lib.load().imx_jit_compile_check(C.byref(c), 2, buf, 8192)
    assert got > 10000, (name, got, buf.value.decode()[:500], _lib.load().imx_last_error())


# --------------------------------------------------------------------------------------
# GPU tests
# --------------------------------------------------------------------------------------
def _actions(rng, N, m, lo, hi):
    """[N, m]: in the clip interval, beyond it, and special values (bounds, signed zeros, infinities, NaN, FLT_MAX, 1e300,
    subnormals)."""
    a, b = min(lo, hi), max(lo, hi)
    cat = rng.uniform(size=(N, m))
    inside = rng.uniform(a, b, size=(N, m)) if b > a else np.full((N, m), a)
    beyond = rng.uniform(-1.4, 1.4, size=(N, m)) * max(1.0, abs(lo), abs(hi))
    sp = np.array([lo, hi, 0.0, -0.0, math.inf, -math.inf, math.nan, FLT_MAX, -FLT_MAX, 1e300, 5e-324, F32_TINY])
    special = rng.choice(sp, size=(N, m))
    return np.where(cat < 0.4, inside, np.where(cat < 0.7, beyond, special))


def _schedule(T, mix):
    """Per period: "cc" (imx_step_cc, from the reset state first), "plain" (imx_step, then imx_cc_observe) or "many" (two
    periods of imx_step_many)."""
    out, t = [], 0
    while t < T:
        if mix and t % 5 == 3 and t + 2 <= T:
            out.append((t, "many", 2))
            t += 2
        elif t == 1 or (mix and t % 5 == 1):
            out.append((t, "plain", 1))
            t += 1
        else:
            out.append((t, "cc", 1))
            t += 1
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_cc_rows_match_the_reference(name, monkeypatch):
    net, io, N, path, switches, opts = CASES[name]
    for k, v in switches.items():
        monkeypatch.setenv(k, v)
    kind = NETS[net][0]
    seed = sum(map(ord, name))
    rng = np.random.default_rng(seed)
    env = make_env(net, io, N)
    m, O, T, R = env.num_nodes, env.obs_len, env.num_periods, len(env._retailers)
    W = (m - 1) * (1 + O) + O
    dt = env.obs_dtype
    act_f32 = env.action_dtype == torch.float32
    demand = rng.poisson(5, size=(N, R, T)).astype(np.int32)
    clips = [CLIPS[(t + seed) % len(CLIPS)] for t in range(T)]
    fills = [t % 4 != 2 for t in range(T)]
    want_obs = [t % 3 != 1 for t in range(T)]
    actions = np.stack([_actions(rng, N, m, *clips[t]) for t in range(T)])
    if act_f32:
        with np.errstate(over="ignore"):                               # 1e300 and FLT_MAX-beyond values become +-inf
            actions = actions.astype(np.float32).astype(np.float64)   # what the handle reads, widened exactly
    mask = (rng.uniform(size=(N, T, m)) < 0.3) if "noisy" in opts else None
    want = c_oracle.COracle(kind, NETS[net][1]).run(demand, actions, delay_mask=mask, all_obs=True)
    env.reset(customer_demand=demand, delay_mask=mask)     # (a delay mask gives the env a new handle, with the carry state)
    lib, h = env._lib, env._handle
    a_dev = torch.as_tensor(actions, device=DEV).to(env.action_dtype).contiguous()

    # the rows go into a sentinel-filled buffer, 8 bytes past a 16-byte boundary for the "offset" cases
    es = torch.empty((), dtype=dt).element_size()
    row_bytes, pad, off = N * m * W * es, 256, (8 if "offset" in opts else 0)
    big = torch.full((row_bytes + 2 * pad,), 0x5A, dtype=torch.uint8, device=DEV)
    rows = big[pad + off:pad + off + row_bytes].view(dt).view(N, m, W)
    outside = torch.ones_like(big, dtype=torch.bool)
    outside[pad + off:pad + off + row_bytes] = False
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def check_obs_rew(obs, rew, t, what):
        if obs is not None:
            assert_bits(obs, narrow(want["obs_all"][t + 1], dt), f"{what}: observations t={t}")
        assert_bits(rew, torch.from_numpy(np.ascontiguousarray(want["reward"][t])), f"{what}: rewards t={t}")

    def ref(t):
        return cc_rows_ref(want["obs_all"][t + 1], actions[t] if fills[t] else None, *clips[t])

    plain_launches, cc_calls = None, []
    for t, what, k in _schedule(T, "mix" in opts):
        n0 = lib.imx_launch_count()
        if what == "plain":
            obs, rew, _ = env.step_packed(a_dev[t])
            plain_launches = lib.imx_launch_count() - n0
            check_obs_rew(obs, rew, t, "step")
            # the gather reads the observations in the env's element type: the reference starts from those values
            stored = narrow(want["obs_all"][t + 1], dt).double().numpy()
            r64 = cc_rows_ref(stored, actions[t] if fills[t] else None, *clips[t])
            for out in (torch.float64, torch.float32, torch.bfloat16):    # the gather, to every output type
                got = cc_observe_raw(env, obs, a_dev[t] if fills[t] else None, clips[t], out)
                assert_bits(got, narrow(r64, out), f"imx_cc_observe to {out} t={t}")
        elif what == "many":
            obs_m, rew_m, _ = env.step_many(a_dev[t:t + k])
            for j in range(k):
                check_obs_rew(obs_m[j], rew_m[j], t + j, "step_many")
        else:
            obs = torch.empty((N, m, O), dtype=dt, device=DEV) if want_obs[t] else None
            rew = torch.empty((N, m), dtype=torch.float64, device=DEV)
            lo, hi = clips[t]
            _lib.check(lib.imx_step_cc(h, C.c_void_p(a_dev[t].data_ptr()), C.c_void_p(obs.data_ptr()) if obs is not None else None,
                                       C.c_void_p(rows.data_ptr()), int(fills[t]), lo, hi, C.c_void_p(rew.data_ptr()), stream))
            cc_calls.append((t, lib.imx_launch_count() - n0, lib.imx_kernel_variant(h)))
            check_obs_rew(obs, rew, t, "step_cc")
            assert_bits(rows, narrow(ref(t), dt), f"critic rows t={t} clip={clips[t]} fill={fills[t]} want_obs={want_obs[t]}")
            assert bool((big[outside] == 0x5A).all()), f"a byte outside the critic rows changed at t={t}"
    assert env.period == T and env._handle.value == h.value
    # the path of every imx_step_cc call: one launch of the fused kernel, or the plain step's launches and one gather
    assert cc_calls and plain_launches
    for t, launches, variant in cc_calls:
        if path == "unfused":
            assert launches == plain_launches + 1, (t, launches, plain_launches)
        else:
            assert (launches, variant) == (1, 2 if path == "one" else 3), (t, launches, variant)
    st = {k: v.cpu().numpy() for k, v in env.state_dict().items()}
    for key in ("inv", "backlog", "order_u", "pipe", "backlog_to"):
        if key in st:
            np.testing.assert_array_equal(st[key], want[key], err_msg=key)
    np.testing.assert_array_equal(env.error_flags.cpu().numpy(), want["err"])
    # past the end of the episode: refused, nothing written
    rew = torch.empty((N, m), dtype=torch.float64, device=DEV)
    assert lib.imx_step_cc(h, C.c_void_p(a_dev[0].data_ptr()), None, C.c_void_p(rows.data_ptr()), 1, -1.0, 1.0,
                           C.c_void_p(rew.data_ptr()), stream) == -6
    assert env.period == T
    torch.cuda.synchronize()


def cc_observe_raw(env, obs, act, clip, out_dtype):
    """imx_cc_observe on the env's packed observations (its own element type) into an `out_dtype` tensor."""
    N, m, O = env.num_envs, env.num_nodes, env.obs_len
    W = env._lib.imx_cc_obs_len(env._handle)
    out = torch.empty((N, m, W), dtype=out_dtype, device=DEV)
    code = {torch.float64: 0, torch.float32: 1, torch.bfloat16: 2}[out_dtype]
    _lib.check(env._lib.imx_cc_observe(env._handle, C.c_void_p(obs.data_ptr()), C.c_void_p(act.data_ptr()) if act is not None else None,
                                       float(clip[0]), float(clip[1]), C.c_void_p(out.data_ptr()), code, env._stream()))
    return out


@pytest.mark.gpu
def test_cc_entry_points_refuse_bad_arguments():
    env = make_env("chain2", "f64", 256)
    lib, h = env._lib, env._handle
    N, m, O = env.num_envs, env.num_nodes, env.obs_len
    W = lib.imx_cc_obs_len(h)
    obs = torch.zeros((N, m, O), dtype=torch.float64, device=DEV)
    act = torch.zeros((N, m), dtype=torch.float64, device=DEV)
    out = torch.zeros((N, m, W), dtype=torch.float64, device=DEV)
    rew = torch.zeros((N, m), dtype=torch.float64, device=DEV)
    p = lambda x: C.c_void_p(x.data_ptr()) if x is not None else None     # noqa: E731
    s = env._stream()
    assert lib.imx_cc_observe(h, p(obs), p(act), -1.0, 1.0, p(out), 3, s) == -1
    assert lib.imx_cc_observe(h, p(obs), p(act), -1.0, 1.0, p(out), -1, s) == -1
    assert lib.imx_cc_observe(h, None, p(act), -1.0, 1.0, p(out), 0, s) == -1
    assert lib.imx_cc_observe(h, p(obs), p(act), -1.0, 1.0, None, 0, s) == -1
    assert lib.imx_cc_observe(None, p(obs), p(act), -1.0, 1.0, p(out), 0, s) == -1
    for a, o, c, r in ((None, obs, out, rew), (act, obs, None, rew), (act, obs, out, None)):
        assert lib.imx_step_cc(h, p(a), p(o), p(c), 1, -1.0, 1.0, p(r), s) == -1
    assert lib.imx_step_cc(None, p(act), p(obs), p(out), 1, -1.0, 1.0, p(rew), s) == -1
    assert env.period == 0                                 # a refused call advances nothing
    # the single-agent kinds have no critic rows
    im = ENV_CLASSES["IM"](dict(presets.serial4(), num_envs=N))
    o4 = torch.zeros((N, 4, im.obs_len), dtype=torch.float64, device=DEV)
    a4 = torch.zeros((N, 4), dtype=torch.float64, device=DEV)
    r4 = torch.zeros((N,), dtype=torch.float64, device=DEV)
    assert im._lib.imx_cc_observe(im._handle, p(o4), p(a4), -1.0, 1.0, p(out), 0, s) == -1
    assert im._lib.imx_step_cc(im._handle, p(a4), p(o4), p(out), 1, -1.0, 1.0, p(r4), s) == -1
    assert im.period == 0
    with pytest.raises(_lib.ImxError):
        im.step_cc(a4)
    torch.cuda.synchronize()
