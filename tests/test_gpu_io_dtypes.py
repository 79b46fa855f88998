"""bfloat16 observations (``obs_dtype="bfloat16"`` / ``IMX_IO_OBS_BF16``) and float32 actions (``action_dtype="float32"`` /
``IMX_IO_ACTIONS_F32``), through every entry point.  Every comparison is bit for bit:
  - a bfloat16 observation is the float32 handle's observation ``.to(torch.bfloat16)`` (compared through an int16 view);
  - a float32-action handle on ``a32`` computes what a float64 handle computes on ``a32.double()``;
  - rewards, every state field, the split's error flags and the diagnostics do not depend on either type."""
import ctypes as C
import struct

import numpy as np
import pytest
import torch

from harness import copy_config, random_case
from marl_for_im_b200 import _lib, presets
from marl_for_im_b200.cc import cc_observe
from marl_for_im_b200.envs import ENV_CLASSES

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# the cases of tests/test_gpu_obs_f32.py: all four kinds, obs modes, non-standardised, share_network
CASES = [("MAIM", "serial4", {}), ("MAIM", "serial8", dict(prev_actions=True, prev_length=3, independent=True)),
         ("IM", "serial4", dict(prev_actions=True, prev_length=2)), ("MAIM", "serial2", {}),
         ("IM", "serial4_dfo", {}), ("MAIM", "serial4", dict(standardise_state=False, standardise_actions=False)),
         ("MAIM_div", "div1", {}), ("MAIM_div", "div2", dict(share_network=True, prev_actions=True)),
         ("IM_div", "div2", dict(prev_length=2))]


def _serial5(**kw):
    """5-stage chain observing (inv, backlog, unfulfilled, last demand, last order): m = 5, O = 5 — a bfloat16 warp tile of the
    direct kernel (4 envs) is 200 bytes, not a whole number of 16-byte units."""
    c = presets.serial8(time_dependency=False, prev_demand=True, prev_actions=True, prev_length=1, **kw)
    c["num_stages"] = 5
    for k in ("init_inv", "inv_target", "inv_max", "stock_cost", "backlog_cost", "delay"):
        c[k] = np.asarray(c[k])[:5]
    c["price"] = np.asarray(c["price"])[:6]
    return c


def _cfg(preset, kw):
    return _serial5(**kw) if preset == "serial5" else presets.PRESETS[preset](**kw)


def _make(kind, cfg, n, obs="float64", act="float64"):
    c = copy_config(cfg)
    c.update(num_envs=n, return_info=False, obs_dtype=obs, action_dtype=act)
    return ENV_CLASSES[kind](c)


def _trace(kind, cfg, n, seed, mode=None):
    """demand [n, R, T] int32 and actions [T, n, m] float32 (values any float64 caller could pass as well)."""
    rng = np.random.default_rng(seed)
    mode = mode or ("near_eq" if kind.endswith("div") else "uniform")
    dem, act = zip(*(random_case(kind, cfg, rng, mu=6, action_mode=mode) for _ in range(n)))
    demand = np.stack(dem).astype(np.int32).reshape(n, -1, cfg["num_periods"])
    a32 = torch.as_tensor(np.ascontiguousarray(np.stack(act, axis=1)), dtype=torch.float32)
    return demand, a32


def _eq(x, y, what=""):
    x, y = x.detach().cpu(), y.detach().cpu()
    assert x.dtype == y.dtype and x.shape == y.shape, (what, x.dtype, y.dtype, x.shape, y.shape)
    if x.dtype == torch.bfloat16:
        x, y = x.view(torch.int16), y.view(torch.int16)
    assert torch.equal(x, y), what


def _eq_bf16(xb, y32, what=""):
    """a bfloat16 output equals a float32 output rounded by torch"""
    assert xb.dtype == torch.bfloat16 and y32.dtype == torch.float32, what
    _eq(xb, y32.to(torch.bfloat16), what)


def _state(env):
    st = {k: v.clone() for k, v in env.state_dict().items()}
    st["err"] = env.error_flags.clone()
    return st


def _episode(env, demand, actions):
    """reset + T steps: stacked observations [T + 1, N, m, O] (the reset observation first), rewards, final state, variant"""
    env.reset(customer_demand=demand)
    obs, rew = [env.last_obs.clone()], []
    a = actions.to(device=DEV, dtype=env.action_dtype)
    for t in range(env.num_periods):
        env.step(a[t])
        obs.append(env.last_obs.clone())
        rew.append(env.last_reward.clone())
    torch.cuda.synchronize()
    return torch.stack(obs), torch.stack(rew), _state(env), env._lib.imx_kernel_variant(env._handle)


def _check_against(kind, cfg, n, demand, a32, got):
    """got = (_episode of a bfloat16 / float32-action handle) against float32- and float64-observation handles on a32.double()"""
    o32, r32, s32, _ = _episode(_make(kind, cfg, n, "float32"), demand, a32.double())
    _, r64, s64, _ = _episode(_make(kind, cfg, n, "float64"), demand, a32.double())
    ob, rb, sb, _ = got
    _eq_bf16(ob, o32, "observations")
    _eq(rb, r64, "rewards")
    _eq(r32, r64, "rewards (float32 observations)")
    for k in s64:
        _eq(sb[k], s64[k], k)


@pytest.mark.parametrize("n", [96, 97, 4096, 4097])
@pytest.mark.parametrize("kind,preset,kw", CASES)
def test_bf16_obs_and_f32_actions_match_the_wider_types(kind, preset, kw, n, monkeypatch):
    if n == 96:
        monkeypatch.setenv("IMX_JIT", "0")           # ahead-of-time kernels
    cfg = _cfg(preset, kw)
    demand, a32 = _trace(kind, cfg, n, 31 + n)
    got = _episode(_make(kind, cfg, n, "bfloat16", "float32"), demand, a32)
    assert got[0].dtype == torch.bfloat16 and got[0].shape[0] == cfg["num_periods"] + 1
    if n == 4096:
        assert got[3] in (2, 3)                      # the runtime-specialised fast path served the whole batch
    _check_against(kind, cfg, n, demand, a32, got)
    # each type on its own
    ob, rb, sb, _ = _episode(_make(kind, cfg, n, "bfloat16", "float64"), demand, a32.double())
    _eq(ob, got[0], "bfloat16 observations with float64 actions")
    o64, r64, s64, _ = _episode(_make(kind, cfg, n, "float64", "float32"), demand, a32)
    o64r, r64r, _, _ = _episode(_make(kind, cfg, n, "float64", "float64"), demand, a32.double())
    _eq(o64, o64r, "float64 observations with float32 actions")
    _eq(r64, r64r)


def _f32(bits):
    return struct.unpack("<f", struct.pack("<I", bits))[0]


def _special_actions(kind, cfg, n, seed):
    """float32 actions with the values decode_order must treat exactly as their float64 widening: +-inf, NaN, +-FLT_MAX, -0.0,
    a subnormal, and the float32 neighbours of order_max and of 2^63 after scaling"""
    m, T = (cfg.get("num_stages") or cfg["num_nodes"]), cfg["num_periods"]
    std = cfg.get("standardise_actions", True) or kind == "MAIM_div"
    a, b = float(cfg.get("a", -1)), float(cfg.get("b", 1))
    om = 30.0 if kind.startswith("MAIM") else 100.0
    om = float(np.max(np.ravel(cfg.get("order_max", [om]))))
    if std:
        edge = [b, a + (2.0 ** 63) * (b - a) / om]                     # the actions that scale to order_max and to 2^63
    else:
        edge = [om, om + 0.5, 2.0 ** 63]
    sp = [float("inf"), -float("inf"), float("nan"), _f32(0x7F7FFFFF), _f32(0xFF7FFFFF), -0.0, _f32(0x00000001)]
    for x in edge:
        x32 = np.float32(x)
        sp += [float(x32), float(np.nextafter(x32, np.float32(np.inf))), float(np.nextafter(x32, np.float32(-np.inf)))]
    rng = np.random.default_rng(seed)
    _, base = _trace(kind, cfg, n, seed)
    pick = torch.as_tensor(rng.uniform(size=(T, n, m)) < 0.3)
    vals = torch.as_tensor(np.asarray(sp, dtype=np.float32)[rng.integers(0, len(sp), size=(T, n, m))])
    return torch.where(pick, vals, base)


@pytest.mark.parametrize("n", [97, 4096])
@pytest.mark.parametrize("kind,preset,kw", [("MAIM", "serial4", {}), ("MAIM", "serial4", dict(standardise_state=False, standardise_actions=False)),
                                            ("IM", "serial4", {}), ("MAIM_div", "div2", {}), ("IM_div", "div1", {})])
def test_f32_action_specials_decode_like_float64(kind, preset, kw, n):
    cfg = _cfg(preset, kw)
    demand, _ = _trace(kind, cfg, n, 3)
    a32 = _special_actions(kind, cfg, n, 11 + n)
    out = []
    for act, a in (("float32", a32), ("float64", a32.double())):
        env = _make(kind, cfg, n, "float64", act)
        env.reset(customer_demand=demand)
        o, r, _, info = env.step_many(a.to(DEV), return_info=True)
        torch.cuda.synchronize()
        out.append((o.clone(), r.clone(), {k: v.clone() for k, v in info.items()}, _state(env)))
    (o1, r1, i1, s1), (o2, r2, i2, s2) = out
    _eq(o1, o2, "obs")
    _eq(r1, r2, "rewards")
    for k in i2:
        _eq(i1[k], i2[k], k)
    for k in s2:
        _eq(s1[k], s2[k], k)


PATHS = {"direct": ({"IMX_STEP_PATH": "direct"}, (0,)), "aot_tma": ({"IMX_JIT": "0", "IMX_STEP_PATH": "tma"}, (1,)),
         "specialised": ({"IMX_PIPE": "0"}, (2,)), "pipelined": ({"IMX_PIPE": "1"}, (3,)),
         "env_per_thread": ({"IMX_STEP_ET": "1", "IMX_PIPE": "0"}, (2,)), "lanes": ({"IMX_STEP_ET": "0"}, (2, 3))}


@pytest.mark.parametrize("path", sorted(PATHS))
@pytest.mark.parametrize("kind,preset", [("MAIM", "serial4"), ("IM", "serial8"), ("MAIM_div", "div2"), ("IM_div", "div1")])
def test_step_on_every_path(kind, preset, path, monkeypatch):
    env_vars, variants = PATHS[path]
    for k, v in env_vars.items():
        monkeypatch.setenv(k, v)
    cfg, n = presets.PRESETS[preset](), 4096
    demand, a32 = _trace(kind, cfg, n, 5)
    got = _episode(_make(kind, cfg, n, "bfloat16", "float32"), demand, a32)
    assert got[3] in variants, got[3]
    _check_against(kind, cfg, n, demand, a32, got)


@pytest.mark.parametrize("fuse", ["1", "0"])
@pytest.mark.parametrize("kind,preset", [("MAIM", "serial4"), ("IM", "serial8"), ("MAIM_div", "div2")])
def test_step_many_fused_and_unfused(kind, preset, fuse, monkeypatch):
    monkeypatch.setenv("IMX_FUSE_PERIODS", fuse)
    cfg, n = presets.PRESETS[preset](), 4096
    demand, a32 = _trace(kind, cfg, n, 6)
    res = {}
    for key, obs, act, a in (("b", "bfloat16", "float32", a32), ("f", "float32", "float64", a32.double()), ("d", "float64", "float64", a32.double())):
        env = _make(kind, cfg, n, obs, act)
        for info_wanted in (False, True):              # without diagnostics the specialised kernels serve, with them the others
            env.reset(customer_demand=demand)
            o, r, _, *info = env.step_many(a.to(DEV), return_info=info_wanted)
            torch.cuda.synchronize()
            res[key, info_wanted] = (o.clone(), r.clone(), info[0] if info else {}, _state(env), env._lib.imx_kernel_variant(env._handle))
    if fuse == "1":
        assert res["b", False][4] == 2 and res["b", True][4] == 1      # the fused multi-period kernels
    for w in (False, True):
        _eq_bf16(res["b", w][0], res["f", w][0], "obs")
        _eq(res["b", w][1], res["d", w][1], "rewards")
        for k in res["d", w][2]:
            _eq(res["b", w][2][k], res["d", w][2][k], k)
        for k in res["d", w][3]:
            _eq(res["b", w][3][k], res["d", w][3][k], k)


@pytest.mark.parametrize("call,preset,want_obs", [("step_many", "serial4", False), ("replay", "serial4", False),
                                                  ("step_many", "serial8", False), ("step_many", "serial8", True),
                                                  ("replay", "serial8", True)])
def test_shared_reward_scratch_with_f32_actions(call, preset, want_obs):
    """The multi-period kernels sum a shared reward through a float64 scratch in the action region (rewards-only replays, and
    networks of 6 or more nodes): with float32 actions it must not overwrite actions that other warps have not read yet."""
    kind, n = "MAIM", 65536
    cfg = presets.PRESETS[preset]()
    assert not cfg.get("independent", False)         # the shared (mean) reward
    demand, a32 = _trace(kind, cfg, n, 14)
    res = {}
    for act, a in (("float32", a32), ("float64", a32.double())):
        env = _make(kind, cfg, n, "float64", act)
        if call == "step_many":
            env.reset(customer_demand=demand)
            o, r, _ = env.step_many(a.to(DEV), want_obs=want_obs)
            out = {"rewards": r, "obs": o}
        else:
            out = env.replay_episode(a.to(DEV), customer_demand=demand, want_obs=want_obs, want_rewards=True, stats=True)
        torch.cuda.synchronize()
        res[act] = ({k: v.clone() for k, v in out.items() if v is not None}, _state(env), env._lib.imx_kernel_variant(env._handle))
    assert res["float32"][2] == (2 if call == "step_many" else 4)      # the fused multi-period / episode kernel
    assert sorted(res["float32"][0]) == sorted(res["float64"][0])
    for k in res["float64"][0]:
        _eq(res["float32"][0][k], res["float64"][0][k], k)
    for k in res["float64"][1]:
        _eq(res["float32"][1][k], res["float64"][1][k], k)


@pytest.mark.parametrize("fuse", ["1", "0"])
@pytest.mark.parametrize("kind,preset", [("MAIM", "serial4"), ("IM", "serial4_dfo"), ("MAIM_div", "div2"), ("IM_div", "div1")])
def test_replay_episode_on_the_episode_kernel_and_the_composition(kind, preset, fuse, monkeypatch):
    monkeypatch.setenv("IMX_FUSE_PERIODS", fuse)
    cfg, n = presets.PRESETS[preset](), 4096
    demand, a32 = _trace(kind, cfg, n, 7)
    env_b = _make(kind, cfg, n, "bfloat16", "float32")
    rb = env_b.replay_episode(a32.to(DEV), customer_demand=demand, want_obs=True, want_rewards=True, stats=True, eval_acc=True)
    variant = env_b._lib.imx_kernel_variant(env_b._handle)
    env_f = _make(kind, cfg, n, "float32", "float64")
    rf = env_f.replay_episode(a32.double().to(DEV), customer_demand=demand, want_obs=True, want_rewards=True, stats=True)
    torch.cuda.synchronize()
    if fuse == "1" and kind in ("MAIM", "IM"):
        assert variant == 4                          # the one-launch episode kernel
    if fuse == "0":
        assert variant != 4
    _eq_bf16(rb["obs"], rf["obs"], "obs")
    for k in ("rewards", "returns", "stats"):
        _eq(rb[k], rf[k], k)
    # the accumulators: a float64 handle's evaluation loop fed the bfloat16 observations widened to float64
    env_d = _make(kind, cfg, n, "float64", "float64")
    env_d.reset(customer_demand=demand)
    _, rew, _, info = env_d.step_many(a32.double().to(DEV), return_info=True, want_obs=False)
    acc = None
    for t in range(cfg["num_periods"]):
        acc = env_d.eval_accumulate(acc, rb["obs"][t].double(), rew[t], info["profit"][t], reset=(t == 0))
    torch.cuda.synchronize()
    _eq(rb["eval"], acc, "eval accumulators")
    _eq(_state(env_b)["inv"], _state(env_d)["inv"])


@pytest.mark.parametrize("n", [97, 4096])
@pytest.mark.parametrize("preset", ["serial4", "serial2", "div2"])
def test_step_cc_rows_and_cc_observe(preset, n):
    kind = "MAIM_div" if preset.startswith("div") else "MAIM"
    cfg = presets.PRESETS[preset]()
    demand, a32 = _trace(kind, cfg, n, 8)
    a32 = a32 * 1.4                                  # beyond the clip interval
    envs = {"b": _make(kind, cfg, n, "bfloat16", "float32"), "f": _make(kind, cfg, n, "float32", "float64")}
    for e in envs.values():
        e.reset(customer_demand=demand)
    for t in range(cfg["num_periods"]):
        ob, cb, rb, _ = envs["b"].step_cc(a32[t].to(DEV), fill_actions=(t % 2 == 0))
        of, cf, rf, _ = envs["f"].step_cc(a32[t].double().to(DEV), fill_actions=(t % 2 == 0))
        _eq_bf16(ob, of, f"obs t={t}")
        _eq_bf16(cb, cf, f"critic rows t={t}")
        _eq(rb, rf, f"rewards t={t}")
    # the stand-alone gather: bfloat16 rows (out_is_f32 = 2) from bfloat16 observations, and from the float32 handle's
    rows_b = cc_observe(envs["b"], envs["b"].last_obs, a32[0].to(DEV), clip=(-1.0, 1.0), dtype=torch.bfloat16)
    rows_f = cc_observe(envs["f"], envs["f"].last_obs, a32[0].double().to(DEV), clip=(-1.0, 1.0), dtype=torch.float32)
    _eq_bf16(rows_b, rows_f, "cc_observe bfloat16 rows")
    _eq(cc_observe(envs["f"], envs["f"].last_obs, a32[0].double().to(DEV), dtype=torch.bfloat16), rows_f.to(torch.bfloat16))
    torch.cuda.synchronize()


@pytest.mark.parametrize("zero_copy", ["1", "0"])
def test_host_buffer_path(zero_copy, monkeypatch):
    monkeypatch.setenv("IMX_HOST_ZERO_COPY", zero_copy)
    cfg, N = presets.serial4(), 4096 + 64
    demand, a32 = _trace("MAIM", cfg, N, 9)
    o32, r64, _, _ = _episode(_make("MAIM", cfg, N, "float32"), demand, a32.double())
    env = _make("MAIM", cfg, N, "bfloat16", "float32")
    m, O, T = env.num_nodes, env.obs_len, env.num_periods
    dem_h, act_h = torch.as_tensor(demand).pin_memory(), a32.contiguous().pin_memory()
    obs_h = torch.empty((N, m, O), dtype=torch.bfloat16).pin_memory()
    rew_h = torch.empty((N, m), dtype=torch.float64).pin_memory()
    p = lambda a: C.c_void_p(a.data_ptr())   # noqa: E731
    _lib.check(env._lib.imx_reset_host(env._handle, p(dem_h), None, 0, 3, p(obs_h)))
    _eq_bf16(obs_h, o32[0], "reset")
    for t in range(T):
        _lib.check(env._lib.imx_step_host(env._handle, p(act_h[t]), p(obs_h), p(rew_h)))
        _eq_bf16(obs_h, o32[t + 1], f"t={t}")
        _eq(rew_h, r64[t].cpu(), f"t={t}")


@pytest.mark.parametrize("kind,preset", [("MAIM", "serial4"), ("IM", "serial4"), ("MAIM_div", "div2")])
def test_eval_accumulate_reads_bf16(kind, preset):
    cfg, n = presets.PRESETS[preset](), 4097
    demand, a32 = _trace(kind, cfg, n, 10)
    ob, rb, _, _ = _episode(_make(kind, cfg, n, "bfloat16", "float32"), demand, a32)
    env_b, env_d = _make(kind, cfg, n, "bfloat16", "float32"), _make(kind, cfg, n, "float64")
    acc_b = acc_d = None
    for t in range(cfg["num_periods"]):
        acc_b = env_b.eval_accumulate(acc_b, ob[t + 1], rb[t], reset=(t == 0))
        acc_d = env_d.eval_accumulate(acc_d, ob[t + 1].double(), rb[t], reset=(t == 0))
    torch.cuda.synchronize()
    _eq(acc_b, acc_d)


def test_both_types_under_graph_capture():
    kind, cfg, N, K = "MAIM", presets.serial4(), 8192, 6
    demand, a32 = _trace(kind, cfg, N, 12)
    env = _make(kind, cfg, N, "bfloat16", "float32")
    lib, h = env._lib, env._handle
    _lib.check(lib.imx_prepare(h, 0))
    m, O = env.num_nodes, env.obs_len
    dem, act = torch.as_tensor(demand, device=DEV), a32[:K].to(DEV).contiguous()
    obs = torch.zeros((K, N, m, O), dtype=torch.bfloat16, device=DEV)
    rew = torch.zeros((K, N, m), dtype=torch.float64, device=DEV)
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            _lib.check(lib.imx_reset(h, C.c_void_p(dem.data_ptr()), None, 0, 1, None, s))
            for t in range(K):
                _lib.check(lib.imx_step(h, C.c_void_p(act[t].data_ptr()), C.c_void_p(obs[t].data_ptr()), C.c_void_p(rew[t].data_ptr()), None, s))
    torch.cuda.current_stream().wait_stream(side)
    assert lib.imx_kernel_variant(h) in (2, 3)
    for _ in range(2):
        g.replay()
    torch.cuda.synchronize()
    o32, r64, _, _ = _episode(_make(kind, cfg, N, "float32"), demand, a32.double())
    _eq_bf16(obs, o32[1:K + 1])
    _eq(rew, r64[:K])


@pytest.mark.parametrize("preset,n,offset", [("serial4", 4095, 0), ("serial4", 4097, 0), ("serial4", 4098, 0), ("serial4", 4096, 2),
                                             ("serial5", 4096, 0), ("serial5", 4100, 0), ("serial5", 4101, 2), ("serial5", 97, 2)])
def test_sentinel_bracketed_caller_buffers(preset, n, offset):
    """Outputs written into caller buffers that sit between sentinel bytes: whole tiles +- 1, N % 4 != 0, pointers off 16-byte
    alignment by 2 (observations) / 4 (actions) bytes, and the 5 x 5 network whose bfloat16 warp tile is 200 bytes."""
    kind = "MAIM"
    cfg = _cfg(preset, {})
    demand, a32 = _trace(kind, cfg, n, 13)
    env = _make(kind, cfg, n, "bfloat16", "float32")
    lib, h = env._lib, env._handle
    m, O, T = env.num_nodes, env.obs_len, env.num_periods
    pad = 64
    obs_bytes, act_bytes, rew_bytes = n * m * O * 2, n * m * 4, n * m * 8
    big = torch.full((obs_bytes + act_bytes + rew_bytes + 8 * pad,), 0xA5, dtype=torch.uint8, device=DEV)
    o0 = pad + offset
    a0 = (o0 + obs_bytes + 2 * pad + 15) // 16 * 16 + 2 * offset
    r0 = (a0 + act_bytes + 2 * pad + 15) // 16 * 16
    obs_v = big[o0:o0 + obs_bytes]
    act_v = big[a0:a0 + act_bytes]
    rew_v = big[r0:r0 + rew_bytes]
    outside = torch.ones_like(big, dtype=torch.bool)
    for s_, ln in ((o0, obs_bytes), (a0, act_bytes), (r0, rew_bytes)):
        outside[s_:s_ + ln] = False
    o32, r64, _, _ = _episode(_make(kind, cfg, n, "float32"), demand, a32.double())
    env.reset(customer_demand=demand)
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for t in range(T):
        act_v.copy_(a32[t].contiguous().view(torch.uint8).reshape(-1).to(DEV))
        _lib.check(lib.imx_step(h, C.c_void_p(act_v.data_ptr()), C.c_void_p(obs_v.data_ptr()), C.c_void_p(rew_v.data_ptr()), None, s))
        torch.cuda.synchronize()
        got_o = obs_v.cpu().view(torch.bfloat16).reshape(n, m, O)
        got_r = rew_v.cpu().view(torch.float64).reshape(n, m)
        _eq_bf16(got_o, o32[t + 1], f"obs t={t}")
        _eq(got_r, r64[t], f"rewards t={t}")
        assert bool((big[outside] == 0xA5).all()), f"a sentinel byte changed at t={t}"
