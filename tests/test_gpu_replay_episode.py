"""imx_replay_episode (a whole stored-plan episode in one launch) against the composition it replaces — reset + step_many +
episode_stats + eval_accumulate per period — byte for byte on every output, the final state, the error flags and the period;
on replayed and Philox demand (sharded too), noisy delays, the reference-generated evaluation fixture, accumulated statistics,
CUDA-graph replay, sentinel-bracketed buffers and the error paths."""
import ctypes as C

import numpy as np
import pytest
import torch

from harness import copy_config
from marl_for_im_b200 import _lib, presets
from marl_for_im_b200.envs import ENV_CLASSES

pytestmark = pytest.mark.gpu

NETS = [("MAIM", "serial4"), ("IM", "serial8"), ("MAIM_div", "div2"), ("IM_div", "div1"), ("MAIM", "serial2")]
# output sets: (want_obs, want_rewards, returns, stats, eval_acc, obs_dtype)
OUTPUTS = {"all": (True, True, True, True, True, "float64"), "scoring": (False, False, True, True, False, "float64"),
           "obs_only": (True, False, False, False, False, "float64"), "eval_only": (False, False, False, False, True, "float64"),
           "all_f32": (True, True, True, True, True, "float32")}
FUSED_N = (4096, 65536, 262144)          # whole tiles of every family's specialised kernel; 96 / 100: no specialisation, 4132: a tail


def _fused(preset, n, want_obs):
    """Where the episode kernel serves (imx_replay_episode's dispatch): whole tiles of the specialised build, and for the
    divergent networks the measured rule — div2 (env-per-thread body) with observations, div1 (lane-mapped) without."""
    if n not in FUSED_N:
        return False
    return {"div2": want_obs, "div1": not want_obs}.get(preset, True)


def _inputs(kind, cfg, n, seed):
    env = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=4))
    m, T, R = env.num_nodes, env.num_periods, len(env._retailers)
    g = torch.Generator(device="cuda:0")
    g.manual_seed(seed)
    demand = torch.poisson(torch.full((n, R, T), 5.0, device="cuda:0"), generator=g).to(torch.int32)
    if kind.endswith("div"):
        actions = (torch.randn((T, n, m), dtype=torch.float64, device="cuda:0", generator=g) * 0.5 - 0.6).clamp(-1, 1)
    else:
        actions = torch.rand((T, n, m), dtype=torch.float64, device="cuda:0", generator=g) * 2.3 - 1.15
    return demand, actions


def _composed(env, actions, demand=None, delay_mask=None, stats=None):
    """The composition on `env`: reset + step_many (with the profit diagnostics) + episode_stats + eval_accumulate."""
    env.reset(customer_demand=demand, delay_mask=delay_mask)
    o, r, _, info = env.step_many(actions, return_info=True)
    ret = torch.empty_like(r[0])
    st = env.episode_stats(r, returns=ret, stats=stats, accumulate=stats is not None)
    acc = None
    for t in range(env.num_periods):
        acc = env.eval_accumulate(acc, o[t], r[t], info["profit"][t], reset=(t == 0))
    return {"obs": o, "rewards": r, "returns": ret, "stats": st, "eval": acc}


def _snapshot(env):
    state = {k: v.clone() for k, v in env.state_dict().items()}
    return state, env.error_flags.clone(), env.period


def _assert_same_env(a, b, what):
    sa, ea, pa = _snapshot(a)
    sb, eb, pb = _snapshot(b)
    assert sa.keys() == sb.keys() and pa == pb, what
    for k in sa:
        assert torch.equal(sa[k], sb[k]), (what, k)
    assert torch.equal(ea, eb), what


def _assert_outputs(got, want, keys, what):
    for k in keys:
        if got[k] is None:
            continue
        assert torch.equal(got[k], want[k]), (what, k)


@pytest.mark.parametrize("out", sorted(OUTPUTS))
@pytest.mark.parametrize("n", [96, 100, 4096, 4096 + 36, 65536, 262144])
@pytest.mark.parametrize("kind,preset", NETS)
def test_equals_composition(kind, preset, n, out):
    if n == 262144 and preset != "div2":
        pytest.skip("the 262 144-env batch is run for div2 (config 4's size)")
    want_obs, want_rew, want_ret, want_stats, want_eval, dtype = OUTPUTS[out]
    cfg = presets.PRESETS[preset]()
    demand, actions = _inputs(kind, cfg, n, seed=n + len(out))
    ref = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n, obs_dtype=dtype))
    want = _composed(ref, actions, demand)
    env = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n, obs_dtype=dtype))
    env.step_many(actions[:7])                                 # mid-episode: the call is a reset
    got = env.replay_episode(actions, customer_demand=demand, want_obs=want_obs, want_rewards=want_rew, returns=want_ret,
                             stats=True if want_stats else None, eval_acc=want_eval)
    for k, on in (("obs", want_obs), ("rewards", want_rew), ("returns", want_ret), ("stats", want_stats), ("eval", want_eval)):
        assert (got[k] is not None) == on, k
    _assert_outputs(got, want, ("obs", "rewards", "returns", "stats", "eval"), (kind, n, out))
    _assert_same_env(env, ref, (kind, n, out))
    variant = env._lib.imx_kernel_variant(env._handle)
    assert (variant == 4) == _fused(preset, n, want_obs), (kind, n, out, variant)
    if want_obs:
        assert torch.equal(env.last_obs, want["obs"][-1])


@pytest.mark.parametrize("kind,preset,extra", [("MAIM", "serial4", {}), ("IM_div", "div1", {}),
                                               ("MAIM_div", "div2", {"noisy_demand": True, "noisy_demand_threshold": 0.2})])
def test_philox_demand_and_sharding(kind, preset, extra):
    """customer_demand=None draws the stream reset(None) draws for the same episode id; two half handles with env_offset 0
    and N/2 give the full handle's outputs."""
    cfg = dict(presets.PRESETS[preset](), **extra)
    n = 8192
    _, actions = _inputs(kind, cfg, n, seed=11)
    ref = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    want = _composed(ref, actions)                             # reset(None): episode 2 of the handle
    env = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    got = env.replay_episode(actions, want_obs=True, want_rewards=True, stats=True, eval_acc=True)
    assert (env._lib.imx_kernel_variant(env._handle) == 4) == _fused(preset, 4096, True)
    _assert_outputs(got, want, ("obs", "rewards", "returns", "stats", "eval"), kind)
    _assert_same_env(env, ref, kind)
    half = n // 2
    for k, off in enumerate((0, half)):
        part = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=half, env_offset=off))
        g = part.replay_episode(actions[:, off:off + half].contiguous(), want_obs=True, want_rewards=True, eval_acc=True)
        assert (part._lib.imx_kernel_variant(part._handle) == 4) == _fused(preset, 4096, True)
        for key in ("obs", "rewards"):
            assert torch.equal(g[key], got[key][:, off:off + half]), (kind, k, key)
        for key in ("returns", "eval"):
            assert torch.equal(g[key], got[key][off:off + half]), (kind, k, key)
        for f, v in part.state_dict().items():
            assert torch.equal(v, env.state_dict()[f][off:off + half]), (kind, k, f)


@pytest.mark.parametrize("kind,preset", [("MAIM", "serial8"), ("MAIM_div", "div2")])
@pytest.mark.parametrize("n", [4096, 100])
def test_noisy_delay(kind, preset, n):
    """Replayed and Philox-drawn noisy-delay outcomes (the carry state lives in the tile like the rest of the state)."""
    cfg = dict(presets.PRESETS[preset](), noisy_delay=True, noisy_delay_threshold=0.3)
    demand, actions = _inputs(kind, cfg, n, seed=5)
    ref = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    env = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    T, m = ref.num_periods, ref.num_nodes
    mask = torch.rand((n, T, m), device="cuda:0") < 0.3
    want = _composed(ref, actions, demand, delay_mask=mask)
    got = env.replay_episode(actions, customer_demand=demand, delay_mask=mask, want_obs=True, want_rewards=True, stats=True, eval_acc=True)
    _assert_outputs(got, want, ("obs", "rewards", "returns", "stats", "eval"), (kind, "mask"))
    _assert_same_env(env, ref, (kind, "mask"))
    assert (env._lib.imx_kernel_variant(env._handle) == 4) == _fused(preset, n, True)
    # Philox outcomes: both handles switched to noisy episodes with the same threshold by a noisy reset (sticky flag)
    ref.reset(noisy_delay=True, noisy_delay_threshold=0.3)
    env.reset(noisy_delay=True, noisy_delay_threshold=0.3)
    want = _composed(ref, actions, demand)
    got = env.replay_episode(actions, customer_demand=demand, want_obs=True, want_rewards=True, stats=True, eval_acc=True)
    _assert_outputs(got, want, ("obs", "rewards", "returns", "stats", "eval"), (kind, "philox"))
    _assert_same_env(env, ref, (kind, "philox"))


def test_eval_accumulators_match_reference_fixture():
    """The evaluation loops' accumulators generated from the reference (tests/golden/evalloop): every case's six episodes
    tiled up to a batch the episode kernel serves, every copy equal to the fixture."""
    from test_eval_loop_golden import CASES, case_config
    for kind, preset, kw, rescaled, demand, actions, want in CASES:
        cfg = case_config(preset, kw)
        reps = 704                                             # N = 4224 = 66 x 64: whole tiles of every family
        N = demand.shape[0] * reps
        dem = np.repeat(demand, reps, axis=0).astype(np.int32)
        act = torch.as_tensor(np.ascontiguousarray(np.repeat(actions, reps, axis=0).transpose(1, 0, 2)), device="cuda:0")
        env = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=N))
        got = env.replay_episode(act, customer_demand=dem, returns=False, eval_acc=True)
        assert (env._lib.imx_kernel_variant(env._handle) == 4) == _fused(preset, 4096, False), (kind, preset)
        np.testing.assert_array_equal(got["eval"].cpu().numpy(), np.repeat(want, reps, axis=0), err_msg=f"{kind}-{preset}")
        summ = env.eval_summary(env.eval_stats(got["eval"]), env.num_nodes)
        np.testing.assert_allclose(summ["episode_reward"][0], want[:, 0].mean(), rtol=1e-12)


@pytest.mark.parametrize("kind,preset,n", [("MAIM", "serial4", 65536), ("IM_div", "div1", 100)])
def test_statistics_accumulate_over_episodes(kind, preset, n):
    cfg = presets.PRESETS[preset]()
    ref = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    env = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    want, got = None, None
    for ep in range(3):
        demand, actions = _inputs(kind, cfg, n, seed=40 + ep)
        want = _composed(ref, actions, demand, stats=want)["stats"]
        got = env.replay_episode(actions, customer_demand=demand, returns=False, stats=got if got is not None else True,
                                 accumulate=ep > 0)["stats"]
    assert torch.equal(got, want) and got[0] == 3 * n


def test_cuda_graph_replay_and_launch_count():
    kind, cfg, n = "MAIM", presets.serial4(), 65536
    demand, actions = _inputs(kind, cfg, n, seed=1)
    ref = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    want = _composed(ref, actions, demand)
    env = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    lib, h = env._lib, env._handle
    _lib.check(lib.imx_prepare(h, _lib.PREPARE_EPISODE))
    T, m, O = env.num_periods, env.num_nodes, env.obs_len
    obs = torch.empty((T, n, m, O), dtype=torch.float64, device="cuda:0")
    rew = torch.empty((T, n, m), dtype=torch.float64, device="cuda:0")
    ret = torch.empty((n, m), dtype=torch.float64, device="cuda:0")
    stats = torch.empty(3 + 2 * m, dtype=torch.float64, device="cuda:0")
    ev = torch.empty((n, 4 + m), dtype=torch.float64, device="cuda:0")
    p = lambda x: C.c_void_p(x.data_ptr()) if x is not None else None   # noqa: E731

    def episode(stream, with_stats=True):
        _lib.check(lib.imx_replay_episode(h, p(demand), None, 0, 2, p(actions), p(obs), p(rew), p(ret), p(stats) if with_stats else None,
                                          0, p(ev), C.c_void_p(stream)))
    s = torch.cuda.current_stream().cuda_stream
    c0 = env.launch_count()
    episode(s, with_stats=False)
    c1 = env.launch_count()
    episode(s)
    c2 = env.launch_count()
    assert (c1 - c0, c2 - c1) == (1, 3) and lib.imx_kernel_variant(h) == 4
    side = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            episode(torch.cuda.current_stream().cuda_stream)
    torch.cuda.current_stream().wait_stream(side)
    for rep in range(25):
        for x in (obs, rew, ret, stats, ev):
            x.zero_()
        g.replay()
        torch.cuda.synchronize()
        for k, x in (("obs", obs), ("rewards", rew), ("returns", ret), ("stats", stats), ("eval", ev)):
            assert torch.equal(x, want[k]), (rep, k)
    _assert_same_env(env, ref, "graph")


@pytest.mark.parametrize("with_io", [False, True])
@pytest.mark.parametrize("n,offset", [(4096, 0), (4096 + 1, 0), (4096 - 1, 0), (4096 + 4, 0), (4096, 8)])
def test_nothing_written_outside_the_requested_buffers(n, offset, with_io):
    """Every caller buffer sits between sentinel bytes; `offset` = 8 bytes breaks the 16-byte alignment (the composition
    serves).  Without obs / reward buffers (NULL) nothing else is touched; with them, nothing lands beyond their ends."""
    kind, cfg = "MAIM", presets.serial4()
    demand, actions = _inputs(kind, cfg, n, seed=7)
    ref = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    want = _composed(ref, actions, demand)
    env = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    T, m, O = env.num_periods, env.num_nodes, env.obs_len
    pad = 512
    nbytes = {"returns": n * m * 8, "stats": (3 + 2 * m) * 8, "eval": n * (4 + m) * 8}
    if with_io:
        nbytes.update({"obs": T * n * m * O * 8, "rewards": T * n * m * 8})
    raw = {k: torch.full((b + 2 * pad + offset,), 0x5A, dtype=torch.uint8, device="cuda:0") for k, b in nbytes.items()}
    ptr = {k: C.c_void_p(raw[k].data_ptr() + pad + offset) for k in nbytes}
    act = torch.empty((actions.numel() * 8 + offset,), dtype=torch.uint8, device="cuda:0")
    act[offset:].copy_(actions.reshape(-1).view(torch.uint8))
    _lib.check(env._lib.imx_replay_episode(env._handle, C.c_void_p(demand.data_ptr()), None, 0, 2, C.c_void_p(act.data_ptr() + offset),
                                           ptr.get("obs"), ptr.get("rewards"), ptr["returns"], ptr["stats"], 0, ptr["eval"],
                                           C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    for k, b in nbytes.items():
        r = raw[k]
        assert bool((r[:pad + offset] == 0x5A).all()) and bool((r[pad + offset + b:] == 0x5A).all()), (n, offset, k)
        assert torch.equal(r[pad + offset:pad + offset + b], want[k].reshape(-1).view(torch.uint8)), (n, offset, k)
    _assert_same_env(env, ref, (n, offset))
    assert (env._lib.imx_kernel_variant(env._handle) == 4) == (n == 4096 and offset == 0)


def test_errors_and_mid_episode_call():
    kind, cfg, n = "MAIM", presets.serial4(), 4096
    demand, actions = _inputs(kind, cfg, n, seed=3)
    env = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    lib, h = env._lib, env._handle
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ret = torch.empty((n, 4), dtype=torch.float64, device="cuda:0")
    p = lambda x: C.c_void_p(x.data_ptr())                    # noqa: E731
    assert lib.imx_replay_episode(h, p(demand), None, 0, 1, None, None, None, p(ret), None, 0, None, s) == -1      # null actions
    assert b"null argument" in lib.imx_last_error()
    assert lib.imx_replay_episode(None, p(demand), None, 0, 1, p(actions), None, None, p(ret), None, 0, None, s) == -1
    assert lib.imx_replay_episode(h, p(demand), None, 1, 1, p(actions), None, None, p(ret), None, 0, None, s) == -1   # no carry
    assert b"noisy_delay = 0" in lib.imx_last_error()
    replay_only = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n, demand_dist="custom"))
    assert replay_only._lib.imx_replay_episode(replay_only._handle, None, None, 0, 1, p(actions), None, None, p(ret), None, 0, None, s) == -1
    assert b"poisson or uniform" in lib.imx_last_error()
    # a scratch buffer the call would have to allocate while the stream is captured: the composition's reward buffer
    # (a batch with a tail tile), never prepared
    tail = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n + 4))
    d2, a2 = _inputs(kind, cfg, n + 4, seed=4)
    r2 = torch.empty((n + 4, 4), dtype=torch.float64, device="cuda:0")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    rc = []
    with torch.cuda.stream(side):
        g = torch.cuda.CUDAGraph()
        try:
            with torch.cuda.graph(g, stream=side):
                rc.append(tail._lib.imx_replay_episode(tail._handle, p(d2), None, 0, 1, p(a2), None, None, p(r2), None, 0, None,
                                                       C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        except RuntimeError:
            pass                                                  # an empty capture may be rejected by torch: the code is what counts
    torch.cuda.current_stream().wait_stream(side)
    assert rc == [-1] and b"IMX_PREPARE_EPISODE" in lib.imx_last_error()
    # from mid-episode (period 7) the call behaves as a reset
    ref = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    want = _composed(ref, actions, demand)
    env.reset(customer_demand=demand)
    env.step_many(actions[:7])
    assert env.period == 7
    got = env.replay_episode(actions, customer_demand=demand, want_rewards=True, stats=True)
    _assert_outputs(got, want, ("rewards", "returns", "stats"), "mid-episode")
    _assert_same_env(env, ref, "mid-episode")
    with pytest.raises(_lib.ImxError):
        ENV_CLASSES[kind](dict(copy_config(cfg))).replay_episode(actions[:, :1])
