"""imx_step_eval (a step with its period's returns, evaluation accumulators and diagnostics) against what it replaces: the
stored-plan episode (replay_episode) bit for bit when driven by the plan's actions, and the per-period composition
step(return_info=True) + eval_accumulate + the returns add on a twin handle, every period; plus closed loops (base-stock
levels, a torch policy reading the observations), episodes in a row, CUDA-graph capture, sentinel-bracketed buffers and the
error paths."""
import ctypes as C

import pytest
import torch

from harness import copy_config
from marl_for_im_b200 import _lib, presets
from marl_for_im_b200.base_restock_policy import base_stock_policy
from marl_for_im_b200.envs import ENV_CLASSES

pytestmark = pytest.mark.gpu

NETS = [("MAIM", "serial2", {"independent": True}), ("MAIM", "serial4", {}), ("IM", "serial8", {}), ("IM", "serial4_dfo", {}),
        ("IM_div", "div1", {}), ("MAIM_div", "div1", {}), ("MAIM_div", "div2", {})]
INFO_KEYS = ("demand", "ship", "acquisition", "actual order", "profit")


def _inputs(env, n, seed):
    m, T, R = env.num_nodes, env.num_periods, len(env._retailers)
    g = torch.Generator(device="cuda:0")
    g.manual_seed(seed)
    demand = torch.poisson(torch.full((n, R, T), 5.0, device="cuda:0"), generator=g).to(torch.int32)
    if env.DIV:
        actions = (torch.randn((T, n, m), dtype=torch.float64, device="cuda:0", generator=g) * 0.5 - 0.6).clamp(-1, 1)
    else:
        actions = torch.rand((T, n, m), dtype=torch.float64, device="cuda:0", generator=g) * 2.3 - 1.15
    if not getattr(env, "standardise_actions", True) and env.KIND != "MAIM_div":
        actions = (actions + 1.2) * 10.0
    return demand, actions


def _make(kind, preset, n, **extra):
    cfg = dict(presets.PRESETS[preset](), **extra)
    return ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))


def _snapshot(env):
    return {k: v.clone() for k, v in env.state_dict().items()}, env.error_flags.clone(), env.period


def _assert_same_env(a, b, what):
    sa, ea, pa = _snapshot(a)
    sb, eb, pb = _snapshot(b)
    assert sa.keys() == sb.keys() and pa == pb, what
    for k in sa:
        assert torch.equal(sa[k], sb[k]), (what, k)
    assert torch.equal(ea, eb), what


@pytest.mark.parametrize("n", [4096, 65536, 4096 + 36, 1000])
@pytest.mark.parametrize("kind,preset,extra", NETS)
def test_open_loop_equals_replay_episode(kind, preset, extra, n):
    """evaluate_policy(lambda obs, t: plan[t]) == replay_episode(plan): returns, statistics, accumulators, rewards, final
    state, watchdog flags and period, bit for bit; the kernel that served is the one the batch size selects."""
    ref = _make(kind, preset, n, **extra)
    env = _make(kind, preset, n, **extra)
    demand, plan = _inputs(ref, n, seed=n + len(preset))
    want = ref.replay_episode(plan, customer_demand=demand, want_rewards=True, stats=True, eval_acc=True)
    got = env.evaluate_policy(lambda obs, t: plan[t], customer_demand=demand, stats=True, eval_acc=True, want_rewards=True)
    for k in ("returns", "stats", "eval", "rewards"):
        assert torch.equal(got[k], want[k]), (kind, preset, n, k)
    _assert_same_env(env, ref, (kind, preset, n))
    variant = env._lib.imx_kernel_variant(env._handle)
    assert (variant in (2, 3)) == (n in (4096, 65536)), (kind, preset, n, variant)


def test_misaligned_buffers_take_the_composition():
    kind, preset, n = "MAIM", "serial4", 4096
    ref, env = _make(kind, preset, n), _make(kind, preset, n)
    demand, plan = _inputs(ref, n, seed=3)
    want = ref.replay_episode(plan, customer_demand=demand, eval_acc=True)
    m = env.num_nodes
    raw = torch.zeros(n * m + 1, dtype=torch.float64, device="cuda:0")
    ret = raw[1:].view(n, m)                                   # 8 bytes off a 16-byte boundary
    ev = torch.empty((n, 4 + m), dtype=torch.float64, device="cuda:0")
    env.reset(customer_demand=demand)
    for t in range(env.num_periods):
        env.step_eval(plan[t], returns=ret, eval_acc=ev, want_obs=False, want_rewards=False)
        assert env._lib.imx_kernel_variant(env._handle) in (0, 1)
    assert torch.equal(ret, want["returns"]) and torch.equal(ev, want["eval"])
    _assert_same_env(env, ref, "misaligned")


def _twin_run(kind, preset, n, extra=None, env_vars=None, monkeypatch=None, io=None, want=(True, True, True, True, INFO_KEYS),
              noisy=None, policy=None, seed=1):
    """Every period: env.step_eval(...) against twin.step(return_info=True) + eval_accumulate + the returns add."""
    if env_vars:
        for k, v in env_vars.items():
            monkeypatch.setenv(k, v)
    io = io or {}
    env = _make(kind, preset, n, **dict(extra or {}, **io))
    twin = _make(kind, preset, n, **dict(extra or {}, **io))
    demand, plan = _inputs(env, n, seed)
    want_obs, want_rew, want_ret, want_ev, info_keys = want
    m, T = env.num_nodes, env.num_periods
    cols = (n, m) if env.MULTI else (n,)
    mask = None
    if noisy == "replay":
        mask = torch.rand((n, T, m), device="cuda:0") < 0.3
    for e in (env, twin):
        e.reset(customer_demand=demand, delay_mask=mask, noisy_delay=noisy == "philox", noisy_delay_threshold=0.3)
    ret = torch.full(cols, 7.0, dtype=torch.float64, device="cuda:0") if want_ret else None
    ev = torch.full((n, 4 + m), 7.0, dtype=torch.float64, device="cuda:0") if want_ev else None
    tret, tev, obs = None, None, env.last_obs
    variants = set()
    for t in range(T):
        act = plan[t] if policy is None else policy(obs, t)
        info = {k: torch.full((n, m), -3, dtype=torch.float64 if k == "profit" else torch.int32, device="cuda:0") for k in info_keys}
        obs_buf = torch.empty((n, m, env.obs_len), dtype=env.obs_dtype, device="cuda:0") if want_obs else None
        rew_buf = torch.empty(cols, dtype=torch.float64, device="cuda:0") if want_rew else None
        struct = _lib.ImxInfoOut(**{f: (info[k].data_ptr() if k in info else None) for k, (f, _) in env.INFO_FIELDS.items()})
        p = lambda x: C.c_void_p(x.data_ptr()) if x is not None else None   # noqa: E731
        act_d = env._actions_to_device(act)
        _lib.check(env._lib.imx_step_eval(env._handle, p(act_d), p(obs_buf), p(rew_buf), C.byref(struct) if info_keys else None,
                                          p(ret), p(ev), env._stream()))
        variants.add(env._lib.imx_kernel_variant(env._handle))
        tobs, trew, _, tinfo = twin.step_many(twin._actions_to_device(act).unsqueeze(0), return_info=True)
        tobs, trew = tobs[0], trew[0]
        tret = trew.clone() + 0.0 if tret is None else tret + trew
        tev = twin.eval_accumulate(tev, tobs, trew, tinfo["profit"][0], reset=(t == 0))
        if want_obs:
            assert torch.equal(obs_buf, tobs), (t, "obs")
        if want_rew:
            assert torch.equal(rew_buf, trew), (t, "reward")
        for k in info_keys:
            assert torch.equal(info[k], tinfo[k][0].to(info[k].dtype)), (t, k)
        if want_ret:
            assert torch.equal(ret, tret), (t, "returns")
        if want_ev:
            assert torch.equal(ev, tev), (t, "eval")
        _assert_same_env(env, twin, t)
        obs = tobs
    return variants


@pytest.mark.parametrize("pipe", ["0", "1"])
@pytest.mark.parametrize("kind,preset", [("MAIM", "serial4"), ("IM", "serial8"), ("MAIM_div", "div2"), ("IM_div", "div1")])
def test_every_period_against_the_composition(kind, preset, pipe, monkeypatch):
    v = _twin_run(kind, preset, 4096, env_vars={"IMX_PIPE": pipe}, monkeypatch=monkeypatch)
    assert v == {3 if pipe == "1" else 2}, v


@pytest.mark.parametrize("pipe", ["0", "1"])
@pytest.mark.parametrize("et", ["0", "1"])
def test_div2_period_bodies(et, pipe, monkeypatch):
    v = _twin_run("MAIM_div", "div2", 4096, env_vars={"IMX_STEP_ET": et, "IMX_PIPE": pipe}, monkeypatch=monkeypatch)
    assert v == {3 if pipe == "1" else 2}, v


@pytest.mark.parametrize("hints", ["0", "1", "2"])
def test_l2_hint_modes(hints, monkeypatch):
    assert _twin_run("MAIM", "serial4", 65536, env_vars={"IMX_L2_HINTS": hints, "IMX_PIPE": "1"}, monkeypatch=monkeypatch) == {3}


@pytest.mark.parametrize("act", ["float64", "float32"])
@pytest.mark.parametrize("obs", ["float64", "float32", "bfloat16"])
def test_io_types(obs, act):
    if obs == "bfloat16" and act == "float64":
        io = {"obs_dtype": "bfloat16"}
    else:
        io = {"obs_dtype": obs, "action_dtype": act}
    for kind, preset in (("MAIM", "serial4"), ("MAIM_div", "div2")):
        assert _twin_run(kind, preset, 4096, io=io) <= {2, 3}


@pytest.mark.parametrize("noisy", ["replay", "philox"])
@pytest.mark.parametrize("kind,preset", [("MAIM", "serial8"), ("MAIM_div", "div2")])
def test_noisy_delays(kind, preset, noisy):
    _twin_run(kind, preset, 4096, extra={"noisy_delay": True, "noisy_delay_threshold": 0.3}, noisy=noisy)


@pytest.mark.parametrize("want", [
    (False, True, True, True, INFO_KEYS), (True, False, True, True, ()), (False, False, True, False, ()),
    (False, False, False, True, ()), (True, True, False, False, ("demand", "profit")), (False, False, True, True, ("ship", "acquisition")),
    (True, True, True, False, ("actual order",)), (False, False, False, False, ())])
@pytest.mark.parametrize("n", [4096, 4096 + 36])
def test_optional_outputs(want, n):
    v = _twin_run("MAIM", "serial4", n, want=want)
    if n == 4096:
        assert v <= {2, 3}, v
    elif want[3] or want[4]:                                   # the composition's step carries the profits: ahead-of-time kernels
        assert v <= {0, 1}, v


@pytest.mark.parametrize("kind,preset", [("MAIM_div", "div2"), ("IM_div", "div2")])
def test_returns_only_on_large_env_per_thread_batches_take_the_composition(kind, preset):
    """The measured rule: returns as the only bookkeeping with the env-per-thread body on a launch that streams more than half
    of L2."""
    n = 262144
    ref, env = _make(kind, preset, n), _make(kind, preset, n)
    demand, plan = _inputs(ref, n, seed=13)
    want = ref.replay_episode(plan, customer_demand=demand, eval_acc=True)
    got = env.evaluate_policy(lambda obs, t: plan[t], customer_demand=demand)
    assert torch.equal(got["returns"], want["returns"])
    assert env._lib.imx_kernel_variant(env._handle) in (2, 3)          # the plain specialised step of the composition
    ret = torch.empty_like(got["returns"])
    ev = torch.empty((n, 4 + env.num_nodes), dtype=torch.float64, device="cuda:0")
    env.reset(customer_demand=demand)
    for t in range(env.num_periods):
        env.step_eval(plan[t], returns=ret, eval_acc=ev, want_obs=False, want_rewards=False)
    assert torch.equal(ret, want["returns"]) and torch.equal(ev, want["eval"])


def test_philox_demand_under_sharding():
    kind, preset, n = "MAIM_div", "div2", 8192
    full = _make(kind, preset, n)
    _, plan = _inputs(full, n, seed=9)
    want = full.evaluate_policy(lambda obs, t: plan[t], eval_acc=True, want_rewards=True)
    half = n // 2
    for off in (0, half):
        part = ENV_CLASSES[kind](dict(copy_config(presets.div2()), num_envs=half, env_offset=off))
        got = part.evaluate_policy(lambda obs, t: plan[t][off:off + half].contiguous(), eval_acc=True, want_rewards=True)
        assert part._lib.imx_kernel_variant(part._handle) in (2, 3)
        assert torch.equal(got["returns"], want["returns"][off:off + half])
        assert torch.equal(got["eval"], want["eval"][off:off + half])
        assert torch.equal(got["rewards"], want["rewards"][:, off:off + half])
        for f, v in part.state_dict().items():
            assert torch.equal(v, full.state_dict()[f][off:off + half]), f


@pytest.mark.parametrize("kind,preset,n", [("IM", "serial4_dfo", 4096), ("IM_div", "div2", 4096), ("IM", "serial4_dfo", 1000)])
def test_base_stock_closed_loop_equals_fused_rollout(kind, preset, n):
    """base_stock_policy(z, env) reads the state every period: the closed loop through evaluate_policy equals the fused
    base-stock rollout (DFO configuration: raw order quantities, no observation or action scaling)."""
    extra = {"time_dependency": False, "prev_demand": False, "prev_actions": False, "standardise_state": False,
             "standardise_actions": False}
    env = _make(kind, preset, n, **extra)
    m, R, T = env.num_nodes, len(env._retailers), env.num_periods
    g = torch.Generator(device="cuda:0")
    g.manual_seed(21)
    demand = torch.poisson(torch.full((n, R, T), 6.0, device="cuda:0"), generator=g).to(torch.int32)
    z = torch.randint(5, 41, (n, m), generator=g, device="cuda:0").to(torch.float64)
    want = env.rollout_basestock(z, customer_demand=demand)["returns"]
    got = env.evaluate_policy(lambda obs, t: base_stock_policy(z, env), customer_demand=demand)
    assert torch.equal(got["returns"], want)


def test_torch_policy_reading_observations():
    torch.manual_seed(0)
    w = torch.randn(5, dtype=torch.float64, device="cuda:0")

    def policy(obs, t):
        o = obs.double()
        return torch.tanh(o[..., :5] @ w[:min(5, o.shape[-1])] + 0.1 * t).contiguous()
    for kind, preset in (("MAIM", "serial4"), ("MAIM_div", "div2")):
        _twin_run(kind, preset, 4096, policy=policy)


@pytest.mark.parametrize("kind,preset,n", [("MAIM", "serial4", 65536), ("IM_div", "div1", 1000)])
def test_episodes_stay_separate(kind, preset, n):
    ref, env = _make(kind, preset, n), _make(kind, preset, n)
    want_st, got_st = None, None
    for ep in range(3):
        demand, plan = _inputs(ref, n, seed=40 + ep)
        want = ref.replay_episode(plan, customer_demand=demand, stats=want_st if want_st is not None else True, accumulate=ep > 0,
                                  eval_acc=True)
        got = env.evaluate_policy(lambda obs, t: plan[t], customer_demand=demand, stats=got_st if got_st is not None else True,
                                  accumulate=ep > 0, eval_acc=True)
        want_st, got_st = want["stats"], got["stats"]
        assert torch.equal(got["returns"], want["returns"]) and torch.equal(got["eval"], want["eval"]), ep
    assert torch.equal(got_st, want_st) and got_st[0] == 3 * n


def test_cuda_graph_capture():
    kind, preset, n = "MAIM", "serial4", 65536
    env, ref = _make(kind, preset, n), _make(kind, preset, n)
    demand, plan = _inputs(env, n, seed=5)
    want = ref.replay_episode(plan, customer_demand=demand, want_rewards=True, eval_acc=True)
    lib, h = env._lib, env._handle
    # without the prepare: an error, nothing launched
    fresh = _make(kind, preset, n)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    rc = []
    ret = torch.empty((n, env.num_nodes), dtype=torch.float64, device="cuda:0")
    ev = torch.empty((n, 4 + env.num_nodes), dtype=torch.float64, device="cuda:0")
    p = lambda x: C.c_void_p(x.data_ptr()) if x is not None else None   # noqa: E731
    c0 = fresh.launch_count()
    with torch.cuda.stream(side):
        g0 = torch.cuda.CUDAGraph()
        try:
            with torch.cuda.graph(g0, stream=side):
                rc.append(fresh._lib.imx_step_eval(fresh._handle, p(plan[0]), None, None, None, p(ret), p(ev),
                                                   C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        except RuntimeError:
            pass                                               # an empty capture may be rejected by torch: the code is what counts
    torch.cuda.current_stream().wait_stream(side)
    assert rc == [-1] and b"IMX_PREPARE_EVAL" in lib.imx_last_error() and fresh.launch_count() == c0 and fresh.period == 0
    _lib.check(lib.imx_prepare(h, _lib.PREPARE_EVAL))
    T, m = env.num_periods, env.num_nodes
    rew = torch.empty((T, n, m), dtype=torch.float64, device="cuda:0")

    def episode(stream):
        _lib.check(lib.imx_reset(h, p(demand), None, 0, 2, None, C.c_void_p(stream)))
        for t in range(T):
            _lib.check(lib.imx_step_eval(h, p(plan[t]), None, p(rew[t]), None, p(ret), p(ev), C.c_void_p(stream)))
    episode(torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert torch.equal(ret, want["returns"]) and torch.equal(ev, want["eval"]) and torch.equal(rew, want["rewards"])
    g = torch.cuda.CUDAGraph()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            episode(torch.cuda.current_stream().cuda_stream)
    torch.cuda.current_stream().wait_stream(side)
    for rep in range(3):
        for x in (ret, ev, rew):
            x.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(ret, want["returns"]) and torch.equal(ev, want["eval"]) and torch.equal(rew, want["rewards"]), rep
    env._lib.imx_set_period(h, T)
    _assert_same_env(env, ref, "graph")


@pytest.mark.parametrize("n,offset", [(4096, 0), (4096 + 36, 0), (4096, 8)])
def test_nothing_written_outside_the_requested_buffers(n, offset):
    """Every caller buffer sits between sentinel bytes; offset 8 breaks the 16-byte alignment (the composition serves)."""
    kind, preset = "MAIM", "serial4"
    env, twin = _make(kind, preset, n), _make(kind, preset, n)
    demand, plan = _inputs(env, n, seed=7)
    m, O, T = env.num_nodes, env.obs_len, env.num_periods
    pad = 512
    nbytes = {"returns": n * m * 8, "eval": n * (4 + m) * 8, "obs": n * m * O * 8, "reward": n * m * 8,
              "demand": n * m * 4, "ship": n * m * 4, "acquisition": n * m * 4, "actual order": n * m * 4, "profit": n * m * 8}
    raw = {k: torch.full((b + 2 * pad + offset,), 0x5A, dtype=torch.uint8, device="cuda:0") for k, b in nbytes.items()}
    ptr = {k: raw[k].data_ptr() + pad + offset for k in nbytes}
    env.reset(customer_demand=demand)
    twin.reset(customer_demand=demand)
    tret, tev = None, None
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    struct = _lib.ImxInfoOut(*[ptr[k] for k in ("demand", "ship", "acquisition", "actual order", "profit")])
    for t in range(T):
        _lib.check(env._lib.imx_step_eval(env._handle, C.c_void_p(plan[t].data_ptr()), C.c_void_p(ptr["obs"]), C.c_void_p(ptr["reward"]),
                                          C.byref(struct), C.c_void_p(ptr["returns"]), C.c_void_p(ptr["eval"]), s))
        assert (env._lib.imx_kernel_variant(env._handle) in (2, 3)) == (n == 4096 and offset == 0)
        tobs, trew, _, tinfo = twin.step_many(plan[t].unsqueeze(0), return_info=True)
        tret = trew[0].clone() + 0.0 if tret is None else tret + trew[0]
        tev = twin.eval_accumulate(tev, tobs[0], trew[0], tinfo["profit"][0], reset=(t == 0))
        want = dict(returns=tret, eval=tev, obs=tobs[0], reward=trew[0], **{k: tinfo[k][0] for k in INFO_KEYS})
        torch.cuda.synchronize()
        for k, b in nbytes.items():
            r = raw[k]
            assert bool((r[:pad + offset] == 0x5A).all()) and bool((r[pad + offset + b:] == 0x5A).all()), (n, offset, t, k)
            assert torch.equal(r[pad + offset:pad + offset + b], want[k].contiguous().reshape(-1).view(torch.uint8)), (n, offset, t, k)
    _assert_same_env(env, twin, (n, offset))


def test_errors():
    kind, preset, n = "MAIM", "serial4", 4096
    env = _make(kind, preset, n)
    lib, h = env._lib, env._handle
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ret = torch.empty((n, 4), dtype=torch.float64, device="cuda:0")
    assert lib.imx_step_eval(h, None, None, None, None, C.c_void_p(ret.data_ptr()), None, s) == -1
    assert b"null argument" in lib.imx_last_error()
    _, plan = _inputs(env, n, seed=2)
    env.reset()
    for t in range(env.num_periods):
        env.step_eval(plan[t], returns=ret, want_obs=False)
    with pytest.raises(IndexError):
        env.step_eval(plan[0], returns=ret)
    assert lib.imx_step_eval(h, C.c_void_p(plan[0].data_ptr()), None, None, None, None, None, s) == -6
    env.reset()
    with pytest.raises(ValueError):
        env.step_eval(plan[0], returns=torch.empty((n,), dtype=torch.float64, device="cuda:0"))
    with pytest.raises(ValueError):
        env.step_eval(plan[0], returns=torch.empty((n, 4), dtype=torch.float32, device="cuda:0"))
    with pytest.raises(ValueError):
        env.step_eval(plan[0], eval_acc=torch.empty((n, 8), dtype=torch.float64, device="cuda:0")[:, ::2])
    with pytest.raises(ValueError):
        env.step_eval(plan[0], eval_acc=torch.empty((n, 8), dtype=torch.float64))
    assert env.period == 0
