"""imx_replay_episode_records / replay_episode(records=...): the reference's per-period history arrays from one call.

Against the reference: every golden episode (tests/golden/*.npz, generated from the reference) replicated over a batch, each
env's records equal to the fixture's inv / backlog / order_u / demand / ship / acq / order / profit.  Against the composition:
reset + T one-period steps with the diagnostics + state snapshots, byte for byte, on fused and unfused batch sizes, with and
without observations, Philox and replayed demand, generated and replayed noisy delays, sharding, reduced-precision I/O and
subsets of fields.  Recording changes nothing else (outputs, final state, error flags, period, launch count); record buffers
are written only inside their rows; CUDA-graph replay; a records call under capture without imx_prepare is refused."""
import ctypes as C

import numpy as np
import pytest
import torch

from harness import copy_config, golden_names, load_golden
from marl_for_im_b200 import _lib, presets
from marl_for_im_b200.envs import ENV_CLASSES

pytestmark = pytest.mark.gpu

NETS = [("MAIM", "serial4"), ("IM", "serial8"), ("MAIM", "serial2"), ("IM_div", "div1"), ("MAIM_div", "div2")]
STATE = ("inv", "backlog", "order_u")
PERIOD = ("demand", "ship", "acquisition", "order_r", "profit")
FIXTURE_KEY = {"inv": "inv", "backlog": "backlog", "order_u": "order_u", "demand": "demand", "ship": "ship", "acquisition": "acq",
               "order_r": "order", "profit": "profit"}
FUSED_N = 4096
SIZES = [FUSED_N, FUSED_N + 36, FUSED_N + 2, 100]     # whole tiles; a tail tile; N % 4 != 0; below the specialisation


def _fused(preset, n, want_obs, records=True):
    """The dispatch rule: whole tiles of the specialised build.  Without records the divergent networks take the episode kernel
    only where it measured ahead of the composition — div2 (env-per-thread body) with observations, div1 without; with records
    it is ahead on every network (the composition is then T ahead-of-time step launches and 3 T copies)."""
    if n != FUSED_N:
        return False
    return records or {"div2": want_obs, "div1": not want_obs}.get(preset, True)


def _inputs(kind, cfg, n, seed, dtype=torch.float64):
    env = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=4))
    m, T, R = env.num_nodes, env.num_periods, len(env._retailers)
    g = torch.Generator(device="cuda:0")
    g.manual_seed(seed)
    demand = torch.poisson(torch.full((n, R, T), 5.0, device="cuda:0"), generator=g).to(torch.int32)
    if kind.endswith("div"):
        actions = (torch.randn((T, n, m), dtype=torch.float64, device="cuda:0", generator=g) * 0.5 - 0.6).clamp(-1, 1)
    else:
        actions = torch.rand((T, n, m), dtype=torch.float64, device="cuda:0", generator=g) * 2.3 - 1.15
    return demand, actions.to(dtype)


def _stepwise(env, actions, demand=None, delay_mask=None):
    """The records the slow way: reset, then T one-period steps with the diagnostics, the state copied after each."""
    env.reset(customer_demand=demand, delay_mask=delay_mask)
    st = env.state_dict()
    rec = {k: [st[k].clone()] for k in STATE}
    per = {k: [] for k in PERIOD}
    obs, rew = [], []
    for t in range(env.num_periods):
        o, r, _, info = env.step_many(actions[t:t + 1], return_info=True)
        obs.append(o[0].clone())
        rew.append(r[0].clone())
        for k in STATE:
            rec[k].append(env.state_dict()[k].clone())
        for k, src in (("demand", "demand"), ("ship", "ship"), ("acquisition", "acquisition"), ("order_r", "actual order"),
                       ("profit", "profit")):
            per[k].append(info[src][0].clone())
    out = {k: torch.stack(v) for k, v in rec.items()}
    out.update({k: torch.stack(v) for k, v in per.items()})
    return out, torch.stack(obs), torch.stack(rew)


def _snapshot(env):
    return {k: v.clone() for k, v in env.state_dict().items()}, env.error_flags.clone(), env.period


def _assert_same_env(a, b, what):
    sa, ea, pa = _snapshot(a)
    sb, eb, pb = _snapshot(b)
    assert sa.keys() == sb.keys() and pa == pb, what
    for k in sa:
        assert torch.equal(sa[k], sb[k]), (what, k)
    assert torch.equal(ea, eb), what


def _assert_records(got, want, fields, what):
    for k in STATE + PERIOD:
        if k in fields:
            assert got[k] is not None and torch.equal(got[k], want[k]), (what, k)
        else:
            assert got[k] is None, (what, k)


@pytest.mark.parametrize("name", golden_names())
def test_records_equal_the_reference_fixture(name):
    """Every reference episode replicated over 4 096 envs: every env's records are the fixture's history arrays, bit for bit.
    Run with and without observations; the T = 30 episodes are served by the episode kernel."""
    g = load_golden(name)
    kind, ref = g["kind"], g["ref"]
    n = FUSED_N
    d = np.asarray(g["demand_trace"])
    demand = np.ascontiguousarray(np.broadcast_to(d[None], (n,) + d.shape)).astype(np.int32)
    actions = torch.as_tensor(np.ascontiguousarray(np.broadcast_to(g["actions"][:, None, :], (g["actions"].shape[0], n, g["actions"].shape[1]))),
                              device="cuda:0")
    mask = None
    if g["delay_mask"] is not None:
        mask = np.ascontiguousarray(np.broadcast_to(np.asarray(g["delay_mask"])[None], (n,) + g["delay_mask"].shape))
    variants = []
    for want_obs in (True, False):
        cfg = dict(copy_config(g["config"]), num_envs=n)
        env = ENV_CLASSES[kind](cfg)
        got = env.replay_episode(actions, customer_demand=demand, delay_mask=mask, want_obs=want_obs, records=True)["records"]
        variants.append(env._lib.imx_kernel_variant(env._handle))
        for k, fk in FIXTURE_KEY.items():
            want = torch.as_tensor(np.asarray(ref[fk]), device="cuda:0")
            want = want.to(torch.float64 if k == "profit" else torch.int32)[:, None, :].expand_as(got[k])
            assert torch.equal(got[k], want), (name, want_obs, k)
        assert int(env.error_flags.abs().sum()) == 0, name
    if g["actions"].shape[0] == 30:
        assert variants == [4, 4], (name, variants)


@pytest.mark.parametrize("want_obs", [True, False])
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("kind,preset", NETS)
def test_records_equal_stepwise_and_change_nothing_else(kind, preset, n, want_obs):
    cfg = presets.PRESETS[preset]()
    demand, actions = _inputs(kind, cfg, n, seed=n + 3 * want_obs)
    ref = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    want, want_obs_t, want_rew = _stepwise(ref, actions, demand)
    plain = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    env = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    kw = dict(customer_demand=demand, want_obs=want_obs, want_rewards=True, stats=True, eval_acc=True)
    base = plain.replay_episode(actions, **kw)
    got = env.replay_episode(actions, records=True, **kw)
    _assert_records(got["records"], want, STATE + PERIOD, (kind, n, want_obs))
    assert base["records"] is None
    for k in ("returns", "stats", "obs", "rewards", "eval"):
        assert (got[k] is None) == (base[k] is None) and (got[k] is None or torch.equal(got[k], base[k])), (kind, n, k)
    assert torch.equal(got["rewards"], want_rew)
    if want_obs:
        assert torch.equal(got["obs"], want_obs_t)
    _assert_same_env(env, plain, (kind, n, want_obs))
    _assert_same_env(env, ref, (kind, n, want_obs))
    v = env._lib.imx_kernel_variant(env._handle)
    assert (v == 4) == _fused(preset, n, want_obs), (kind, n, want_obs, v)
    assert (plain._lib.imx_kernel_variant(plain._handle) == 4) == _fused(preset, n, want_obs, records=False)


# (kind, preset, handle options, call options) — the inputs and types the fused and the composed path must agree on
MODES = {
    "philox": ("MAIM", "serial4", {}, {"demand": False}),
    "philox_div2_noisy_demand": ("MAIM_div", "div2", {"noisy_demand": True, "noisy_demand_threshold": 0.2}, {"demand": False}),
    "noisy_replayed": ("MAIM", "serial8", {"noisy_delay": True, "noisy_delay_threshold": 0.3}, {"mask": True}),
    "noisy_generated": ("MAIM_div", "div2", {"noisy_delay": True, "noisy_delay_threshold": 0.3}, {"noisy": True}),
    "obs_f32": ("MAIM", "serial4", {"obs_dtype": "float32"}, {}),
    "obs_bf16_actions_f32": ("MAIM_div", "div2", {"obs_dtype": "bfloat16", "action_dtype": "float32"}, {}),
    "actions_f32_div1": ("IM_div", "div1", {"action_dtype": "float32"}, {}),
    "subset_state": ("MAIM", "serial4", {}, {"fields": ("inv", "order_u")}),
    "subset_period": ("MAIM_div", "div2", {}, {"fields": ("ship", "profit")}),
    "subset_mixed": ("IM", "serial8", {}, {"fields": ("backlog", "demand", "order_r")}),
}


@pytest.mark.parametrize("n", [FUSED_N, FUSED_N + 36])
@pytest.mark.parametrize("mode", sorted(MODES))
def test_records_modes(mode, n):
    kind, preset, opts, call = MODES[mode]
    cfg = dict(presets.PRESETS[preset](), **opts)
    adt = torch.float32 if opts.get("action_dtype") == "float32" else torch.float64
    demand, actions = _inputs(kind, cfg, n, seed=17, dtype=adt)
    demand = demand if call.get("demand", True) else None
    ref = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    env = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    plain = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    mask = None
    if call.get("mask"):
        mask = torch.rand((n, ref.num_periods, ref.num_nodes), device="cuda:0") < 0.3
    if call.get("noisy"):                                      # the sticky flag: Philox outcomes from here on
        for e in (ref, env, plain):
            e.reset(noisy_delay=True, noisy_delay_threshold=0.3)
    # (the three handles count their episodes alike: Philox demand and delays are drawn for the same episode id)
    want, _, _ = _stepwise(ref, actions, demand, mask)
    fields = call.get("fields", STATE + PERIOD)
    kw = dict(customer_demand=demand, delay_mask=mask, want_obs=True, want_rewards=True, stats=True)
    got = env.replay_episode(actions, records=list(fields) if "fields" in call else True, **kw)
    base = plain.replay_episode(actions, **kw)
    _assert_records(got["records"], want, fields, (mode, n))
    for k in ("returns", "stats", "obs", "rewards"):
        assert torch.equal(got[k], base[k]), (mode, n, k)
    _assert_same_env(env, plain, (mode, n))
    _assert_same_env(env, ref, (mode, n))
    assert (env._lib.imx_kernel_variant(env._handle) == 4) == _fused(preset, n, True), (mode, n)


@pytest.mark.parametrize("kind,preset", [("MAIM", "serial4"), ("MAIM_div", "div2")])
def test_records_are_independent_of_sharding(kind, preset):
    """Philox demand: two half handles with env_offset 0 and N/2 record the full handle's rows."""
    cfg = presets.PRESETS[preset]()
    n = 8192
    _, actions = _inputs(kind, cfg, n, seed=23)
    full = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    got = full.replay_episode(actions, want_obs=True, records=True)["records"]
    assert full._lib.imx_kernel_variant(full._handle) == 4
    half = n // 2
    for off in (0, half):
        part = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=half, env_offset=off))
        r = part.replay_episode(actions[:, off:off + half].contiguous(), want_obs=True, records=True)["records"]
        assert part._lib.imx_kernel_variant(part._handle) == 4
        for k in STATE + PERIOD:
            assert torch.equal(r[k], got[k][:, off:off + half]), (kind, off, k)


def _record_bytes(T, n, m):
    return {k: (T + 1) * n * m * 4 for k in STATE} | {k: T * n * m * 4 for k in PERIOD[:4]} | {"profit": T * n * m * 8}


def _call(env, demand, actions, ptrs, s, obs=None, ret=None, stats=None):
    st = _lib.ImxRecordsOut(*[ptrs.get(k) for k in STATE + PERIOD])
    return env._lib.imx_replay_episode_records(env._handle, C.c_void_p(demand.data_ptr()), None, 0, 2, C.c_void_p(actions.data_ptr()),
                                               obs, None, ret, stats, 0, None, C.byref(st), s)


@pytest.mark.parametrize("offset", [0, 8])
def test_record_buffers_are_written_only_inside_their_rows(offset):
    """Sentinel bytes around every record buffer; offset 8 breaks the 16-byte alignment of every record pointer (the call
    falls back to the composition) and still gives the same bytes."""
    kind, cfg, n = "MAIM", presets.serial4(), FUSED_N
    demand, actions = _inputs(kind, cfg, n, seed=31)
    ref = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    want, _, _ = _stepwise(ref, actions, demand)
    env = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    T, m = env.num_periods, env.num_nodes
    pad = 512
    nbytes = _record_bytes(T, n, m)
    raw = {k: torch.full((b + 2 * pad + offset,), 0x5A, dtype=torch.uint8, device="cuda:0") for k, b in nbytes.items()}
    ptrs = {k: raw[k].data_ptr() + pad + offset for k in nbytes}
    ret = torch.empty((n, m), dtype=torch.float64, device="cuda:0")
    _lib.check(_call(env, demand, actions, ptrs, C.c_void_p(torch.cuda.current_stream().cuda_stream), ret=C.c_void_p(ret.data_ptr())))
    torch.cuda.synchronize()
    for k, b in nbytes.items():
        r = raw[k]
        assert bool((r[:pad + offset] == 0x5A).all()) and bool((r[pad + offset + b:] == 0x5A).all()), (offset, k)
        assert torch.equal(r[pad + offset:pad + offset + b], want[k].reshape(-1).view(torch.uint8)), (offset, k)
    _assert_same_env(env, ref, offset)
    assert (env._lib.imx_kernel_variant(env._handle) == 4) == (offset == 0)


def test_cuda_graph_replay_and_launch_count():
    kind, cfg, n = "MAIM", presets.serial4(), 65536
    demand, actions = _inputs(kind, cfg, n, seed=41)
    ref = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    want, want_obs, _ = _stepwise(ref, actions, demand)
    env = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    lib, h = env._lib, env._handle
    _lib.check(lib.imx_prepare(h, _lib.PREPARE_EPISODE | _lib.PREPARE_RECORDS))
    T, m, O = env.num_periods, env.num_nodes, env.obs_len
    bufs = {k: torch.empty(b // (8 if k == "profit" else 4), dtype=torch.float64 if k == "profit" else torch.int32, device="cuda:0")
            for k, b in _record_bytes(T, n, m).items()}
    ptrs = {k: v.data_ptr() for k, v in bufs.items()}
    obs = torch.empty((T, n, m, O), dtype=torch.float64, device="cuda:0")
    ret = torch.empty((n, m), dtype=torch.float64, device="cuda:0")
    stats = torch.empty(3 + 2 * m, dtype=torch.float64, device="cuda:0")
    p = lambda x: C.c_void_p(x.data_ptr())                    # noqa: E731
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    c0 = env.launch_count()
    _lib.check(_call(env, demand, actions, ptrs, s, obs=p(obs), ret=p(ret)))
    c1 = env.launch_count()
    _lib.check(_call(env, demand, actions, ptrs, s, obs=p(obs), ret=p(ret), stats=p(stats)))
    c2 = env.launch_count()
    assert (c1 - c0, c2 - c1) == (1, 3) and lib.imx_kernel_variant(h) == 4
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            _lib.check(_call(env, demand, actions, ptrs, C.c_void_p(torch.cuda.current_stream().cuda_stream), obs=p(obs), ret=p(ret)))
    torch.cuda.current_stream().wait_stream(side)
    for rep in range(5):
        for v in list(bufs.values()) + [obs]:
            v.zero_()
        g.replay()
        torch.cuda.synchronize()
        for k in STATE + PERIOD:
            assert torch.equal(bufs[k].view(want[k].shape), want[k]), (rep, k)
        assert torch.equal(obs, want_obs), rep
    _assert_same_env(env, ref, "graph")


def test_composition_under_capture_after_prepare():
    """A batch the episode kernel cannot serve (a tail tile): the composition's T steps and state copies, captured and replayed."""
    kind, cfg, n = "MAIM_div", presets.div2(), FUSED_N + 36
    demand, actions = _inputs(kind, cfg, n, seed=43)
    ref = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    want, _, _ = _stepwise(ref, actions, demand)
    env = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    _lib.check(env._lib.imx_prepare(env._handle, _lib.PREPARE_RECORDS))
    T, m = env.num_periods, env.num_nodes
    bufs = {k: torch.zeros(b // (8 if k == "profit" else 4), dtype=torch.float64 if k == "profit" else torch.int32, device="cuda:0")
            for k, b in _record_bytes(T, n, m).items()}
    ptrs = {k: v.data_ptr() for k, v in bufs.items()}
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            _lib.check(_call(env, demand, actions, ptrs, C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.current_stream().wait_stream(side)
    g.replay()
    torch.cuda.synchronize()
    for k in STATE + PERIOD:
        assert torch.equal(bufs[k].view(want[k].shape), want[k]), k
    assert env._lib.imx_kernel_variant(env._handle) != 4


def test_records_call_under_capture_without_prepare_is_refused():
    kind, cfg, n = "MAIM", presets.serial4(), FUSED_N
    demand, actions = _inputs(kind, cfg, n, seed=47)
    env = ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n))
    env.replay_episode(actions, customer_demand=demand)        # the episode module without records is loaded; not the records one
    T, m = env.num_periods, env.num_nodes
    bufs = {k: torch.empty(b // 4, dtype=torch.int32, device="cuda:0") for k, b in _record_bytes(T, n, m).items() if k != "profit"}
    ptrs = {k: v.data_ptr() for k, v in bufs.items()}
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    rc = []
    with torch.cuda.stream(side):
        g = torch.cuda.CUDAGraph()
        try:
            with torch.cuda.graph(g, stream=side):
                rc.append(_call(env, demand, actions, ptrs, C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        except RuntimeError:
            pass                                                  # an empty capture may be rejected by torch: the code is what counts
    torch.cuda.current_stream().wait_stream(side)
    assert rc == [-1] and b"IMX_PREPARE_RECORDS" in env._lib.imx_last_error()
    # outside capture the call builds its module and records
    got = env.replay_episode(actions, customer_demand=demand, records=("inv",))["records"]
    assert got["inv"].shape == (T + 1, n, m) and got["profit"] is None


def test_unknown_record_field_is_refused():
    env = ENV_CLASSES["MAIM"](dict(presets.serial4(), num_envs=8))
    with pytest.raises(ValueError):
        env.replay_episode(torch.zeros((env.num_periods, 8, env.num_nodes), dtype=torch.float64), records=("inventory",))
