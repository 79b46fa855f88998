"""Every kernel family at the limits imx_create accepts, against the oracles on distinct per-env traces: the 32-lane divergent
kernels (32 nodes, 8 children), the top of the 16-lane tile, 6-8 active children in the split, the env-per-thread boundary, a
32-stage chain at lead time and history 8, capacities without a rescale table (float64 and float32 observations), T = 1 and 2,
noisy delays at thresholds 0 and 1, and the split watchdog at demand_max near INT32_MAX.  Each test pins the kernel variant it
means to exercise (imx_kernel_variant: 0 direct, 1 ahead-of-time TMA, 2 specialised, 3 pipelined, 4 episode kernel)."""
import numpy as np
import pytest
import torch

from harness import copy_config
from marl_for_im_b200.envs import ENV_CLASSES
from oracle import c_oracle, im_oracle
from test_config_limits_cpu import CASES, WATCHDOG_CASES, carry_cfg, draw, python_run, watchdog_case, watchdog_inputs, watchdog_loop_ran

pytestmark = pytest.mark.gpu

# step paths: environment switches read by imx_create -> the variant that serves step() (return_info forces the direct kernel)
PATHS = {"specialised": ({"IMX_PIPE": "0"}, 2), "pipelined": ({"IMX_PIPE": "1", "IMX_PIPE_CTAS": "1"}, 3),
         "aot_tma": ({"IMX_JIT": "0", "IMX_STEP_PATH": "tma"}, 1), "direct": ({"IMX_STEP_PATH": "direct"}, 0)}
SIZES = (4096, 4096 + 36)                      # whole tiles of every tile width, and a tail for the direct kernel


def _env(kind, cfg, n, monkeypatch, switches=(), **extra):
    for k, v in dict(switches).items():
        monkeypatch.setenv(k, v)
    return ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n, **extra))


def _variant(env):
    return env._lib.imx_kernel_variant(env._handle)


def _packed_reward(env, r):
    return (torch.stack([r[a] for a in env.agent_names], dim=1) if env.MULTI else r[:, None]).cpu().numpy()


def _assert_state(env, want, what):
    """Every state field the handle keeps, the watchdog flags and the period, against the C oracle."""
    N, m = env.num_envs, env.num_nodes
    st = {k: v.cpu().numpy() for k, v in env.state_dict().items()}
    for k in ("inv", "backlog", "order_u", "pipe"):
        np.testing.assert_array_equal(st[k], want[k], err_msg=f"{what}: {k}")
    if "backlog_to" in st:
        np.testing.assert_array_equal(st["backlog_to"], want["backlog_to"], err_msg=f"{what}: backlog_to")
    for k in ("hist_d", "hist_o"):
        if k in st:
            np.testing.assert_array_equal(st[k].reshape(N, m, -1), want[k], err_msg=f"{what}: {k}")
    assert not want["err"].any() and not env.error_flags.cpu().numpy().any(), what
    assert env.period == env.num_periods, what


def _obs_want(env, obs):
    return obs.astype(np.float32) if env.obs_dtype == torch.float32 else obs


def _inputs(name, n, seed=0):
    kind, cfg, mu, mode = CASES[name]
    demand, actions = draw(kind, cfg, n, np.random.default_rng(seed + sorted(CASES).index(name)), mu, mode)
    return kind, cfg, demand, actions


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("path", sorted(PATHS))
@pytest.mark.parametrize("name", sorted(CASES))
def test_step_matches_c_oracle(name, path, n, monkeypatch):
    kind, cfg, demand, actions = _inputs(name, n)
    switches, variant = PATHS[path]
    env = _env(kind, cfg, n, monkeypatch, switches)
    env.reset(customer_demand=demand)
    a = torch.as_tensor(actions, device="cuda:0")
    rews, variants = [], set()
    for t in range(env.num_periods):
        _, r, _, _ = env.step(a[t])
        variants.add(_variant(env))
        rews.append(_packed_reward(env, r))
    assert variants == {variant}, (name, path, variants)
    want = c_oracle.COracle(kind, cfg).run(demand, actions)
    np.testing.assert_array_equal(np.stack(rews), want["reward"])
    np.testing.assert_array_equal(env.last_obs.cpu().numpy(), _obs_want(env, want["obs_last"]))
    _assert_state(env, want, (name, path, n))


@pytest.mark.parametrize("name", sorted(CASES))
def test_step_with_info_matches_python_oracle(name, monkeypatch):
    """return_info: the diagnostics of every period, against the Python oracle on a sample of envs."""
    n = 4096 + 36
    kind, cfg, demand, actions = _inputs(name, n, seed=50)
    env = _env(kind, cfg, n, monkeypatch, return_info=True)
    env.reset(customer_demand=demand)
    a = torch.as_tensor(actions, device="cuda:0")
    infos, rews = [], []
    for t in range(env.num_periods):
        _, r, _, info = env.step(a[t])
        assert _variant(env) == 1                   # the diagnostics keep the specialised kernels out: ahead-of-time TMA
        rews.append(_packed_reward(env, r))
        if env.MULTI:
            info = {k: torch.stack([info[ag][k] for ag in env.agent_names], dim=1) for k in ("demand", "ship", "acquisition", "actual order", "profit")}
        infos.append({k: v.cpu().numpy() for k, v in info.items() if k != "period"})
    want = c_oracle.COracle(kind, cfg).run(demand, actions)
    np.testing.assert_array_equal(np.stack(rews), want["reward"])
    _assert_state(env, want, name)
    for k in range(0, n, 517):
        o = im_oracle.OracleEnv(kind, copy_config(cfg))
        o.reset(demand[k] if o.div else demand[k].reshape(-1))
        for t in range(o.T):
            _, _, _, wi = o.step(actions[t, k])
            for f in ("demand", "ship", "acquisition", "actual order", "profit"):
                np.testing.assert_array_equal(infos[t][f][k], wi[f], err_msg=f"{name} env {k} t {t} {f}")


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("fuse", ["1", "0"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_step_many_matches_c_oracle(name, fuse, n, monkeypatch):
    """step_many over the whole episode: one multi-period launch, or (IMX_FUSE_PERIODS=0, and with a tail) T plain launches."""
    kind, cfg, demand, actions = _inputs(name, n, seed=100)
    env = _env(kind, cfg, n, monkeypatch, {"IMX_FUSE_PERIODS": fuse, "IMX_PIPE": "0"})
    env.reset(customer_demand=demand)
    obs, rew, _ = env.step_many(torch.as_tensor(actions, device="cuda:0"))
    assert _variant(env) == 2
    want = c_oracle.COracle(kind, cfg).run(demand, actions, all_obs=True)
    np.testing.assert_array_equal(rew.cpu().numpy().reshape(want["reward"].shape), want["reward"])
    np.testing.assert_array_equal(obs.cpu().numpy(), _obs_want(env, want["obs_all"][1:]))
    _assert_state(env, want, (name, fuse))


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("name", sorted(CASES))
def test_replay_episode_matches_oracles(name, n, monkeypatch):
    """replay_episode against the oracles directly: rewards, returns (the oracle's rewards summed in period order), the
    evaluation accumulators (im_oracle.eval_loop_accumulators on a sample of envs) and the final state."""
    kind, cfg, demand, actions = _inputs(name, n, seed=200)
    env = _env(kind, cfg, n, monkeypatch)
    got = env.replay_episode(torch.as_tensor(actions, device="cuda:0"), customer_demand=demand, want_obs=True, want_rewards=True,
                             eval_acc=True)
    assert _variant(env) == (4 if (name, n) in EPISODE_KERNEL else 1), _variant(env)
    want = c_oracle.COracle(kind, cfg).run(demand, actions, all_obs=True)
    cols = want["reward"].shape[2]
    np.testing.assert_array_equal(got["rewards"].cpu().numpy().reshape(want["reward"].shape), want["reward"])
    np.testing.assert_array_equal(got["obs"].cpu().numpy(), _obs_want(env, want["obs_all"][1:]))
    ret = np.zeros((n, cols))
    for t in range(env.num_periods):
        ret = ret + want["reward"][t]
    np.testing.assert_array_equal(got["returns"].cpu().numpy().reshape(n, cols), ret)
    _assert_state(env, want, (name, n))
    if env.obs_dtype == torch.float32:
        return                      # the accumulators read float32 observations back: their float64 twins check the sums
    ev = got["eval"].cpu().numpy()
    for k in range(0, n, 1031):
        o = im_oracle.OracleEnv(kind, copy_config(cfg))
        w = im_oracle.eval_loop_accumulators(o, demand[k] if o.div else demand[k].reshape(-1), actions[:, k], rescaled=bool(o.std_state))
        if o.multi:
            np.testing.assert_array_equal(ev[k], w, err_msg=f"{name} env {k}")
        else:
            # the single-agent loop totals a period's stages with the builtin sum(), which CPython 3.12 made compensated; the
            # kernels (and earlier CPythons) add them in stage order, so those two columns may differ in the last bits
            np.testing.assert_array_equal(ev[k, [0, 3]], w[[0, 3]], err_msg=f"{name} env {k}")
            np.testing.assert_array_equal(ev[k, 4:], w[4:], err_msg=f"{name} env {k}")
            np.testing.assert_allclose(ev[k, 1:3], w[1:3], rtol=1e-14, atol=0, err_msg=f"{name} env {k}")


# where imx_replay_episode's one-launch episode kernel serves (whole tiles that fit its layout; divergent networks only under
# the measured rule of its dispatch); elsewhere the library runs the composition, whose step_many keeps the profit diagnostics
# for the evaluation accumulators and so takes the ahead-of-time TMA kernel.  A retune of that dispatch moves entries here.
EPISODE_KERNEL = {(name, 4096) for name in CASES if name[0] in "efg" and "div" not in name} | \
    {("g_imdiv_t2", 4096), ("f_maimdiv_div_big", 4096), ("f_maimdiv_div_big_f32", 4096), ("e_im_chain32", 4132), ("e_maim_chain32", 4132)}


@pytest.mark.parametrize("et", ["1", "0"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_rollout_matches_c_oracle(name, et, monkeypatch):
    """rollout_basestock (returns and step rewards), env-per-thread (IMX_ROLLOUT_ET=1, where the network allows it) and
    lane-mapped rollouts, on distinct per-env traces and base-stock levels, with a tail."""
    kind, cfg, _, _ = CASES[name]
    cfg = dict(copy_config(cfg), time_dependency=False, prev_demand=False, prev_actions=False)
    if kind in ("IM", "IM_div"):
        cfg.update(standardise_state=False, standardise_actions=False)
    n = 4096 + 36
    demand = _inputs(name, n, seed=300)[2]
    env = _env(kind, cfg, n, monkeypatch, {"IMX_ROLLOUT_ET": et})
    m = env.num_nodes
    rng = np.random.default_rng(7)
    om = np.asarray(env.order_max, dtype=np.float64)
    z = rng.uniform(0, 3, size=(n, m)) * np.minimum(om, 40)
    z = np.floor(z) + rng.choice([0.0, 0.37], size=(n, m))
    out = env.rollout_basestock(z, customer_demand=demand, step_rewards=True, write_state=True)
    assert _variant(env) == 2
    want = c_oracle.COracle(kind, cfg).rollout(z, demand, step_rewards=True)
    assert want["bad"] == 0 and not env.error_flags.cpu().numpy().any()
    np.testing.assert_array_equal(out["step_rewards"].cpu().numpy().reshape(want["step_rewards"].shape), want["step_rewards"])
    np.testing.assert_array_equal(out["returns"].cpu().numpy().reshape(want["returns"].shape), want["returns"])
    st = {k: v.cpu().numpy() for k, v in env.state_dict().items()}
    for k in ("inv", "backlog", "order_u", "pipe"):
        np.testing.assert_array_equal(st[k], want[k], err_msg=k)
    if "backlog_to" in st:
        np.testing.assert_array_equal(st["backlog_to"], want["backlog_to"])


@pytest.mark.parametrize("source", ["replayed", "philox"])
@pytest.mark.parametrize("thr", [0.0, 1.0])
@pytest.mark.parametrize("name", ["a_maimdiv_tree32", "a_imdiv_tree32", "e_maim_chain32", "e_im_chain32"])
def test_noisy_delay_extremes(name, thr, source, monkeypatch):
    """Threshold 1 holds every arrival back until the last period (goods carry over many periods), threshold 0 none; the
    outcomes replayed from a mask or drawn from Philox (then read back and given to the oracle)."""
    n = 4096 + 36
    kind, cfg, demand, actions = _inputs(name, n, seed=400)
    env = _env(kind, cfg, n, monkeypatch, {"IMX_PIPE": "0"})
    T, m = env.num_periods, env.num_nodes
    if source == "replayed":
        mask = np.random.default_rng(5).uniform(size=(n, T, m)) <= thr
        env.reset(customer_demand=demand, delay_mask=mask)
    else:
        env.reset(customer_demand=demand, noisy_delay=True, noisy_delay_threshold=thr)
        mask = env.delay_mask_device().cpu().numpy().transpose(1, 0, 2).astype(bool)
        assert mask[:, T - 1].all() if thr == 1.0 else not mask.any()
    a = torch.as_tensor(actions, device="cuda:0")
    rews = []
    for t in range(T):
        _, r, _, _ = env.step(a[t])
        assert _variant(env) == 2
        rews.append(_packed_reward(env, r))
    want = c_oracle.COracle(kind, cfg).run(demand, actions, mask)
    np.testing.assert_array_equal(np.stack(rews), want["reward"])
    np.testing.assert_array_equal(env.last_obs.cpu().numpy(), want["obs_last"])
    _assert_state(env, want, (name, thr, source))
    carry = env.state_dict()["carry"].cpu().numpy()
    for k in range(0, n, 1031):
        np.testing.assert_array_equal(carry[k], python_run(kind, cfg, demand[k], actions[:, k], mask[k])[2]["carry"])


@pytest.mark.parametrize("path", ["specialised", "direct"])
@pytest.mark.parametrize("case", sorted(WATCHDOG_CASES))
def test_split_watchdog_near_int32_max(case, path, monkeypatch):
    """demand_max[0] * 4 (or * 2) above INT32_MAX: the split drains without a spurious 'Infinite Loop', like the Python
    oracle, through step() on the specialised and the direct kernel."""
    kind, cfg = watchdog_case(case)
    n = 4096
    demand, actions = watchdog_inputs(kind, cfg, n, np.random.default_rng(2))
    env = _env(kind, cfg, n, monkeypatch, PATHS[path][0])
    env.reset(customer_demand=demand)
    a = torch.as_tensor(actions, device="cuda:0")
    rews = []
    for t in range(env.num_periods):
        _, r, _, _ = env.step(a[t])
        assert _variant(env) == PATHS[path][1]
        rews.append(_packed_reward(env, r))
    want = c_oracle.COracle(kind, cfg).run(demand, actions)
    np.testing.assert_array_equal(np.stack(rews), want["reward"])
    _assert_state(env, want, case)
    for k in range(0, n, 811):
        assert watchdog_loop_ran(kind, cfg, demand[k], actions[:, k])
        rew, _, st = python_run(kind, cfg, demand[k], actions[:, k])
        np.testing.assert_array_equal(np.stack(rews)[:, k], rew)
        for f in ("inv", "backlog", "order_u", "backlog_to"):
            np.testing.assert_array_equal(env.state_dict()[f][k].cpu().numpy(), st[f])


ET_CASES = ["d_maimdiv_tree8_d4p2", "d_maimdiv_tree8_d5p2", "d_imdiv_tree8_d4p3", "g_imdiv_t2"]


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("pipe", ["0", "1"])
@pytest.mark.parametrize("et", ["0", "1"])
@pytest.mark.parametrize("name", ET_CASES)
def test_step_env_per_thread_boundary(name, et, pipe, n, monkeypatch):
    """IMX_STEP_ET=1 / 0 on the specialised and the pipelined step.  The env-per-thread body is built for networks up to 8
    nodes, lead time 4 and history 2 (imx_api.cu, et_ok): d_maimdiv_tree8_d4p2 is the largest such config and takes it; the
    d5 / p3 configs sit just outside and take the lane kernels whatever the switch says; g_imdiv_t2 (div2, 6 nodes) takes it by
    default and the lanes with IMX_STEP_ET=0.  imx_kernel_variant reports 2 / 3 for either body, so the variant pins the
    specialised / pipelined kernel and the body follows from the config."""
    kind, cfg, demand, actions = _inputs(name, n, seed=500)
    switches = {"IMX_STEP_ET": et, "IMX_PIPE": pipe, "IMX_PIPE_CTAS": "1"}
    env = _env(kind, cfg, n, monkeypatch, switches)
    env.reset(customer_demand=demand)
    a = torch.as_tensor(actions, device="cuda:0")
    rews = []
    for t in range(env.num_periods):
        _, r, _, _ = env.step(a[t])
        assert _variant(env) == (3 if pipe == "1" else 2)
        rews.append(_packed_reward(env, r))
    want = c_oracle.COracle(kind, cfg).run(demand, actions)
    np.testing.assert_array_equal(np.stack(rews), want["reward"])
    np.testing.assert_array_equal(env.last_obs.cpu().numpy(), want["obs_last"])
    _assert_state(env, want, (name, et, pipe, n))


@pytest.mark.parametrize("path", ["specialised", "direct"])
def test_noisy_carry_at_the_edge_of_the_domain(path, monkeypatch):
    """Every arrival held back until the last period at 2^28 capacity, on the largest T imx_create accepts for it: the carry
    reaches 5 x 2^28 without wrapping."""
    kind, cfg = "MAIM", carry_cfg(6)
    n = 4096
    rng = np.random.default_rng(9)
    demand = rng.integers(0, 10, size=(n, 1, 6)).astype(np.int32)
    actions = np.where(rng.uniform(size=(6, n, 4)) < 0.9, 1.0, rng.uniform(-1, 1, size=(6, n, 4)))
    mask = rng.uniform(size=(n, 6, 4)) < 0.95
    env = _env(kind, cfg, n, monkeypatch, PATHS[path][0])
    env.reset(customer_demand=demand, delay_mask=mask)
    a = torch.as_tensor(actions, device="cuda:0")
    rews = []
    for t in range(6):
        _, r, _, _ = env.step(a[t])
        assert _variant(env) == PATHS[path][1]
        rews.append(_packed_reward(env, r))
    want = c_oracle.COracle(kind, cfg).run(demand, actions, mask)
    np.testing.assert_array_equal(np.stack(rews), want["reward"])
    np.testing.assert_array_equal(env.last_obs.cpu().numpy(), want["obs_last"])
    _assert_state(env, want, path)
    for k in range(0, n, 1031):
        rew, _, st = python_run(kind, cfg, demand[k], actions[:, k], mask[k])
        np.testing.assert_array_equal(np.stack(rews)[:, k], rew)
        np.testing.assert_array_equal(env.state_dict()["inv"][k].cpu().numpy(), st["inv"])
