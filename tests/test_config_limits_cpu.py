"""The edges of what imx_create accepts, without a GPU: the Python and C oracles agree on configs at the limits (32 nodes, 8
children, lead time and history 8, capacities without a rescale table, T = 1 and 2, noisy delays at thresholds 0 and 1, the
split watchdog at demand_max near INT32_MAX), the runtime-specialised kernels build for sm_100a at those limits, and
imx_create refuses every config whose int32 state could wrap.  The configs here are shared with test_gpu_config_limits.py."""
import ctypes

import numpy as np
import pytest

from harness import copy_config
from marl_for_im_b200 import _lib, presets
from marl_for_im_b200.envs import ENV_CLASSES
from oracle import c_oracle, im_oracle

INT32_MAX = 2 ** 31 - 1


def _tree(conn, m, periods, delay, P, inv_max=40, **flags):
    cfg = {"num_nodes": m, "num_periods": periods, "connections": {i: list(conn.get(i, [])) for i in range(m)},
           "init_inv": np.full(m, 12.0), "inv_target": np.arange(m) % 4 * 1.0, "inv_max": np.full(m, float(inv_max)),
           "stock_cost": 0.1 + 0.4 * (np.arange(m) % 5) / 5, "backlog_cost": 0.3 + 0.6 * (np.arange(m) % 7) / 7,
           "delay": np.asarray(delay if np.ndim(delay) else np.full(m, delay), dtype=np.int64),
           "time_dependency": True, "prev_demand": True, "prev_actions": True, "prev_length": P,
           "independent": False, "share_network": False}
    cfg.update(flags)
    return cfg


def tree32(periods=12, **flags):
    """Config a: 32 nodes, nodes 0-3 carry 8, 8, 8 and 7 children (28 retailers), lead time 8 and history 8 everywhere."""
    conn = {0: list(range(1, 9)), 1: list(range(9, 17)), 2: list(range(17, 25)), 3: list(range(25, 32))}
    return _tree(conn, 32, periods, 8, 8, **flags)


def tree_n(m, periods=12, **flags):
    """Config b: breadth-first trees of 13 and 16 nodes (the top of the 16-lane tile)."""
    conn, nxt, parent = {}, 1, 0
    while nxt < m:
        k = min(3 + parent % 3, m - nxt)
        conn[parent] = list(range(nxt, nxt + k))
        nxt += k
        parent += 1
    return _tree(conn, m, periods, 1 + np.arange(m) % 5, 3, **flags)


def star8(periods=40, **flags):
    """Config c: node 0 with 8 retailer children; node 0 short of goods so that every split loop runs with 6-8 children."""
    cfg = _tree({0: list(range(1, 9))}, 9, periods, np.array([1, 2, 1, 3, 1, 2, 1, 1, 2]), 2, prev_actions=False, **flags)
    cfg["inv_max"] = np.array([60.0] + [25.0] * 8)
    cfg["init_inv"] = np.array([30.0] + [5.0] * 8)
    return cfg


def tree8(delay, P, **flags):
    """Config d: an 8-node tree; delay 4 / P 2 is the largest env-per-thread config, delay 5 or P 3 takes the lane kernels."""
    return _tree({0: [1, 2, 3], 1: [4, 5], 2: [6], 3: [7]}, 8, 14, delay, P, **flags)


def chain32(kind, periods=12, **flags):
    """Config e: a 32-stage serial chain, lead time 8 and history 8."""
    m = 32
    cfg = {"num_stages": m, "num_periods": periods, "init_inv": np.full(m, 10.0), "inv_target": np.arange(m) % 3 * 1.0,
           "inv_max": np.full(m, 30.0), "price": np.arange(m + 1, 0, -1).astype(float) + 0.25,
           "stock_cost": 0.1 + 0.3 * (np.arange(m) % 4) / 4, "backlog_cost": 0.4 + 0.5 * (np.arange(m) % 3) / 3,
           "delay": np.full(m, 8), "time_dependency": True, "prev_demand": True, "prev_actions": True, "prev_length": 8,
           "independent": kind == "MAIM", "standardise_state": True, "standardise_actions": True, "a": -1, "b": 1}
    cfg.update(flags)
    return cfg


def serial_big(inv_max, **flags):
    """Config f: serial4 at a capacity without a rescale table (the tables stop at 8 MiB: 4 rows x m nodes x 2 inv_max)."""
    cfg = presets.serial4(prev_actions=True, prev_length=2)
    cfg.update(inv_max=np.full(4, float(inv_max)), init_inv=np.full(4, float(inv_max // 3)), num_periods=10, **flags)
    return cfg


def div_big(inv_max0, **flags):
    """Config f: a divergent net whose factory capacity is large (no table); its children's order_max = inv_max[0]."""
    cfg = _tree({0: [1, 2], 1: [3, 4], 2: [5]}, 6, 10, np.array([1, 2, 1, 3, 2, 1]), 2, **flags)
    cfg["inv_max"] = np.array([float(inv_max0), 60, 50, 40, 40, 40])
    cfg["init_inv"] = np.array([float(inv_max0 // 2), 20, 20, 10, 10, 10])
    return cfg


# the largest inv_max whose serial4 table still fits 8 MiB: 4 rows x 4 nodes x (2 inv_max + 17) doubles
TABLE_EDGE = ((8 << 20) // (4 * 4 * 8) - 17) // 2


def cases():
    """name -> (kind, config, demand mean, action mode).  Action modes: "near_eq" standardised actions around the
    equilibrium, "uniform" in [-1.15, 1.15], "raw" small integral orders for unstandardised actions."""
    return {
        "a_maimdiv_tree32": ("MAIM_div", tree32(share_network=True), 3, "near_eq"),
        "a_imdiv_tree32": ("IM_div", tree32(), 3, "near_eq"),
        "b_maimdiv_tree13": ("MAIM_div", tree_n(13, independent=True), 4, "near_eq"),
        "b_imdiv_tree16": ("IM_div", tree_n(16), 4, "near_eq"),
        "c_maimdiv_star8": ("MAIM_div", star8(), 9, "star"),
        "c_imdiv_star8": ("IM_div", star8(), 9, "star"),
        "d_maimdiv_tree8_d4p2": ("MAIM_div", tree8(4, 2), 5, "near_eq"),
        "d_maimdiv_tree8_d5p2": ("MAIM_div", tree8(5, 2), 5, "near_eq"),
        "d_imdiv_tree8_d4p3": ("IM_div", tree8(4, 3), 5, "near_eq"),
        "e_maim_chain32": ("MAIM", chain32("MAIM"), 5, "uniform"),
        "e_im_chain32": ("IM", chain32("IM"), 5, "uniform"),
        "f_maim_serial_40000": ("MAIM", serial_big(40000), 9000, "uniform"),
        "f_im_serial_40000_raw": ("IM", serial_big(40000, standardise_state=False, standardise_actions=False), 9000, "raw"),
        "f_maimdiv_div_big": ("MAIM_div", div_big(60000), 20, "near_eq"),
        "f_maim_table_edge": ("MAIM", serial_big(TABLE_EDGE), TABLE_EDGE + 50, "uniform"),
        # float32 observations: without a table the kernels convert, at the table's edge they read its float32 copy
        "f_maim_serial_40000_f32": ("MAIM", serial_big(40000, obs_dtype="float32"), 9000, "uniform"),
        "f_maimdiv_div_big_f32": ("MAIM_div", div_big(60000, obs_dtype="float32"), 20, "near_eq"),
        "f_maim_table_edge_f32": ("MAIM", serial_big(TABLE_EDGE, obs_dtype="float32"), TABLE_EDGE + 50, "uniform"),
        "g_maim_t1": ("MAIM", dict(presets.serial4(), num_periods=1), 5, "uniform"),
        "g_imdiv_t2": ("IM_div", dict(presets.div2(prev_actions=True), num_periods=2), 5, "near_eq"),
        "g_maimdiv_t1": ("MAIM_div", dict(presets.div1(), num_periods=1), 5, "near_eq"),
    }


CASES = cases()


def draw(kind, cfg, n, rng, mu, mode):
    """Distinct per-env demand [N, R, T] and actions [T, N, m]."""
    env = im_oracle.OracleEnv(kind, copy_config(cfg))
    m, T, R = env.m, env.T, env.R
    demand = rng.poisson(mu, size=(n, R, T)).astype(np.int32)
    if mode == "raw":
        actions = rng.integers(0, 40, size=(T, n, m)).astype(np.float64) + rng.choice([0.0, 0.5], size=(T, n, m))
    elif mode == "uniform":
        actions = rng.uniform(-1.15, 1.15, size=(T, n, m))
    elif mode == "star":                          # children order a lot (and node 0 little) so that node 0 rations
        actions = np.clip(rng.normal(-0.2, 0.5, size=(T, n, m)), -1, 1)
        actions[:, :, 0] = np.clip(rng.normal(-0.75, 0.2, size=(T, n)), -1, 1)
    else:
        actions = np.clip(rng.normal(-0.6, 0.5, size=(T, n, m)), -1, 1)
    return demand, actions


def python_run(kind, cfg, demand, actions, mask=None):
    """One env through the Python oracle: per-period rewards [T, cols], observations [T + 1, m, O] and the final state."""
    env = im_oracle.OracleEnv(kind, copy_config(cfg))
    obs = [env.reset(demand if env.div else demand.reshape(-1), mask)]
    rew = []
    for t in range(env.T):
        o, r, _, _ = env.step(actions[t])
        obs.append(o)
        rew.append(np.atleast_1d(np.asarray(r, dtype=np.float64)))
    return np.stack(rew), np.stack(obs), env.state_vector()


def assert_oracles_agree(kind, cfg, demand, actions, mask=None):
    N = demand.shape[0]
    got = c_oracle.COracle(kind, cfg).run(demand, actions, mask, all_obs=True)
    assert got["bad"] == 0
    for n in range(N):
        rew, obs, st = python_run(kind, cfg, demand[n], actions[:, n], None if mask is None else mask[n])
        np.testing.assert_array_equal(got["reward"][:, n], rew, err_msg=f"env {n}: reward")
        np.testing.assert_array_equal(got["obs_all"][:, n], obs, err_msg=f"env {n}: obs")
        for k in ("inv", "backlog", "order_u", "pipe"):
            np.testing.assert_array_equal(got[k][n], st[k], err_msg=f"env {n}: {k}")
        if st["backlog_to"].size:
            np.testing.assert_array_equal(got["backlog_to"][n], st["backlog_to"], err_msg=f"env {n}: backlog_to")
    return got


@pytest.mark.parametrize("name", sorted(CASES))
def test_python_and_c_oracles_agree_at_the_limits(name):
    kind, cfg, mu, mode = CASES[name]
    rng = np.random.default_rng(sorted(CASES).index(name))
    demand, actions = draw(kind, cfg, 6, rng, mu, mode)
    assert_oracles_agree(kind, cfg, demand, actions)


@pytest.mark.parametrize("thr", [0.0, 1.0])
@pytest.mark.parametrize("name", ["a_maimdiv_tree32", "e_im_chain32"])
def test_oracles_agree_on_noisy_delay_extremes(name, thr):
    """Config h: threshold 1 delays every arrival until the last period, so goods carry over many consecutive periods."""
    kind, cfg, mu, mode = CASES[name]
    rng = np.random.default_rng(int(thr * 10) + 3)
    demand, actions = draw(kind, cfg, 4, rng, mu, mode)
    T, m = actions.shape[0], actions.shape[2]
    mask = rng.uniform(size=(4, T, m)) <= thr
    assert_oracles_agree(kind, cfg, demand, actions, mask)


def star_activity(kind, cfg, demand, actions):
    """For every period of every env in which node 0 of the star ships less than its children ask for, the number of
    children that take part in the split's drain: those with a positive ledger entry when node 0 has a backlog, else those
    with a positive order.  Returns the set of counts seen."""
    seen = set()
    for n in range(demand.shape[0]):
        env = im_oracle.OracleEnv(kind, copy_config(cfg))
        env.reset(demand[n])
        for t in range(env.T):
            orders = env.decode_orders(actions[t, n])
            wanted = env.backlog[0] + sum(orders[1:])
            avail = env.inv[0] + (env.carry[0] + env.pipe[0][0] if t >= env.delay[0] else env.carry[0])
            if avail < wanted:
                cnt = env.backlog_to[0] if env.backlog[0] > 0 else orders[1:]
                seen.add(sum(1 for v in cnt if v > 0))
            env.step(actions[t, n])
    return seen


@pytest.mark.parametrize("kind", ["MAIM_div", "IM_div"])
def test_star_drains_ration_between_six_seven_and_eight_children(kind):
    """Config c exercises ceil_div_pos with 6, 7 and 8 active children: shown on the oracle's own trajectory."""
    cfg = CASES[f"c_{kind.lower().replace('_', '')}_star8"][1]
    _, _, mu, mode = CASES[f"c_{kind.lower().replace('_', '')}_star8"]
    demand, actions = draw(kind, cfg, 16, np.random.default_rng(7), mu, mode)
    seen = star_activity(kind, cfg, demand, actions)
    assert {6, 7, 8} <= seen, seen


# ---------------------------------------------------------------------------------------------------------------------
# the split watchdog at demand_max near INT32_MAX
# ---------------------------------------------------------------------------------------------------------------------
def watchdog_cfg(kind, nchild, inv_max0, periods=2, init0=0):
    """A star whose factory capacity makes demand_max[0] = nchild * inv_max0 (the children's order_max is inv_max[0])."""
    m = nchild + 1
    cfg = _tree({0: list(range(1, m))}, m, periods, 1, 1, prev_actions=False)
    cfg["inv_max"] = np.array([float(inv_max0)] + [30.0] * nchild)
    cfg["init_inv"] = np.array([float(init0)] + [10.0] * nchild)
    return cfg


# IM_div's LOOP1 limit is 4 * demand_max and the others 2 * demand_max: with demand_max[0] = 2^29 the first wraps, with
# 5 * 2^28 the second.  Two periods: the first leaves node 0 a backlog (it starts empty), the second drains it with LOOP1
# (node 0's own order arrives).  One period: node 0 holds 3 units, less than its children ask for (LOOP4).
WATCHDOG_CASES = {"imdiv_2x2^28_loop1": ("IM_div", 2, 1 << 28, 2, 0), "imdiv_8x2^26_loop1": ("IM_div", 8, 1 << 26, 2, 0),
                  "imdiv_5x2^28_loop4": ("IM_div", 5, 1 << 28, 1, 3)}


def watchdog_case(case):
    kind, nchild, inv0, periods, init0 = WATCHDOG_CASES[case]
    return kind, watchdog_cfg(kind, nchild, inv0, periods, init0)


def watchdog_inputs(kind, cfg, n, rng):
    """Small integral orders (standardised actions that decode exactly to them); node 0 orders 40 units in the first period."""
    env = im_oracle.OracleEnv(kind, copy_config(cfg))
    demand = rng.integers(3, 9, size=(n, env.R, env.T)).astype(np.int32)
    om = np.asarray(env.order_max, dtype=np.float64)
    raw = rng.integers(1, 6, size=(env.T, n, env.m)).astype(np.float64)
    raw[..., 0] = 0.0
    raw[0, :, 0] = 40.0
    actions = -1.0 + 2.0 * raw / om
    return demand, actions


def watchdog_loop_ran(kind, cfg, demand, actions):
    """True when the split drained node 0's backlog in period 1 (LOOP1), or rationed goods in period 0 (LOOP4)."""
    env = im_oracle.OracleEnv(kind, copy_config(cfg))
    env.reset(demand)
    _, _, _, info = env.step(actions[0])
    if env.T == 1:
        return 0 < info["ship"][0] < info["demand"][0]
    if env.backlog[0] <= 0:
        return False
    _, _, _, info = env.step(actions[1])
    return info["ship"][0] >= info["demand"][0]


@pytest.mark.parametrize("case", sorted(WATCHDOG_CASES))
def test_c_oracle_watchdog_limit_does_not_wrap(case):
    kind, cfg = watchdog_case(case)
    env = im_oracle.OracleEnv(kind, copy_config(cfg))
    assert env.demand_max[0] * (4 if env.T > 1 else 2) > INT32_MAX       # the limit the split used to wrap
    demand, actions = watchdog_inputs(kind, cfg, 5, np.random.default_rng(1))
    got = assert_oracles_agree(kind, cfg, demand, actions)
    assert not got["err"].any()
    assert all(watchdog_loop_ran(kind, cfg, demand[n], actions[:, n]) for n in range(5))


# ---------------------------------------------------------------------------------------------------------------------
# runtime specialisation at the limits
# ---------------------------------------------------------------------------------------------------------------------
def imx_config(kind, cfg, n=8192, **extra):
    return ENV_CLASSES[kind](dict(copy_config(cfg), num_envs=n, _config_only=True, **extra)).imx_config


@pytest.mark.parametrize("kind,name,variants", [("MAIM_div", "a_maimdiv_tree32", (0, 1, 2, 3, 4)), ("IM_div", "a_imdiv_tree32", (0, 1, 3, 4)),
                                                ("MAIM", "e_maim_chain32", (0, 1, 2, 3, 4))])
def test_specialised_kernels_compile_at_the_limits(kind, name, variants):
    c = imx_config(kind, CASES[name][1])
    lib = _lib.load()
    for v in variants:
        buf = ctypes.create_string_buffer(8192)
        size = lib.imx_jit_compile_check(ctypes.byref(c), v, buf, 8192)
        assert size > 10000, (name, v, size, buf.value.decode()[:600], lib.imx_last_error())


# ---------------------------------------------------------------------------------------------------------------------
# the int32 domain: imx_create refuses configs whose state could wrap, before it looks for a device
# ---------------------------------------------------------------------------------------------------------------------
def create(kind, cfg, **extra):
    """imx_create's return code and message; a handle created on a GPU machine is destroyed again.  cfg["noisy_delay"] asks
    for the carry state (the serial envs only ask for it at a noisy reset)."""
    lib = _lib.load()
    c = imx_config(kind, cfg, n=64, **extra)
    c.noisy_delay = int(bool(cfg.get("noisy_delay", False)))
    h = ctypes.c_void_p()
    rc = lib.imx_create(ctypes.byref(c), ctypes.byref(h))
    msg = lib.imx_last_error().decode() if rc else ""
    if rc == 0:
        lib.imx_destroy(h)
    return rc, msg


def _in_domain(rc):
    return rc in (0, -2)                              # -2: no CUDA device on this machine


def carry_cfg(periods):
    """serial4 at 2^28 with noisy delays: inv_max + T * order_max fits int32 for T <= 6."""
    cfg = serial_big(1 << 28, noisy_delay=True)
    cfg.update(num_periods=periods, delay=np.ones(4, dtype=np.int64), init_inv=np.zeros(4))
    return cfg


OUT_OF_DOMAIN = {
    # 8 children at 2^28: demand_max[0] = 2^31
    "demand_max_8x2^28": ("MAIM_div", lambda: watchdog_cfg("MAIM_div", 8, 1 << 28, periods=1), "demand_max[0]"),
    # IM with raw state: 9 periods x 2^28 of unmet demand
    "im_uncapped_backlog": ("IM", lambda: dict(serial_big(1 << 28, standardise_state=False, standardise_actions=False), num_periods=9),
                            "uncapped backlog"),
    # the same reached at an ordinary capacity by a long episode
    "im_uncapped_backlog_long": ("IM", lambda: dict(serial_big(50000, standardise_state=False), num_periods=50000), "uncapped backlog"),
    "imdiv_uncapped_backlog": ("IM_div", lambda: dict(div_big(1 << 27, standardise_state=False), num_periods=20), "uncapped backlog"),
    # MAIM with raw state does not cap the backlog either
    "maim_uncapped_backlog": ("MAIM", lambda: dict(serial_big(1 << 28, standardise_state=False), num_periods=9), "uncapped backlog"),
    # a split node's per-child ledger is never capped
    "maimdiv_ledger": ("MAIM_div", lambda: watchdog_cfg("MAIM_div", 2, 1 << 28, periods=5), "ledger"),
    # the noisy-delay carry holds every arrival of a run of delayed periods: 2^28 + 10 x 2^28
    "maim_noisy_carry": ("MAIM", lambda: carry_cfg(10), "noisy delays"),
    # the same at an ordinary capacity over a long episode: 65 535 x 40 000
    "maim_noisy_carry_long": ("MAIM", lambda: dict(serial_big(40000), num_periods=65535, noisy_delay=True), "noisy delays"),
    # a divergent child may receive twice what it orders: node 5 orders up to inv_max[2] = 2^27, 40 + 2 x 10 x 2^27
    "maimdiv_noisy_carry_child": ("MAIM_div", lambda: dict(div_big(60000), num_periods=10, noisy_delay=True,
                                                             inv_max=np.array([60000.0, 60, 1 << 27, 40, 40, 40])), "noisy delays"),
}
IN_DOMAIN = {
    "maimdiv_7x2^28_t1": ("MAIM_div", lambda: watchdog_cfg("MAIM_div", 7, 1 << 28, periods=1)),
    "imdiv_2x2^28_t3": ("IM_div", lambda: watchdog_cfg("IM_div", 2, 1 << 28, periods=3)),
    **{"watchdog_" + k: (WATCHDOG_CASES[k][0], lambda k=k: watchdog_case(k)[1]) for k in WATCHDOG_CASES},
    "im_uncapped_backlog_t7": ("IM", lambda: dict(serial_big(1 << 28, standardise_state=False, standardise_actions=False), num_periods=7)),
    "maim_capped_2^28_long": ("MAIM", lambda: dict(serial_big(1 << 28), num_periods=65535)),
    "im_std_state_long": ("IM", lambda: dict(serial_big(50000), num_periods=50000)),
    "maim_noisy_carry_t6": ("MAIM", lambda: carry_cfg(6)),
    "maim_noisy_long_small": ("MAIM", lambda: dict(serial_big(30000), num_periods=65535, noisy_delay=True)),
}


@pytest.mark.parametrize("case", sorted(OUT_OF_DOMAIN))
def test_create_refuses_configs_whose_int32_state_could_wrap(case):
    kind, make, words = OUT_OF_DOMAIN[case]
    rc, msg = create(kind, make())
    assert rc == -1, (rc, msg)
    assert words in msg and "INT32_MAX" in msg, msg


@pytest.mark.parametrize("case", sorted(IN_DOMAIN))
def test_create_accepts_the_edge_of_the_int32_domain(case):
    kind, make = IN_DOMAIN[case]
    rc, msg = create(kind, make())
    assert _in_domain(rc), (rc, msg)


def test_oracles_agree_at_the_edge_of_the_carry_bound():
    """Every arrival held back until the last period at 2^28 capacity, on the largest T the domain accepts."""
    kind, cfg = "MAIM", carry_cfg(6)
    demand = np.full((3, 1, 6), 5, dtype=np.int32)
    actions = np.full((6, 3, 4), 1.0)                 # every stage orders order_max = 2^28
    mask = np.ones((3, 6, 4), dtype=bool)
    assert_oracles_agree(kind, cfg, demand, actions, mask)
    _, _, st = python_run(kind, cfg, demand[0], actions[:, 0], mask[0])
    assert st["inv"][3] == 1 << 28                    # the factory stage received 5 x 2^28 at the last period (clipped)
