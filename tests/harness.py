"""Shared trajectory runners for the parity tests.

``run_reference`` drives the UNMODIFIED reference env (only where its source tree is present, see oracle/ref_import.py),
``run_oracle`` drives oracle/im_oracle.py; both return the same dict of arrays so the
tests can compare them (and the CUDA path) field by field:

    obs      [T+1, m, O] float64   (obs[0] = after reset)
    reward   [T, m] float64        (IM kinds: the scalar repeated in column 0, rest 0)
    demand / ship / acq / order / profit   [T, m] float64
    inv / backlog / order_u               [T+1, m] int64   (state at the start of each period)
"""
from __future__ import annotations

import os
import sys
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import im_oracle  # noqa: E402
from oracle.ref_import import load_reference, reference_available  # noqa: E402,F401

KIND_TO_CLASS = {"IM": "InvManagement", "MAIM": "MultiAgentInvManagement",
                 "IM_div": "InvManagementDiv", "MAIM_div": "MultiAgentInvManagementDiv"}


def agent_names(kind, m):
    prefix = "node_" if kind.endswith("_div") else "stage_"
    return [prefix + str(i) for i in range(m)]


def copy_config(cfg):
    out = {}
    for k, v in cfg.items():
        out[k] = v.copy() if isinstance(v, np.ndarray) else (dict(v) if isinstance(v, dict) else v)
    return out


def make_delay_mask(kind, delay, T, thr, rng):
    """Bernoulli(u <= thr) per (period, stage); the reference only consumes a draw when
    t >= delay[i] (MAIM_env.py:447-452), other entries are ignored by all implementations."""
    m = len(delay)
    return rng.uniform(0, 1, size=(T, m)) <= thr


def _uniform_replayer(kind, delay, T, mask):
    """Builds the sequence of ``np.random.uniform`` return values that makes the reference
    reproduce ``mask``: draw order is factory first (serial: stage m-1, then 0..m-2;
    divergent: node 0, then 1..m-1), one draw per eligible stage per period."""
    m = len(delay)
    order = ([m - 1] + list(range(m - 1))) if not kind.endswith("_div") else list(range(m))
    seq = []
    for t in range(T):
        for i in order:
            if t - delay[i] >= 0:
                seq.append(0.0 if mask[t, i] else 1.0)
    return seq


def run_reference(kind, cfg, demand, actions, delay_mask=None):
    R = load_reference()
    cls = getattr(R, KIND_TO_CLASS[kind])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        env = cls(copy_config(cfg))
        m, T = env.num_nodes, env.num_periods
        names = agent_names(kind, m)
        multi = kind.startswith("MAIM")
        saved_uniform = np.random.uniform
        try:
            if delay_mask is not None:
                seq = iter(_uniform_replayer(kind, [int(d) for d in env.delay], T, delay_mask))
                np.random.uniform = lambda *a, **k: next(seq)
                obs0 = env.reset(customer_demand=np.array(demand), noisy_delay=True, noisy_delay_threshold=0.5)
            else:
                obs0 = env.reset(customer_demand=np.array(demand))

            def pack(o):
                return np.stack([o[n] for n in names]) if multi else np.array(o)

            obs = [pack(obs0)]
            out = {k: np.zeros((T, m)) for k in ("reward", "demand", "ship", "acq", "order", "profit")}
            for t in range(T):
                if multi:
                    act = {names[i]: np.array([actions[t, i]]) for i in range(m)}
                else:
                    act = np.array(actions[t])
                o, r, done, info = env.step(act)
                obs.append(pack(o))
                if multi:
                    for i, n in enumerate(names):
                        out["reward"][t, i] = r[n]
                        out["demand"][t, i] = info[n]["demand"]
                        out["ship"][t, i] = info[n]["ship"]
                        out["acq"][t, i] = info[n]["acquisition"]
                        out["order"][t, i] = info[n]["actual order"]
                        out["profit"][t, i] = info[n]["profit"]
                    assert done["__all__"] == (t == T - 1)
                else:
                    out["reward"][t, 0] = r
                    out["demand"][t] = info["demand"]
                    out["ship"][t] = info["ship"]
                    out["acq"][t] = info["acquisition"]
                    out["order"][t] = env.order_r[t]
                    out["profit"][t] = info["profit"]
                    assert done == (t == T - 1)
        finally:
            np.random.uniform = saved_uniform
    out["obs"] = np.stack(obs)
    out["inv"] = env.inv.astype(np.int64)
    out["backlog"] = env.backlog.astype(np.int64)
    out["order_u"] = env.order_u.astype(np.int64)
    return out


def run_oracle(kind, cfg, demand, actions, delay_mask=None):
    env = im_oracle.OracleEnv(kind, copy_config(cfg))
    m, T = env.m, env.T
    obs = [env.reset(np.array(demand), delay_mask)]
    out = {k: np.zeros((T, m)) for k in ("reward", "demand", "ship", "acq", "order", "profit")}
    st = {k: [np.array(getattr(env, k), dtype=np.int64)] for k in ("inv", "backlog", "order_u")}
    for t in range(T):
        o, r, done, info = env.step(actions[t])
        obs.append(o)
        if env.multi:
            out["reward"][t] = r
        else:
            out["reward"][t, 0] = r
        out["demand"][t] = info["demand"]
        out["ship"][t] = info["ship"]
        out["acq"][t] = info["acquisition"]
        out["order"][t] = info["actual order"]
        out["profit"][t] = info["profit"]
        for k in st:
            st[k].append(np.array(getattr(env, k), dtype=np.int64))
        assert done == (t == T - 1)
    out["obs"] = np.stack(obs)
    for k in st:
        out[k] = np.stack(st[k])
    return out


def assert_same(a, b, what=""):
    """Bit-exact on every field (the oracle restates the same IEEE operations in the same order)."""
    for k in ("inv", "backlog", "order_u"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=f"{what}: {k}")
    for k in ("demand", "ship", "acq", "order", "profit", "reward", "obs"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=f"{what}: {k}")


def random_case(kind, cfg, rng, mu=5.0, action_mode="uniform"):
    """Random demand trace + action trace for one episode of ``cfg``."""
    div = kind.endswith("_div")
    m = cfg["num_nodes"] if div else cfg["num_stages"]
    T = cfg["num_periods"]
    std_actions = cfg.get("standardise_actions", True) or kind == "MAIM_div"
    if div:
        conn = cfg["connections"]
        R = sum(1 for k in range(m) if not conn.get(k))
        demand = rng.poisson(mu, size=(R, T))
    else:
        demand = rng.poisson(mu, size=T)
    if std_actions:
        if action_mode == "uniform":
            actions = rng.uniform(-1.15, 1.15, size=(T, m))        # slightly out of range on purpose
        else:                                                      # near-equilibrium (exercises every split branch)
            actions = np.clip(rng.normal(-0.6, 0.5, size=(T, m)), -1, 1)
    else:
        actions = rng.uniform(-3, 36, size=(T, m))
        half = rng.uniform(size=(T, m)) < 0.2                      # exact .5 values: round-half-to-even
        actions = np.where(half, np.floor(actions) + 0.5, actions)
    return demand, actions


# --------------------------------------------------------------------------------------
# golden fixtures (generated from the reference by tests/golden/make_golden.py)
# --------------------------------------------------------------------------------------
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def golden_names():
    return sorted(f[:-4] for f in os.listdir(GOLDEN_DIR) if f.endswith(".npz"))


def load_golden(name):
    import json
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False)
    raw = json.loads(str(z["config"]))
    cfg = {}
    for k, v in raw.items():
        if isinstance(v, dict) and "__nd__" in v:
            cfg[k] = np.array(v["__nd__"], dtype=v["dtype"])
        elif isinstance(v, dict) and "__dict__" in v:
            cfg[k] = {int(a): list(b) for a, b in v["__dict__"].items()}
        else:
            cfg[k] = v
    mask = z["delay_mask"]
    g = {k: z[k] for k in ("obs", "reward", "demand", "ship", "acq", "order", "profit", "inv", "backlog", "order_u")}
    return dict(kind=str(z["kind"]), config=cfg, demand_trace=z["demand_trace"], actions=z["actions"],
                delay_mask=(mask if mask.size else None), ref=g)


# --------------------------------------------------------------------------------------
# random divergent networks (breadth-first numbering: a child never has a smaller index than its parent,
# utils.py:87-92, and the last node is among the deepest, which the reference's price tables assume)
# --------------------------------------------------------------------------------------
def random_tree_config(rng, m, max_children=4, periods=20, **flags):
    conn = {i: [] for i in range(m)}
    nxt, frontier = 1, [0]
    while nxt < m:
        parent = frontier.pop(0) if frontier else nxt - 1
        k = int(rng.integers(1 if (not frontier) else 0, max_children + 1))
        k = min(k, m - nxt)
        for _ in range(k):
            conn[parent].append(nxt)
            frontier.append(nxt)
            nxt += 1
    cfg = {"num_nodes": m, "num_periods": periods, "connections": conn,
           "init_inv": rng.integers(5, 15, m).astype(float), "inv_target": rng.integers(0, 4, m).astype(float),
           "inv_max": rng.integers(20, 45, m).astype(float), "stock_cost": rng.uniform(0.1, 0.5, m),
           "backlog_cost": rng.uniform(0.3, 0.9, m), "delay": rng.integers(1, 5, m),
           "time_dependency": True, "prev_demand": True, "prev_actions": False, "prev_length": 1,
           "independent": False, "share_network": False}
    cfg.update(flags)
    return cfg


def random_serial_config(rng, m, periods=16):
    """A random serial chain: heterogeneous capacities, targets, costs, lead times, a random rescale interval and a random
    legal observation mode (prices strictly decreasing, MAIM_env.py:167-168)."""
    a, b = [(-1, 1), (0, 1), (-2, 2), (0, 3)][int(rng.integers(0, 4))]
    td, pd, pa = bool(rng.integers(0, 2)), bool(rng.integers(0, 2)), bool(rng.integers(0, 2))
    cfg = {"num_stages": m, "num_periods": periods, "init_inv": rng.integers(3, 15, m).astype(float),
           "inv_target": rng.integers(0, 5, m).astype(float) + rng.choice([0.0, 0.5], m),
           "inv_max": rng.integers(15, 45, m).astype(float), "price": np.arange(m + 1, 0, -1).astype(float) + rng.uniform(0, 0.9),
           "stock_cost": rng.uniform(0.1, 0.5, m), "backlog_cost": rng.uniform(0.3, 0.9, m), "delay": rng.integers(1, 6, m),
           "time_dependency": td, "prev_demand": pd, "prev_actions": pa, "prev_length": int(rng.integers(1, 5)),
           "independent": bool(rng.integers(0, 2)), "standardise_state": True, "standardise_actions": bool(rng.integers(0, 2)),
           "a": a, "b": b}
    return cfg
