#!/usr/bin/env python
"""Per-handle I/O element types: bfloat16 observations and float32 actions against float64 / float32-observation handles.

In one process, alternating the (observation, action) dtype pairs (f64, f64), (f32, f64), (bf16, f64), (bf16, f32), after
checking that their outputs agree bit for bit (bf16 = the float32 handle's observations rounded by torch, rewards equal):
  - imx_step: us per launch, the median over rounds of a captured 30-step graph (config 2 at 65 536, 1 Mi and 4 Mi envs;
    div2 at 262 144 envs), with the algorithmic bytes per env-step B = 8 S + 4 R + m (act + 8 + O obs) and their share of the
    6 542 GB/s device copy peak measured on the B200 (DESIGN.md section 7);
  - imx_step_many with observations (K = 30) at 1 Mi envs; imx_replay_episode (observations + rewards + statistics) at 65 536;
  - imx_step_host at 65 536 envs, zero-copy and staged;
  - the stand-in policy loop of examples/rl_loop_cuda_graph.py per period: float32 observations -> bf16 linear policy -> a
    float64 action copy, against bf16 observations -> the same policy -> float32 actions written into the env's buffer.
One JSON line per measurement, each with the card's name, power limit and max SM clock.

    python benchmarks/bench_io_dtypes.py [--rounds 7] [--out results/r3_io_dtypes.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from marl_for_im_b200 import _lib, presets  # noqa: E402
from marl_for_im_b200.envs import ENV_CLASSES  # noqa: E402

PAIRS = [("float64", "float64"), ("float32", "float64"), ("bfloat16", "float64"), ("bfloat16", "float32")]
ES = {"float64": 8, "float32": 4, "bfloat16": 2}
COPY_PEAK_GBS = 6542.0
DEV = "cuda:0"


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:
        q = f"unknown ({exc})"
    return {"gpu": torch.cuda.get_device_name(0), "power_limit_and_max_sm_clock": q}


def make(kind, preset, n, obs, act):
    return ENV_CLASSES[kind](dict(presets.PRESETS[preset](), num_envs=n, return_info=False, obs_dtype=obs, action_dtype=act))


def bytes_per_env_step(env, obs, act):
    m, O, R, S = env.num_nodes, env.obs_len, len(env._retailers), env.state_words
    return 8 * S + 4 * R + m * (ES[act] + 8 + O * ES[obs])


def capture(fn):
    """A graph of fn(stream).  The caller keeps every tensor the graph reads or writes alive as long as the graph: entering a
    capture empties torch's allocator cache, so a tensor freed after an earlier capture is unmapped, not just reused."""
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn(s.cuda_stream)
        s.synchronize()
        with torch.cuda.graph(g, stream=s):
            fn(torch.cuda.current_stream().cuda_stream)
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(2):
        g.replay()
    torch.cuda.synchronize()
    return g


def time_graph(g):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3


def setup_step(kind, preset, n, obs, act, K=30):
    """a handle, its K-period action block (values exact in float32) and a graph of K steps (the period counter is reset on the
    host before every replay)"""
    env = make(kind, preset, n, obs, act)
    _lib.check(env._lib.imx_prepare(env._handle, 0))
    m, O = env.num_nodes, env.obs_len
    gen = torch.Generator(device=DEV).manual_seed(1)
    a = (torch.rand((K, n, m), generator=gen, device=DEV) * 2.3 - 1.15).to(getattr(torch, act))
    ob = torch.empty((n, m, O), dtype=getattr(torch, obs), device=DEV)
    rw = torch.empty((n, m) if env.MULTI else (n,), dtype=torch.float64, device=DEV)
    lib, h = env._lib, env._handle

    def body(s):
        lib.imx_set_period(h, 0)
        for t in range(K):
            _lib.check(lib.imx_step(h, C.c_void_p(a[t].data_ptr()), C.c_void_p(ob.data_ptr()), C.c_void_p(rw.data_ptr()), None, C.c_void_p(s)))

    env.reset()
    g = capture(body)
    return env, g, ob, rw, a


def step_rows(rounds, info):
    out = []
    for name, kind, preset, n in (("config2_serial4", "MAIM", "serial4", 65536), ("config2_serial4_1Mi", "MAIM", "serial4", 1 << 20),
                                  ("config2_serial4_4Mi", "MAIM", "serial4", 4 << 20), ("div2", "MAIM_div", "div2", 262144)):
        runs = {p: setup_step(kind, preset, n, *p) for p in PAIRS}
        # outputs first: one graph (30 periods from the same reset state) per pair, then compare the last period's outputs
        for p, (env, g, ob, rw, a) in runs.items():
            env.reset()
            env._lib.imx_set_period(env._handle, 0)
            g.replay()
        torch.cuda.synchronize()
        ref_obs32, ref_rew = runs[("float32", "float64")][2], runs[("float64", "float64")][3]
        same = all(torch.equal(rw, ref_rew) for (_, _, _, rw, _) in runs.values())
        same &= torch.equal(runs[("float64", "float64")][2].float(), ref_obs32)
        for p in (("bfloat16", "float64"), ("bfloat16", "float32")):
            same &= torch.equal(runs[p][2].view(torch.int16), ref_obs32.to(torch.bfloat16).view(torch.int16))
        times = {p: [] for p in PAIRS}
        for _ in range(rounds):                          # alternating the pairs inside every round
            for p, (env, g, *_rest) in runs.items():
                env._lib.imx_set_period(env._handle, 0)
                times[p].append(time_graph(g) / 30.0)
        variants = {f"{p[0]}/{p[1]}": runs[p][0]._lib.imx_kernel_variant(runs[p][0]._handle) for p in PAIRS}
        for p in PAIRS:
            env = runs[p][0]
            us = statistics.median(times[p])
            b = bytes_per_env_step(env, *p)
            out.append(dict(info, measurement="imx_step", workload=name, envs=n, obs_dtype=p[0], action_dtype=p[1], identical_outputs=bool(same),
                            us_per_launch=us, us_rounds=times[p], bytes_per_env_step=b,
                            copy_peak_fraction=b * n / (us * 1e-6) / (COPY_PEAK_GBS * 1e9), kernel_variants=variants))
        del runs
        torch.cuda.empty_cache()
    return out


def step_many_rows(rounds, info, n=1 << 20, K=30):
    out, runs = [], {}
    for p in PAIRS:
        env = make("MAIM", "serial4", n, *p)
        m, O = env.num_nodes, env.obs_len
        gen = torch.Generator(device=DEV).manual_seed(2)
        a = (torch.rand((K, n, m), generator=gen, device=DEV) * 2.3 - 1.15).to(getattr(torch, p[1]))
        ob = torch.empty((K, n, m, O), dtype=getattr(torch, p[0]), device=DEV)
        rw = torch.empty((K, n, m), dtype=torch.float64, device=DEV)
        lib, h = env._lib, env._handle

        def body(s, lib=lib, h=h, a=a, ob=ob, rw=rw):
            lib.imx_set_period(h, 0)
            _lib.check(lib.imx_step_many(h, C.c_void_p(a.data_ptr()), K, C.c_void_p(ob.data_ptr()), C.c_void_p(rw.data_ptr()), None, C.c_void_p(s)))
        env.reset()
        runs[p] = (env, capture(body), ob, rw, body)    # (body's defaults keep the graph's input tensors alive)
    times = {p: [] for p in PAIRS}
    for _ in range(rounds):
        for p, (env, g, *_keep) in runs.items():
            env._lib.imx_set_period(env._handle, 0)
            times[p].append(time_graph(g))
    for p, (env, g, *_keep) in runs.items():
        out.append(dict(info, measurement="imx_step_many", workload="config2_serial4_1Mi", envs=n, periods=K, obs_dtype=p[0], action_dtype=p[1],
                        us_per_call=statistics.median(times[p]), us_rounds=times[p], kernel_variant=env._lib.imx_kernel_variant(env._handle)))
    del runs
    torch.cuda.empty_cache()
    return out


def replay_rows(rounds, info, n=65536):
    out, runs = [], {}
    for p in PAIRS:
        env = make("MAIM", "serial4", n, *p)
        _lib.check(env._lib.imx_prepare(env._handle, _lib.PREPARE_EPISODE))
        m, O, T = env.num_nodes, env.obs_len, env.num_periods
        gen = torch.Generator(device=DEV).manual_seed(3)
        a = (torch.rand((T, n, m), generator=gen, device=DEV) * 2.3 - 1.15).to(getattr(torch, p[1]))
        ob = torch.empty((T, n, m, O), dtype=getattr(torch, p[0]), device=DEV)
        rw = torch.empty((T, n, m), dtype=torch.float64, device=DEV)
        st = torch.zeros(3 + 2 * m, dtype=torch.float64, device=DEV)
        lib, h = env._lib, env._handle

        def body(s, lib=lib, h=h, a=a, ob=ob, rw=rw, st=st):
            _lib.check(lib.imx_replay_episode(h, None, None, 0, 1, C.c_void_p(a.data_ptr()), C.c_void_p(ob.data_ptr()), C.c_void_p(rw.data_ptr()),
                                              None, C.c_void_p(st.data_ptr()), 0, None, C.c_void_p(s)))
        runs[p] = (env, capture(body), body)
    times = {p: [] for p in PAIRS}
    for _ in range(rounds):
        for p, (env, g, _body) in runs.items():
            times[p].append(time_graph(g))
    for p, (env, g, _body) in runs.items():
        out.append(dict(info, measurement="imx_replay_episode", workload="config2_serial4", outputs="obs+rewards+stats", envs=n, obs_dtype=p[0],
                        action_dtype=p[1], us_per_episode=statistics.median(times[p]), us_rounds=times[p],
                        kernel_variant=env._lib.imx_kernel_variant(env._handle)))
    return out


def host_rows(rounds, info, n=65536, steps=30):
    out = []
    for zc in ("1", "0"):
        os.environ["IMX_HOST_ZERO_COPY"] = zc
        runs = {}
        for p in PAIRS:
            env = make("MAIM", "serial4", n, *p)
            m, O = env.num_nodes, env.obs_len
            a = (torch.rand((n, m)) * 2.3 - 1.15).to(getattr(torch, p[1])).pin_memory()
            ob = torch.empty((n, m, O), dtype=getattr(torch, p[0])).pin_memory()
            rw = torch.empty((n, m), dtype=torch.float64).pin_memory()
            _lib.check(env._lib.imx_prepare(env._handle, 4))
            runs[p] = (env, a, ob, rw)
        times = {p: [] for p in PAIRS}
        for _ in range(rounds):
            for p, (env, a, ob, rw) in runs.items():
                lib, h = env._lib, env._handle
                lib.imx_set_period(h, 0)
                t0 = time.perf_counter()
                for _t in range(steps):
                    _lib.check(lib.imx_step_host(h, C.c_void_p(a.data_ptr()), C.c_void_p(ob.data_ptr()), C.c_void_p(rw.data_ptr())))
                times[p].append((time.perf_counter() - t0) / steps * 1e6)
        for p in PAIRS:
            out.append(dict(info, measurement="imx_step_host", workload="config2_serial4", envs=n, zero_copy=zc == "1", obs_dtype=p[0],
                            action_dtype=p[1], us_per_step=statistics.median(times[p]), us_rounds=times[p]))
    os.environ.pop("IMX_HOST_ZERO_COPY", None)
    return out


def policy_rows(rounds, info, n=65536, hidden=256):
    """One period of an RL loop: the policy reads the observations, writes actions, the env steps.  The stand-in policy is a
    bf16 two-layer MLP (torch / cuBLAS GEMMs) over each agent's observation row."""
    out, runs = [], {}
    for name, (obs, act) in (("f32_obs_f64_action_copy", ("float32", "float64")), ("bf16_obs_f32_actions_in_place", ("bfloat16", "float32"))):
        env = make("MAIM", "serial4", n, obs, act)
        _lib.check(env._lib.imx_prepare(env._handle, 0))
        m, O = env.num_nodes, env.obs_len
        gen = torch.Generator(device=DEV).manual_seed(4)
        w1 = (torch.randn((hidden, O), generator=gen, device=DEV) * 0.3).to(torch.bfloat16)
        w2 = (torch.randn((1, hidden), generator=gen, device=DEV) * 0.1).to(torch.bfloat16)
        ob = torch.zeros((n, m, O), dtype=getattr(torch, obs), device=DEV)
        rw = torch.empty((n, m), dtype=torch.float64, device=DEV)
        act_buf = torch.zeros((n, m), dtype=getattr(torch, act), device=DEV)
        lib, h = env._lib, env._handle

        def body(s, lib=lib, h=h, ob=ob, rw=rw, act_buf=act_buf, w1=w1, w2=w2, obs=obs):
            lib.imx_set_period(h, 0)
            for _t in range(30):
                x = ob if obs == "bfloat16" else ob.to(torch.bfloat16)
                y = torch.nn.functional.linear(torch.relu(torch.nn.functional.linear(x, w1)), w2).reshape(n, m)
                if obs == "bfloat16":
                    torch.tanh(y.float(), out=act_buf)          # float32 output layer straight into the env's action buffer
                else:
                    act_buf.copy_(torch.tanh(y.float()))         # float32 -> the float64 action buffer
                _lib.check(lib.imx_step(h, C.c_void_p(act_buf.data_ptr()), C.c_void_p(ob.data_ptr()), C.c_void_p(rw.data_ptr()), None, C.c_void_p(s)))
        env.reset()
        runs[name] = (env, capture(body), body)
    times = {k: [] for k in runs}
    for _ in range(rounds):
        for k, (env, g, _body) in runs.items():
            env._lib.imx_set_period(env._handle, 0)
            times[k].append(time_graph(g) / 30.0)
    for k in runs:
        out.append(dict(info, measurement="policy_loop_period", workload="config2_serial4", envs=n, variant=k, policy=f"bf16 MLP {hidden} hidden",
                        us_per_period=statistics.median(times[k]), us_rounds=times[k]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default="results/r3_io_dtypes.jsonl")
    ap.add_argument("--only", default="step,many,replay,host,policy")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this benchmark measures on the device only")
    info = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    parts = {"step": step_rows, "many": step_many_rows, "replay": replay_rows, "host": host_rows, "policy": policy_rows}
    with open(args.out, "w") as f:
        for k in args.only.split(","):
            for row in parts[k](args.rounds, info):
                f.write(json.dumps(row) + "\n")
                f.flush()
                print({kk: (round(v, 3) if isinstance(v, float) else v) for kk, v in row.items() if kk not in ("us_rounds",)}, flush=True)


if __name__ == "__main__":
    np.random.seed(0)
    main()
