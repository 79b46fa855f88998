#!/usr/bin/env python
"""imx_step_eval (one launch per closed-loop evaluation period: step + returns + evaluation accumulators) against the route it
replaces, each arm captured as one CUDA graph of reset + T periods on pre-staged per-period actions (the policy is left out, so
the env side is isolated).  The arms alternate round by round in one process, and their outputs are compared bit for bit
before any timing:
  (a)  imx_step with imx_info_out.profit + imx_eval_accumulate + a torch returns add (today's route)
  (b)  imx_step_eval with returns and accumulators
  (a') imx_step + a torch returns add (returns only)
  (b') imx_step_eval with returns only
  (c)  plain imx_step (the floor)
Every arm writes the observations and the rewards each period, as a closed loop needs them.

Workloads: config 2 (serial 4-stage) at 65 536 and 1 Mi envs, config 4 div1 / div2 at 262 144 and 32 768 envs (one 8-GPU
shard), each with float64 observations and with bfloat16 observations + float32 actions.  One JSON line per row with the card's
name, power limit and maximum SM clock.

    python benchmarks/bench_step_eval.py [--rounds 7] [--reps 10] [--out results/r3_step_eval.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from marl_for_im_b200 import _lib, presets  # noqa: E402
from marl_for_im_b200.envs import ENV_CLASSES  # noqa: E402

WORKLOADS = [("config2_serial4", "MAIM", presets.serial4, 65536), ("config2_serial4_1Mi", "MAIM", presets.serial4, 1 << 20),
             ("config4_div1", "MAIM_div", presets.div1, 262144), ("config4_div2", "MAIM_div", presets.div2, 262144),
             ("config4_div1_shard8", "MAIM_div", presets.div1, 32768), ("config4_div2_shard8", "MAIM_div", presets.div2, 32768)]
IO = {"f64": {}, "bf16_obs_f32_act": {"obs_dtype": "bfloat16", "action_dtype": "float32"}}
ARMS = ("a", "b", "a_ret", "b_ret", "c")


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:                                   # the number is still reported, marked as unknown
        q = f"unknown ({exc})"
    return {"gpu": name, "power_limit_and_max_sm_clock": q}


def capture(fn):
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn(s.cuda_stream)
        s.synchronize()
        with torch.cuda.graph(g, stream=s):
            fn(torch.cuda.current_stream().cuda_stream)
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    return g


def time_ms(g, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def bytes_per_env_step(env, arm):
    """Bytes one period moves per env, from shapes (config 2 float64: plain step 476 B, arm (b) 668 B)."""
    m, O, S, R = env.num_nodes, env.obs_len, env.state_words, len(env._retailers)
    es = {torch.float64: 8, torch.float32: 4, torch.bfloat16: 2}[env.obs_dtype]
    aes = 4 if env.action_dtype == torch.float32 else 8
    cols = m if env.MULTI else 1
    plain = 8 * S + 4 * R + m * aes + cols * 8 + m * O * es
    ret, acc, prof = 2 * cols * 8, 2 * (4 + m) * 8, m * 8
    return {"c": plain, "b": plain + ret + acc, "b_ret": plain + ret,
            "a": plain + prof + (prof + m * 2 * es + cols * 8 + acc) + (2 * cols * 8 + cols * 8),
            "a_ret": plain + 2 * cols * 8 + cols * 8}[arm]


def run(name, kind, preset, N, io, rounds, reps):
    dev = torch.device("cuda:0")
    env = ENV_CLASSES[kind](dict(preset(), num_envs=N, **IO[io]))
    lib, h = env._lib, env._handle
    _lib.check(lib.imx_prepare(h, _lib.PREPARE_EVAL))
    m, T, O, R = env.num_nodes, env.num_periods, env.obs_len, len(env._retailers)
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    demand = torch.poisson(torch.full((N, R, T), 5.0, device=dev), generator=g).to(torch.int32)
    if kind == "MAIM_div":
        actions = (torch.randn((T, N, m), dtype=torch.float64, device=dev, generator=g) * 0.5 - 0.6).clamp(-1, 1)
    else:
        actions = torch.rand((T, N, m), dtype=torch.float64, device=dev, generator=g) * 2 - 1
    actions = actions.to(env.action_dtype).contiguous()
    f64 = dict(dtype=torch.float64, device=dev)
    cols = (N, m) if env.MULTI else (N,)
    obs = torch.empty((N, m, O), dtype=env.obs_dtype, device=dev)
    rew = torch.empty(cols, **f64)
    profit = torch.empty((N, m), **f64)
    bufs = {a: {"ret": torch.empty(cols, **f64), "acc": torch.empty((N, 4 + m), **f64)} for a in ARMS}
    info = _lib.ImxInfoOut(None, None, None, None, profit.data_ptr())
    p = lambda x: C.c_void_p(x.data_ptr()) if x is not None else None   # noqa: E731

    def arm(which):
        b = bufs[which]

        def fn(stream):
            s = C.c_void_p(stream)
            _lib.check(lib.imx_reset(h, p(demand), None, 0, 1, None, s))
            if which in ("a", "a_ret"):
                b["ret"].zero_()
            for t in range(T):
                if which in ("b", "b_ret"):
                    _lib.check(lib.imx_step_eval(h, p(actions[t]), p(obs), p(rew), None, p(b["ret"]),
                                                 p(b["acc"]) if which == "b" else None, s))
                    continue
                _lib.check(lib.imx_step(h, p(actions[t]), p(obs), p(rew), C.byref(info) if which == "a" else None, s))
                if which == "a":
                    _lib.check(lib.imx_eval_accumulate(h, p(obs), p(rew), p(profit), p(b["acc"]), int(t == 0), s))
                if which != "c":
                    b["ret"].add_(rew)
        return fn
    graphs = {}
    variants = {}
    for a in ARMS:
        graphs[a] = capture(arm(a))
        variants[a] = lib.imx_kernel_variant(h)
    torch.cuda.synchronize()
    same = torch.equal(bufs["a"]["ret"], bufs["b"]["ret"]) and torch.equal(bufs["a"]["acc"], bufs["b"]["acc"]) and \
        torch.equal(bufs["a_ret"]["ret"], bufs["b_ret"]["ret"]) and torch.equal(bufs["a"]["ret"], bufs["a_ret"]["ret"])
    times = {a: [] for a in ARMS}
    for _ in range(rounds):                                    # alternate the arms round by round
        for a, gr in graphs.items():
            times[a].append(time_ms(gr, reps))
    rec = {"workload": name, "envs": N, "io": io, "periods": T, "identical_outputs": bool(same), "kernel_variant": variants,
           "rounds": rounds, "reps_per_round": reps}
    for a in ARMS:
        us = statistics.median(times[a]) * 1e3
        B = bytes_per_env_step(env, a)
        rec[a] = {"us_per_episode": us, "us_per_period": us / T, "spread_us": [min(times[a]) * 1e3, max(times[a]) * 1e3],
                  "bytes_per_env_step": B, "algorithmic_GB_per_s": B * N * T / (us * 1e-6) / 1e9}
    rec["b_le_a"] = rec["b"]["us_per_episode"] <= rec["a"]["us_per_episode"]
    rec["b_ret_le_a_ret"] = rec["b_ret"]["us_per_episode"] <= rec["a_ret"]["us_per_episode"]
    rec["bookkeeping_us_per_period"] = (rec["b"]["us_per_episode"] - rec["c"]["us_per_episode"]) / T
    del graphs
    torch.cuda.synchronize()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--only", default="")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("this benchmark needs a CUDA device")
    info = card()
    lines = []
    for name, kind, preset, N in WORKLOADS:
        if args.only and args.only not in name:
            continue
        for io in IO:
            rec = run(name, kind, preset, N, io, args.rounds, args.reps)
            rec.update(info)
            line = json.dumps(rec)
            print(line, flush=True)
            lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
