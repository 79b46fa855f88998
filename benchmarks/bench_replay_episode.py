#!/usr/bin/env python
"""imx_replay_episode (one launch per stored-plan episode) against the composition it replaces (imx_reset + imx_step_many +
imx_episode_stats), alternating in one process, each path captured as one CUDA graph per episode.

Workloads: config 2 (serial 4-stage, 65 536 envs and 1 Mi envs), config 4 div1 / div2 at 262 144 envs and at one 8-GPU shard
(32 768 envs).  Output sets: "scoring" = returns + statistics only (scoring a batch of plans); "replay" = observations +
rewards + statistics (bench.py's config-4 replay_fused episode).  Both paths replay the same inputs back to back (a working set
that fits in L2 stays there for both).  One JSON line per (workload, output set), with the card's name and power limit.

    python benchmarks/bench_replay_episode.py [--rounds 7] [--reps 20] [--out results/r3_replay_episode.jsonl]
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

WORKLOADS = [("config2_serial4", "MAIM", presets.serial4, 65536), ("config4_div1", "MAIM_div", presets.div1, 262144),
             ("config4_div2", "MAIM_div", presets.div2, 262144), ("config4_div1_shard8", "MAIM_div", presets.div1, 32768),
             ("config4_div2_shard8", "MAIM_div", presets.div2, 32768), ("config2_serial4_1Mi", "MAIM", presets.serial4, 1 << 20)]


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


def algorithmic_bytes(env, outputs):
    """Bytes each path must move per episode, from shapes: inputs read once, outputs written once, plus what only the
    composition has — the state written by reset and loaded back by step_many, the [N][R][T] trace transposed into
    [T][R][N] and read again, and the step rewards written and read back by the statistics."""
    N, m, T, O, R, S = env.num_envs, env.num_nodes, env.num_periods, env.obs_len, len(env._retailers), env.state_words
    cols = m if env.MULTI else 1
    es = 4 if env.obs_dtype == torch.float32 else 8
    rewards, returns = T * N * cols * 8, N * cols * 8
    common = T * N * m * 8 + N * R * T * 4 + S * 4 * N                        # actions, trace, final state
    if outputs == "replay":
        common += T * N * m * O * es + rewards                                # observations, rewards
        comp = common + rewards                                               # the statistics read the rewards back
        new = common + 2 * returns                                            # returns (scratch) written, read by the statistics
    else:
        comp = common + 2 * rewards + returns                                 # rewards written and read back, returns written
        new = common + 2 * returns                                            # returns written, read by the statistics
    comp += 2 * S * 4 * N + 2 * N * R * T * 4                                 # state written by reset and loaded; trace transposed
    return {"composition": comp, "replay_episode": new}


def run(name, kind, preset, N, rounds, reps):
    dev = torch.device("cuda:0")
    env = ENV_CLASSES[kind](dict(preset(), num_envs=N))
    lib, h = env._lib, env._handle
    _lib.check(lib.imx_prepare(h, _lib.PREPARE_EPISODE))
    m, T, O, R = env.num_nodes, env.num_periods, env.obs_len, len(env._retailers)
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    demand = torch.poisson(torch.full((N, R, T), 5.0, device=dev), generator=g).to(torch.int32)
    if kind == "MAIM_div":
        actions = (torch.randn((T, N, m), dtype=torch.float64, device=dev, generator=g) * 0.5 - 0.6).clamp(-1, 1)
    else:
        actions = torch.rand((T, N, m), dtype=torch.float64, device=dev, generator=g) * 2 - 1
    f64 = dict(dtype=torch.float64, device=dev)
    rew = torch.empty((T, N, m), **f64)
    obs = torch.empty((T, N, m, O), **f64)
    out = []
    for outputs in ("scoring", "replay"):
        rp = outputs == "replay"
        bufs = {}
        for path in ("composition", "replay_episode"):
            bufs[path] = {"ret": torch.empty((N, m), **f64), "stats": torch.zeros(3 + 2 * m, **f64)}
        p = lambda x: C.c_void_p(x.data_ptr()) if x is not None else None   # noqa: E731

        def composition(stream, b=bufs["composition"]):
            s = C.c_void_p(stream)
            _lib.check(lib.imx_reset(h, p(demand), None, 0, 1, None, s))
            _lib.check(lib.imx_step_many(h, p(actions), T, p(obs) if rp else None, p(rew), None, s))
            _lib.check(lib.imx_episode_stats(h, p(rew), T, None if rp else p(b["ret"]), p(b["stats"]), 0, s))

        def replay_episode(stream, b=bufs["replay_episode"]):
            _lib.check(lib.imx_replay_episode(h, p(demand), None, 0, 1, p(actions), p(obs) if rp else None, p(rew) if rp else None,
                                              None if rp else p(b["ret"]), p(b["stats"]), 0, None, C.c_void_p(stream)))
        graphs = {"composition": capture(composition), "replay_episode": capture(replay_episode)}
        variant = lib.imx_kernel_variant(h)
        # same outputs (statistics always; returns for the scoring set)
        same = torch.equal(bufs["composition"]["stats"], bufs["replay_episode"]["stats"]) and \
            (rp or torch.equal(bufs["composition"]["ret"], bufs["replay_episode"]["ret"]))
        times = {"composition": [], "replay_episode": []}
        for _ in range(rounds):                                 # alternate the two paths round by round
            for path, gr in graphs.items():
                times[path].append(time_ms(gr, reps))
        B = algorithmic_bytes(env, outputs)
        rec = {"workload": name, "envs": N, "outputs": outputs, "periods": T, "identical_outputs": bool(same),
               "replay_episode_kernel_variant": variant, "rounds": rounds, "reps_per_round": reps}
        for path in graphs:
            ms = statistics.median(times[path])
            rec[path] = {"ms_per_episode": ms, "spread_ms": [min(times[path]), max(times[path])],
                         "agent_steps_per_sec": N * m * T / (ms * 1e-3), "algorithmic_bytes": B[path],
                         "algorithmic_GB_per_s": B[path] / (ms * 1e-3) / 1e9}
        rec["speedup"] = rec["composition"]["ms_per_episode"] / rec["replay_episode"]["ms_per_episode"]
        out.append(rec)
        del graphs
        torch.cuda.synchronize()
    del env
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--reps", type=int, default=20)
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
        for rec in run(name, kind, preset, N, args.rounds, args.reps):
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
