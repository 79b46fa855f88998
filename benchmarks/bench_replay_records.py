#!/usr/bin/env python
"""Per-period records of a stored-plan episode: what they cost on each route, alternating in one process, every arm captured
as one CUDA graph per episode.

Arms (each with and without observations):
  (a) "composition"   today's route to the records: imx_reset, then per period imx_step with imx_info_out pointing into row t
                      and a device-to-device copy of inv / backlog / order_u into row t + 1 (T ahead-of-time step launches);
  (b) "records"       imx_replay_episode_records with every field, on a handle with the default dispatch rule (the episode
                      kernel serves every workload here);
  (b') "records_composed" the same call on a handle with IMX_EPISODE_FUSE=0, which sends it to the library's own composition
                      (reset, T steps with the diagnostics, cudaMemcpyAsync state copies): the other side of the dispatch rule;
  (c) "no_records"    imx_replay_episode without records (what recording costs on top).
All arms also write returns and statistics.  The records of (a), (b) and (b') and the returns / statistics of every arm are
compared before anything is timed.  Workloads: config 2 (serial 4-stage) at 65 536 and 1 Mi envs; config 4 div1 / div2 at
262 144 and 32 768 envs (one 8-GPU shard).  Bytes: records add 36 B per agent-step (12 state, 16 diagnostics, 8 profit) plus
12 B per agent for row 0; "records_GB_per_s" is those bytes over the arm's time, set against an HBM copy peak measured in the
same run (a 2 GiB device-to-device copy, read + write bytes).  One JSON line per (workload, observations), with the card's
name and power limit.

    python benchmarks/bench_replay_records.py [--rounds 7] [--reps 10] [--only div2] [--out results/r3_replay_records.jsonl]
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
REC_NAMES = ("inv", "backlog", "order_u", "demand", "ship", "acquisition", "order_r", "profit")


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


def copy_peak_GB_per_s(reps=20):
    src = torch.empty(1 << 31, dtype=torch.uint8, device="cuda:0")
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    del src, dst
    return 2 * (1 << 31) / (ms * 1e-3) / 1e9


def record_buffers(T, N, m, dev):
    i32 = dict(dtype=torch.int32, device=dev)
    r = {k: torch.empty((T + 1, N, m), **i32) for k in ("inv", "backlog", "order_u")}
    r.update({k: torch.empty((T, N, m), **i32) for k in ("demand", "ship", "acquisition", "order_r")})
    r["profit"] = torch.empty((T, N, m), dtype=torch.float64, device=dev)
    return r


def records_struct(r):
    return _lib.ImxRecordsOut(r["inv"].data_ptr(), r["backlog"].data_ptr(), r["order_u"].data_ptr(), r["demand"].data_ptr(),
                              r["ship"].data_ptr(), r["acquisition"].data_ptr(), r["order_r"].data_ptr(), r["profit"].data_ptr())


def make_env(kind, preset, N, composed):
    old = os.environ.pop("IMX_EPISODE_FUSE", None)
    if composed:
        os.environ["IMX_EPISODE_FUSE"] = "0"
    try:
        env = ENV_CLASSES[kind](dict(preset(), num_envs=N))
    finally:
        os.environ.pop("IMX_EPISODE_FUSE", None)
        if old is not None:
            os.environ["IMX_EPISODE_FUSE"] = old
    _lib.check(env._lib.imx_prepare(env._handle, _lib.PREPARE_EPISODE | _lib.PREPARE_RECORDS))
    return env


def run(name, kind, preset, N, rounds, reps, peak):
    dev = torch.device("cuda:0")
    div = kind.endswith("_div")
    envs = {"default": make_env(kind, preset, N, False), "composed": make_env(kind, preset, N, True)}
    env = envs["default"]
    lib = env._lib
    m, T, O, R = env.num_nodes, env.num_periods, env.obs_len, len(env._retailers)
    cells = N * m
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    demand = torch.poisson(torch.full((N, R, T), 5.0, device=dev), generator=g).to(torch.int32)
    if div:
        actions = (torch.randn((T, N, m), dtype=torch.float64, device=dev, generator=g) * 0.5 - 0.6).clamp(-1, 1)
    else:
        actions = torch.rand((T, N, m), dtype=torch.float64, device=dev, generator=g) * 2 - 1
    f64 = dict(dtype=torch.float64, device=dev)
    p = lambda x: C.c_void_p(x.data_ptr()) if x is not None else None   # noqa: E731
    rec_bytes = 36 * cells * T + 12 * cells
    out = []
    for with_obs in (True, False):
        obs = torch.empty((T, N, m, O), dtype=env.obs_dtype, device=dev) if with_obs else None
        arms = ["composition", "records", "records_composed", "no_records"]
        bufs = {a: {"rew": torch.empty((T, N, m), **f64), "ret": torch.empty((N, m), **f64), "stats": torch.zeros(3 + 2 * m, **f64),
                    "rec": record_buffers(T, N, m, dev) if a != "no_records" else None} for a in arms}
        views = {k: env._state_view(f) for k, f in (("inv", _lib.F_INV), ("backlog", _lib.F_BACKLOG), ("order_u", _lib.F_ORDER_U))}

        def composition(stream, b=bufs["composition"]):
            s, h, r = C.c_void_p(stream), env._handle, b["rec"]
            _lib.check(lib.imx_reset(h, p(demand), None, 0, 1, None, s))
            for k, v in views.items():
                r[k][0].copy_(v.reshape(N, m))
            for t in range(T):
                info = _lib.ImxInfoOut(r["demand"][t].data_ptr(), r["ship"][t].data_ptr(), r["acquisition"][t].data_ptr(),
                                       r["order_r"][t].data_ptr(), r["profit"][t].data_ptr())
                _lib.check(lib.imx_step(h, p(actions[t]), p(obs[t]) if obs is not None else None, p(b["rew"][t]), C.byref(info), s))
                for k, v in views.items():
                    r[k][t + 1].copy_(v.reshape(N, m))
            _lib.check(lib.imx_episode_stats(h, p(b["rew"]), T, p(b["ret"]), p(b["stats"]), 0, s))

        def episode(e, b, with_rec):
            def fn(stream):
                st = records_struct(b["rec"]) if with_rec else None
                _lib.check(e._lib.imx_replay_episode_records(e._handle, p(demand), None, 0, 1, p(actions), p(obs), None, p(b["ret"]),
                                                             p(b["stats"]), 0, None, C.byref(st) if st is not None else None,
                                                             C.c_void_p(stream)))
            return fn
        fns = {"composition": composition, "records": episode(env, bufs["records"], True), "no_records": episode(env, bufs["no_records"], False)}
        fns["records_composed"] = episode(envs["composed"], bufs["records_composed"], True)
        graphs, variants = {}, {}
        for a in arms:
            e = envs["composed"] if a == "records_composed" else env
            graphs[a] = capture(fns[a])
            variants[a] = e._lib.imx_kernel_variant(e._handle)
        same = True
        for a in arms[1:]:
            same &= torch.equal(bufs[a]["ret"], bufs["composition"]["ret"]) and torch.equal(bufs[a]["stats"], bufs["composition"]["stats"])
            if bufs[a]["rec"] is not None:
                same &= all(torch.equal(bufs[a]["rec"][k], bufs["composition"]["rec"][k]) for k in REC_NAMES)
        times = {a: [] for a in arms}
        for _ in range(rounds):                                 # alternate the arms round by round
            for a in arms:
                times[a].append(time_ms(graphs[a], reps))
        row = {"workload": name, "envs": N, "nodes": m, "periods": T, "observations": with_obs, "obs_dtype": str(env.obs_dtype),
               "identical_outputs": bool(same), "kernel_variant": variants, "rounds": rounds, "reps_per_round": reps,
               "records_bytes": rec_bytes, "hbm_copy_peak_GB_per_s": peak}
        for a in arms:
            ms = statistics.median(times[a])
            row[a] = {"us_per_episode": ms * 1e3, "spread_us": [min(times[a]) * 1e3, max(times[a]) * 1e3]}
            if a != "no_records":
                row[a]["records_GB_per_s"] = rec_bytes / (ms * 1e-3) / 1e9
                row[a]["records_share_of_copy_peak"] = row[a]["records_GB_per_s"] / peak
        base = row["no_records"]["us_per_episode"]
        for a in arms:
            if a != "no_records":
                extra = row[a]["us_per_episode"] - base
                row[a]["extra_us_over_no_records"] = extra
                row[a]["records_GB_per_s_on_extra_time"] = rec_bytes / (extra * 1e-6) / 1e9 if extra > 0 else None
        row["speedup_records_vs_composition"] = row["composition"]["us_per_episode"] / row["records"]["us_per_episode"]
        row["speedup_records_vs_records_composed"] = row["records_composed"]["us_per_episode"] / row["records"]["us_per_episode"]
        out.append(row)
        del graphs
        torch.cuda.synchronize()
    del envs, env
    return out


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
    peak = copy_peak_GB_per_s()
    print(json.dumps(dict(info, hbm_copy_peak_GB_per_s=peak)), flush=True)
    lines = []
    for name, kind, preset, N in WORKLOADS:
        if args.only and args.only not in name:
            continue
        for rec in run(name, kind, preset, N, args.rounds, args.reps, peak):
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
