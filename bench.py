#!/usr/bin/env python
"""Benchmark of the environment-step hot path (BASELINE.json config 2).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--envs E] [--dump-outputs DIR]

Workload (per GPU, weak scaling): ``MultiAgentInvManagement`` 4-stage chain in preset MA_6 mode
(hyperparams.py:482-484), 65 536 environments, replayed Poisson(5) demand, host-random uniform
actions pre-staged on the device.  One bench *step* = one 30-period episode of the whole batch
(reset + 30 step() launches, replayed as a CUDA graph) = 65 536 x 4 x 30 agent-steps.

Prints ONE JSON line (rank 0).  Keys beyond the base contract: ``roofline`` (step kernel:
algorithmic bytes / CUDA-event time vs. the measured HBM copy peak), ``roofline_large_n`` (same
kernel at 4 Mi envs, working set >> L2), ``replay_fused`` (the same 30 periods as ONE imx_step_many launch),
``cpu_baseline`` (the oracle port on the host cores; ``cpu_baseline_c``: the plain-C OpenMP restatement),
``e2e`` (same metric through the host-buffer ABI with H2D/D2H inside the timed region; ``e2e_f32_obs``: the same
with float32 observations).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

T_PERIODS = 30
M_STAGES = 4
KERNEL_VARIANTS = {0: "imx::step_kernel (ahead-of-time, direct global accesses)",
                   1: "imx::step_kernel_tma (ahead-of-time, TMA-staged tiles)",
                   2: "imx::step_kernel_tma (NVRTC-specialised, TMA-staged tiles, one tile per CTA)",
                   3: "imx::step_kernel_pipe (NVRTC-specialised, persistent warp-specialised TMA pipeline)"}
ENVS_PER_GPU = 65536
NCU_TRAFFIC_JSON = os.path.join(ROOT, "profiles", "ncu_traffic.json")     # written by benchmarks/ncu_summary.py --traffic-json from the ncu captures
REFERENCE_TIMING_JSON = os.path.join(ROOT, "profiles", "r2_reference_cpu_timing.json")   # benchmarks/time_reference.py (build container)
WORKLOAD = ("MAIM_env 4-stage serial, MA_6 obs mode (td=T,pd=T,pa=F,P=1, shared reward), step() on "
            "65536 envs per GPU, 30-period episodes, replayed Poisson(5) demand, uniform(-1,1) actions pre-staged")


# ----------------------------------------------------------------------------------------
# CPU baseline: the oracle port (oracle/im_oracle.py) on the host cores, one env per worker
# ----------------------------------------------------------------------------------------
def _cpu_worker(args):
    seed, episodes = args
    from marl_for_im_b200 import presets
    from oracle import im_oracle
    cfg = presets.serial4()
    env = im_oracle.OracleEnv("MAIM", cfg)
    rng = np.random.default_rng(seed)
    demand = rng.poisson(5, size=(episodes, T_PERIODS))
    actions = rng.uniform(-1, 1, size=(episodes, T_PERIODS, M_STAGES))
    t0 = time.perf_counter()
    for e in range(episodes):
        env.reset(demand[e])
        for t in range(T_PERIODS):
            env.step(actions[e, t])
    return time.perf_counter() - t0


def ncu_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the kernel `key`, from the committed ncu capture
    (profiles/ncu_traffic.json: {key: {"bytes": ..., "source": profile file, "commit": ...}}); None when not captured."""
    try:
        rec = json.load(open(NCU_TRAFFIC_JSON)).get(key)
        return (int(rec["bytes"]), f"{rec['source']} @ {rec.get('commit', '?')}") if rec else (None, None)
    except (OSError, ValueError, KeyError):
        return None, None


def reference_timing(name):
    """the UNMODIFIED reference timed on the build container (benchmarks/time_reference.py); the GPU box has no reference tree"""
    try:
        doc = json.load(open(REFERENCE_TIMING_JSON))
        row = doc["configs"][name]
        return {"value": row["reference"]["agent_steps_per_sec_all_cores"], "value_1core": row["reference"]["agent_steps_per_sec_1core"],
                "unit": "agent-steps/s", "cores": row["reference"]["cores"], "kind": "reference",
                "port_over_reference_1core_same_machine": row["port_over_reference_1core"],
                "sample": f"{doc['episodes_per_measurement']} episodes x {doc['periods']} periods per core of the same workload through the "
                          f"unmodified environments/*.py, measured on the build container ({doc['machine']['cores_available']} cores, {doc['when']}), "
                          "not on this box: the reference tree cannot travel"}
    except (OSError, ValueError, KeyError):
        return None


def bench_config(world, n_per_gpu):
    """`config` of the JSON line — identical in both arms (workload description only)."""
    return {"workload": WORKLOAD, "envs_per_gpu": n_per_gpu, "periods_per_step": T_PERIODS, "agents": M_STAGES,
            "agent_steps_per_step": world * n_per_gpu * M_STAGES * T_PERIODS}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_baseline(episodes_per_worker=6000, pool=None):
    """agent-steps/s of the oracle port with one process per host core (bounded sample)."""
    import multiprocessing as mp
    cores = host_cores()
    own_pool = pool is None
    if own_pool:
        pool = mp.get_context("fork").Pool(cores)
    try:
        t0 = time.perf_counter()
        pool.map(_cpu_worker, [(1000 + i, episodes_per_worker) for i in range(cores)])
        wall = time.perf_counter() - t0
    finally:
        if own_pool:
            pool.close()
            pool.join()
    agent_steps = cores * episodes_per_worker * T_PERIODS * M_STAGES
    return {"value": agent_steps / wall, "unit": "agent-steps/s", "cores": cores, "kind": "port",
            "sample": f"{cores} processes x {episodes_per_worker} episodes x {T_PERIODS} periods of the same 4-stage "
                      f"MA_6 workload through oracle/im_oracle.py (one env per process, like the reference); {wall:.2f} s wall"}


def cpu_baseline_c():
    """The plain-C restatement (oracle/imx_oracle.c) with all OpenMP threads on the full 65536-env
    episode: the strongest CPU implementation of the same path we can offer, for context."""
    from marl_for_im_b200 import presets
    from oracle import c_oracle
    N, T, m = ENVS_PER_GPU, T_PERIODS, M_STAGES
    demand = np.random.default_rng(420).poisson(5, size=(N, T)).astype(np.int32)
    actions = np.random.default_rng(0).uniform(-1, 1, size=(T, N, m))
    co = c_oracle.COracle("MAIM", presets.serial4())
    co.run(demand[:1024], actions[:, :1024])               # warm-up
    best = None
    for _ in range(3):
        t0 = time.perf_counter()
        co.run(demand, actions)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return {"value": N * T * m / best, "unit": "agent-steps/s", "cores": c_oracle.max_threads(), "kind": "port (plain C, OpenMP)",
            "sample": f"full config-2 episode batch ({N} envs x {T} periods), best of 3, {best * 1e3:.1f} ms"}


def run_reference_arm(args):
    """--impl reference: the reference's CPU design (per-env Python/numpy objects), restated by the
    oracle port because the reference tree cannot travel to the GPU box; all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = host_cores()
    pool = mp.get_context("fork").Pool(cores)
    per_worker = 400                                       # ~0.3 s of wall clock per step on 16 cores
    try:
        for _ in range(max(args.warmup, 1)):
            pool.map(_cpu_worker, [(i, 4) for i in range(cores)])
        t0 = time.perf_counter()
        for s in range(args.steps):
            pool.map(_cpu_worker, [(s * cores + i, per_worker) for i in range(cores)])
        wall = time.perf_counter() - t0
    finally:
        pool.close()
        pool.join()
    agent_steps = args.steps * cores * per_worker * T_PERIODS * M_STAGES
    value = agent_steps / wall
    sample = (f"each step = {cores} processes x {per_worker} episodes x {T_PERIODS} periods (a bounded sample of the "
              f"65536-env batch), oracle/im_oracle.py port of the reference's per-env numpy path")
    line = {
        "impl": "reference", "metric": "agent_steps_per_sec", "value": value, "unit": "agent-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": bench_config(args.gpus, args.envs), "sample": sample,
        "cpu_baseline": {"value": value, "unit": "agent-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "cpu_baseline_reference": reference_timing("config2_maim4_ma6"),
        "e2e": {"value": value, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------
# clocks sampling during the timed region
# ----------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, reasons, smax = [], set(), None
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                smax = float(r[2])
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                continue
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------
def algorithmic_bytes_per_env_step(env):
    """SURVEY.md §8(d): B = 2*4*S + 4*R + 8*m*(2 + O)."""
    S, R, m, O = env.state_words, len(env._retailers), env.num_nodes, env.obs_len
    return 2 * 4 * S + 4 * R + 8 * m * (2 + O)


class RawEpisode:
    """reset + T step launches through the C ABI on preallocated device buffers (graph-capturable)."""

    def __init__(self, env, demand_dev, actions_dev, obs_bufs, rew_bufs, obs0):
        from marl_for_im_b200 import _lib
        self.env, self.lib, self._lib = env, env._lib, _lib
        self.demand, self.actions, self.obs, self.rew, self.obs0 = demand_dev, actions_dev, obs_bufs, rew_bufs, obs0

    def reset(self, stream):
        self._lib.check(self.lib.imx_reset(self.env._handle, C.c_void_p(self.demand.data_ptr()), None, 0, 1,
                                           C.c_void_p(self.obs0.data_ptr()), C.c_void_p(stream)))

    def steps_many(self, stream, periods):
        """the same periods as ONE imx_step_many call on the stored plan; needs the per-period observation / reward
        buffers to be consecutive slices of one tensor"""
        self._lib.check(self.lib.imx_step_many(self.env._handle, C.c_void_p(self.actions.data_ptr()), periods,
                                               C.c_void_p(self.obs[0].data_ptr()), C.c_void_p(self.rew[0].data_ptr()), None, C.c_void_p(stream)))

    def steps(self, stream, periods):
        h = self.env._handle
        for t in range(periods):
            self._lib.check(self.lib.imx_step(h, C.c_void_p(self.actions[t].data_ptr()),
                                              C.c_void_p(self.obs[t % len(self.obs)].data_ptr()),
                                              C.c_void_p(self.rew[t % len(self.rew)].data_ptr()), None, C.c_void_p(stream)))


def capture(fn, torch):
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn(s.cuda_stream)            # warm-up outside capture (module load, attribute setup)
        s.synchronize()
        with torch.cuda.graph(g, stream=s):
            fn(torch.cuda.current_stream().cuda_stream)
    torch.cuda.current_stream().wait_stream(s)
    return g


def timed_replays(graph, reps, torch):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3


# ----------------------------------------------------------------------------------------
# the other BASELINE.json configs, measured at this run's world size (rows g2 of the coverage table)
# ----------------------------------------------------------------------------------------
def _timed_region(fn, reps, torch, dist, world, dev, post=None):
    """barrier + sync, `reps` calls of fn, optional collective, CUDA events; returns the max over ranks in seconds"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    if post is not None:
        post()
    e1.record()
    torch.cuda.synchronize()
    dt = e0.elapsed_time(e1) * 1e-3
    if world > 1:
        tmax = torch.tensor([dt], dtype=torch.float64, device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dt = float(tmax.item())
    return dt


def config4_episode_loop(name, total_envs, world, rank, dev, torch, dist, peak, reps, action_mode="near_eq"):
    """BASELINE config 4: MAIM_div_env (div1 / div2), `total_envs` envs in total split over the ranks (STRONG scaling),
    reset + 30 x imx_step + episode statistics per episode as one CUDA graph, one all-reduce per evaluation batch."""
    from marl_for_im_b200 import _lib, presets
    from marl_for_im_b200.envs import MultiAgentInvManagementDiv
    cfg = presets.PRESETS[name]()
    N = total_envs // world
    env = MultiAgentInvManagementDiv(dict(cfg, num_envs=N, device=str(dev), env_offset=rank * N))
    m, T, O, R = env.num_nodes, env.num_periods, env.obs_len, len(env._retailers)
    g = torch.Generator(device=dev)
    g.manual_seed(1000 + rank)
    demand = torch.poisson(torch.full((N, R, T), 5.0, device=dev), generator=g).to(torch.int32)
    if action_mode == "uniform":
        actions = torch.rand((T, N, m), dtype=torch.float64, device=dev, generator=g) * 2 - 1
    else:                                                   # near-equilibrium: exercises every branch of the split (SURVEY config 4 (ii))
        actions = (torch.randn((T, N, m), dtype=torch.float64, device=dev, generator=g) * 0.5 - 0.6).clamp(-1, 1)
    nbuf = 4 if N * m * O * 8 > (64 << 20) else T          # > L2 either way: T distinct buffers, or 4 x (> 64 MB)
    obs = [torch.empty((N, m, O), dtype=torch.float64, device=dev) for _ in range(nbuf)]
    rew = torch.empty((T, N, m), dtype=torch.float64, device=dev)
    stats = torch.zeros(3 + 2 * m, dtype=torch.float64, device=dev)
    lib, h = env._lib, env._handle

    def steps(stream):
        for t in range(T):
            _lib.check(lib.imx_step(h, C.c_void_p(actions[t].data_ptr()), C.c_void_p(obs[t % nbuf].data_ptr()), C.c_void_p(rew[t].data_ptr()),
                                    None, C.c_void_p(stream)))

    def episode(stream):
        _lib.check(lib.imx_reset(h, C.c_void_p(demand.data_ptr()), None, 0, 1, C.c_void_p(obs[0].data_ptr()), C.c_void_p(stream)))
        steps(stream)
        _lib.check(lib.imx_episode_stats(h, C.c_void_p(rew.data_ptr()), T, None, C.c_void_p(stats.data_ptr()), 1, C.c_void_p(stream)))

    def steps_only(stream):
        lib.imx_set_period(h, 0)
        steps(stream)

    g_ep, g_st = capture(episode, torch), capture(steps_only, torch)
    variant = lib.imx_kernel_variant(h)
    for _ in range(3):
        g_ep.replay()
    stats.zero_()
    dt = _timed_region(g_ep.replay, reps, torch, dist, world, dev, post=(lambda: dist.all_reduce(stats)) if world > 1 else None)
    timed_replays(g_st, 3, torch)
    dts = timed_replays(g_st, max(reps, 10), torch) / (max(reps, 10) * T)
    # the same episode with the 30 periods as ONE imx_step_many launch (the pre-staged actions are a stored plan): no per-period
    # launch floor, which is what bounds the strong-scaling curve of the per-step loop at 32 768 envs per GPU
    fused = None
    if True:
        obs_all = torch.empty((T, N, m, O), dtype=torch.float64, device=dev)    # (at most 2.3 GB: div2, 262 144 envs)

        def episode_many(stream):
            _lib.check(lib.imx_reset(h, C.c_void_p(demand.data_ptr()), None, 0, 1, None, C.c_void_p(stream)))
            _lib.check(lib.imx_step_many(h, C.c_void_p(actions.data_ptr()), T, C.c_void_p(obs_all.data_ptr()), C.c_void_p(rew.data_ptr()), None,
                                         C.c_void_p(stream)))
            _lib.check(lib.imx_episode_stats(h, C.c_void_p(rew.data_ptr()), T, None, C.c_void_p(stats.data_ptr()), 1, C.c_void_p(stream)))

        g_many = capture(episode_many, torch)
        for _ in range(3):
            g_many.replay()
        keep = stats.clone()
        dtm = _timed_region(g_many.replay, reps, torch, dist, world, dev)
        stats.copy_(keep)
        fused = {"agent_steps_per_sec": world * N * m * T * reps / dtm, "ms_per_episode": dtm / reps * 1e3,
                 "api": "imx_reset + imx_step_many(K=30) + imx_episode_stats per episode (one CUDA graph)"}
        del obs_all
    B = algorithmic_bytes_per_env_step(env)
    flags = int(env.error_flags.abs().sum())
    out = {"workload": f"MAIM_div_env {name}, MA_6 obs mode, {total_envs} envs in total over {world} GPU(s) = {N} per GPU (strong scaling), "
                       f"Poisson(5) demand [N,{R},30], clip(N(-0.6,0.5),-1,1) actions pre-staged, reset + 30 imx_step + statistics per episode",
           "scaling": "strong", "envs_total": total_envs, "envs_per_gpu": N, "agent_steps_per_sec": world * N * m * T * reps / dt,
           "ms_per_episode": dt / reps * 1e3,
           "step_kernel": {"us_per_launch": dts * 1e6, "achieved": B * N / dts / 1e9, "peak": peak, "unit": "GB/s", "frac": B * N / dts / 1e9 / peak,
                           "algorithmic_bytes_per_env_step": B, "kernel": KERNEL_VARIANTS[variant],
                           "traffic": ncu_traffic(f"step_kernel_{name}_{N}")[0], "traffic_source": ncu_traffic(f"step_kernel_{name}_{N}")[1]},
           "replay_fused": fused,
           "watchdog_flags": flags, "mean_return": float((stats[1] / stats[0]).item()) if float(stats[0].item()) > 0 else None,
           "cpu_baseline_reference": reference_timing("config4_" + name)}
    del env
    return out


def config3_fused_rollout(total_envs, world, rank, dev, torch, dist, reps):
    """BASELINE config 3: MAIM_env 8-stage, `total_envs` envs over the ranks, fused 30-period base-stock rollout (z = 25),
    Philox Poisson(5) demand drawn in the kernel, per-batch return statistics + one all-reduce."""
    from marl_for_im_b200 import _lib, presets
    from marl_for_im_b200.envs import MultiAgentInvManagement
    cfg = presets.serial8(time_dependency=False, prev_demand=False)
    cfg["standardise_actions"] = False
    cfg.update(demand_dist="poisson", mu=5)
    N = total_envs // world
    env = MultiAgentInvManagement(dict(cfg, num_envs=N, device=str(dev), env_offset=rank * N))
    m, T = env.num_nodes, env.num_periods
    z = torch.full((m,), 25.0, dtype=torch.float64, device=dev)
    ret = torch.empty((N, m), dtype=torch.float64, device=dev)
    stats = torch.zeros(3 + 2 * m, dtype=torch.float64, device=dev)
    lib, h = env._lib, env._handle
    s = torch.cuda.current_stream().cuda_stream
    ep = [0]

    def batch():
        ep[0] += 1                                          # a new episode id = new Philox draws
        _lib.check(lib.imx_rollout_basestock(h, C.c_void_p(z.data_ptr()), 0, None, None, 0, ep[0], None, C.c_void_p(ret.data_ptr()), None, None, 0,
                                             C.c_void_p(s)))
        # statistics of the batch added into `stats` on the device (imx_episode_stats over ONE row of returns, accumulate = 1)
        _lib.check(lib.imx_episode_stats(h, C.c_void_p(ret.data_ptr()), 1, None, C.c_void_p(stats.data_ptr()), 1, C.c_void_p(s)))

    for _ in range(3):
        batch()
    stats.zero_()
    dt = _timed_region(batch, reps, torch, dist, world, dev, post=(lambda: dist.all_reduce(stats)) if world > 1 else None)
    out = {"workload": f"MAIM_env 8-stage serial (MA_inv_management.py:40-61), {total_envs} envs in total over {world} GPU(s) = {N} per GPU, fused "
                       "30-period base-stock rollout (z = 25), Philox Poisson(5) demand in-kernel, return statistics + 1 all-reduce per batch",
           "scaling": "strong", "envs_total": total_envs, "envs_per_gpu": N, "agent_steps_per_sec": world * N * m * T * reps / dt,
           "ms_per_batch": dt / reps * 1e3, "bound": "instruction issue (about 1 byte of HBM traffic per agent-step)",
           "kernel": "imx::rollout_kernel (NVRTC-specialised)" if lib.imx_kernel_variant(h) >= 2 else "imx::rollout_kernel (ahead-of-time)",
           "mean_return": float((stats[1] / stats[0]).item()), "cpu_baseline_reference": reference_timing("maim8_ma6")}
    del env
    return out


def config5_env_plus_observer(n_per_gpu, world, rank, dev, torch, dist, peak, reps):
    """BASELINE config 5, the part of it that is this path: 2-stage MAIM_env in CC_5 obs mode + the centralised-critic
    observation (central_critic_observer + FillInActions, models/CC_Model.py:165-214) emitted by the step itself
    (imx_step_cc: one kernel writes obs, reward, state and the [N][m][W] critic rows).  float32 observations (RLlib's cast).
    The policy / value networks of config 5 are RLlib's and out of scope (SURVEY section 2)."""
    from marl_for_im_b200 import _lib, presets
    from marl_for_im_b200.envs import MultiAgentInvManagement
    N = n_per_gpu
    env = MultiAgentInvManagement(dict(presets.serial2(), num_envs=N, device=str(dev), env_offset=rank * N, obs_dtype="float32"))
    m, T, O = env.num_nodes, env.num_periods, env.obs_len
    W = (m - 1) * (1 + O) + O
    g = torch.Generator(device=dev)
    g.manual_seed(2000 + rank)
    demand = torch.poisson(torch.full((N, 1, T), 5.0, device=dev), generator=g).to(torch.int32)
    actions = torch.rand((T, N, m), dtype=torch.float64, device=dev, generator=g) * 2 - 1
    obs = torch.empty((T, N, m, O), dtype=torch.float32, device=dev)
    cc = torch.empty((T, N, m, W), dtype=torch.float32, device=dev)
    rew = torch.empty((T, N, m), dtype=torch.float64, device=dev)
    lib, h = env._lib, env._handle
    fused = hasattr(lib, "imx_step_cc")

    def steps_only(stream):
        lib.imx_set_period(h, 0)
        for t in range(T):
            if fused:
                _lib.check(lib.imx_step_cc(h, C.c_void_p(actions[t].data_ptr()), C.c_void_p(obs[t].data_ptr()), C.c_void_p(cc[t].data_ptr()), 1,
                                           -1.0, 1.0, C.c_void_p(rew[t].data_ptr()), C.c_void_p(stream)))
            else:
                _lib.check(lib.imx_step(h, C.c_void_p(actions[t].data_ptr()), C.c_void_p(obs[t].data_ptr()), C.c_void_p(rew[t].data_ptr()), None,
                                        C.c_void_p(stream)))
                _lib.check(lib.imx_cc_observe(h, C.c_void_p(obs[t].data_ptr()), C.c_void_p(actions[t].data_ptr()), -1.0, 1.0,
                                              C.c_void_p(cc[t].data_ptr()), 1, C.c_void_p(stream)))

    s = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.imx_reset(h, C.c_void_p(demand.data_ptr()), None, 0, 1, None, C.c_void_p(s)))
    gs = capture(steps_only, torch)
    for _ in range(3):
        gs.replay()
    dt = _timed_region(gs.replay, reps, torch, dist, world, dev)
    per_step = dt / (reps * T)
    S_words = env.state_words
    B = 2 * 4 * S_words + 4 + 8 * m * 2 + 4 * m * O + 4 * m * W        # state r+w, demand, actions + rewards (f64), obs + critic rows (f32)
    out = {"workload": f"MAIM_env 2-stage (Oracle_2.py:26-37), CC_5 obs mode (O = {O}), {N} envs per GPU, step + centralised-critic observation "
                       f"rows [N][{m}][{W}] float32 (models/CC_Model.py:165-214) per period",
           "scaling": "weak", "envs_per_gpu": N, "samples_per_sec": world * N * m / per_step, "us_per_period": per_step * 1e6,
           "fused_in_step_kernel": bool(fused), "algorithmic_bytes_per_env_step": B, "achieved": B * N / per_step / 1e9, "peak": peak, "unit": "GB/s",
           "frac": B * N / per_step / 1e9 / peak, "cpu_baseline_reference": reference_timing("config5_maim2_cc5"),
           "note": "samples = agent-steps of env + critic-observation build; the policy / value MLPs of config 5 are RLlib's (out of scope)"}
    del env
    return out


def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    cpu = cpu_c = cpu_1 = None
    if world == 1 and not args.skip_cpu:
        cpu = cpu_baseline()                       # before CUDA is initialised (fork-safe)
        t1 = _cpu_worker((999, 400))               # the same port on ONE core (BASELINE.md section 4a)
        cpu_1 = {"value": 400 * T_PERIODS * M_STAGES / t1, "unit": "agent-steps/s", "cores": 1, "kind": "port",
                 "sample": f"400 episodes x {T_PERIODS} periods in this process; {t1:.2f} s"}
        try:
            cpu_c = cpu_baseline_c()
        except Exception as exc:
            cpu_c = {"error": str(exc)[:200]}

    import torch
    import torch.distributed as dist
    from marl_for_im_b200 import _lib as _lib_mod
    from marl_for_im_b200 import presets
    from marl_for_im_b200.envs import MultiAgentInvManagement

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    from marl_for_im_b200.dist import bind_host_to_gpu      # host buffers of the e2e leg next to this rank's GPU
    numa_cores = bind_host_to_gpu(local_rank)                # (2 GPUs: 0.99 -> 1.37 G agent-steps/s end to end)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"

    N, T, m = args.envs, T_PERIODS, M_STAGES
    cfg = presets.serial4()
    env = MultiAgentInvManagement(dict(cfg, num_envs=N, device=str(dev), env_offset=rank * N))
    O = env.obs_len
    rng = np.random.default_rng(420 + rank)
    demand_h = rng.poisson(5, size=(N, 1, T)).astype(np.int32)
    actions_h = np.random.default_rng(rank).uniform(-1, 1, size=(T, N, m))
    demand = torch.as_tensor(demand_h, device=dev)
    actions = torch.as_tensor(actions_h, device=dev)
    obs_all = torch.empty((T, N, m, O), dtype=torch.float64, device=dev)                  # one buffer per period (trajectory storage)
    obs = [obs_all[t] for t in range(T)]
    rew = torch.empty((T, N, m), dtype=torch.float64, device=dev)
    obs0 = torch.empty((N, m, O), dtype=torch.float64, device=dev)
    ep = RawEpisode(env, demand, actions, obs, [rew[t] for t in range(T)], obs0)

    # Episode statistics [n, sum, sum of squares, per-agent ...] accumulate on the device; like the reference's
    # evaluation loops (np.mean / np.std over all test episodes, MA_inv_management.py:591-595) they are
    # reduced ONCE per evaluation batch = the K timed episodes: a single NCCL all-reduce of 3 + 2m doubles.
    stats_acc = torch.zeros(3 + 2 * m, dtype=torch.float64, device=dev)

    def episode(stream):
        ep.reset(stream)
        ep.steps(stream, T)                                  # 30 step() launches: the per-step API an RL loop calls
        _lib_mod.check(env._lib.imx_episode_stats(env._handle, C.c_void_p(rew.data_ptr()), T, None, C.c_void_p(stats_acc.data_ptr()),
                                                  1, C.c_void_p(stream)))

    launches0 = env.launch_count()
    episode(torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    launches_per_episode = env.launch_count() - launches0
    g_episode = capture(episode, torch)

    def steps_only(stream):
        env._lib.imx_set_period(env._handle, 0)
        ep.steps(stream, T)

    g_steps = capture(steps_only, torch)
    step_variant = env._lib.imx_kernel_variant(env._handle)      # which kernel the per-step launches use (before imx_step_many changes it)

    def steps_only_many(stream):
        env._lib.imx_set_period(env._handle, 0)
        ep.steps_many(stream, T)

    g_steps_many = capture(steps_only_many, torch)
    def bench_step():
        g_episode.replay()                                   # reset + 30 step launches + episode statistics, one graph

    def reduce_batch():
        if world > 1:
            dist.all_reduce(stats_acc)                       # the single collective of the data path
        return stats_acc

    for _ in range(max(args.warmup, 3)):
        bench_step()
    reduce_batch()                                           # also initialises the NCCL communicator outside the timed region
    stats_acc.zero_()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                                      # before the barrier: spawning nvidia-smi must not skew the ranks
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(args.steps):
        bench_step()
    final_stats = reduce_batch()                             # inside the timed region
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    elapsed = e0.elapsed_time(e1) * 1e-3
    # device copies of the last timed episode's outputs, taken before the replays below overwrite the buffers; they reach
    # the host only after the clocks have been sampled
    dumped = sample_outputs(obs0, obs_all, rew, final_stats) if args.dump_outputs and rank == 0 else None
    if os.environ.get("IMX_BENCH_DEBUG"):
        print(f"[rank {rank}] elapsed {elapsed * 1e3:.3f} ms for {args.steps} steps", file=sys.stderr, flush=True)
    # keep the GPU busy a little longer so that the 100 ms clock sampler sees the kernel under load
    t_end = time.perf_counter() + 0.6
    while rank == 0 and time.perf_counter() < t_end:
        g_steps.replay()
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        tmax = torch.tensor([elapsed], dtype=torch.float64, device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        elapsed = float(tmax.item())
    agent_steps_per_bench_step = world * N * m * T
    value = agent_steps_per_bench_step * args.steps / elapsed

    # ---- roofline of the step kernel (live, CUDA events, steps-only graph: 30 dependent launches) ----
    B = algorithmic_bytes_per_env_step(env)
    reps = max(10, args.steps)
    timed_replays(g_steps, 3, torch)
    dt = timed_replays(g_steps, reps, torch) / (reps * T)
    achieved = B * N / dt / 1e9
    # the same 30 periods as ONE imx_step_many launch (stored action plan; the tiles' state stays in shared memory):
    # state moves once per launch instead of once per period, so its algorithmic bytes per env-step are lower
    timed_replays(g_steps_many, 3, torch)
    dt_many = timed_replays(g_steps_many, reps, torch) / reps
    S_words, R_rows = env.state_words, len(env._retailers)
    B_many = 4 * R_rows + 8 * m * (2 + O) + 2 * 4 * S_words / T
    replay_fused = {"agent_steps_per_sec": world * N * m * T / dt_many, "ms_per_30_periods": dt_many * 1e3,
                    "algorithmic_bytes_per_env_step": B_many, "achieved": B_many * N * T / dt_many / 1e9, "peak": peak, "unit": "GB/s",
                    "frac": B_many * N * T / dt_many / 1e9 / peak,
                    "api": "imx_step_many(K=30): one launch per episode, state resident in shared memory, inputs prefetched two periods "
                           "ahead, outputs streamed behind the compute; bit-identical to 30 imx_step calls (tests/test_gpu_step_many.py)"}
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "frac_of_nominal_8000_GBs": achieved / 8000.0,
                "traffic": ncu_traffic("step_kernel_config2_65536")[0] if N == ENVS_PER_GPU else None,
                "traffic_source": (ncu_traffic("step_kernel_config2_65536")[1] or "not captured for this kernel revision")
                                  + " (ncu --set full: dram__bytes_read+write per launch, cold L2; the 31 MB working set of one launch is "
                                    "L2-resident in the bench loop, hence traffic << algorithmic bytes)",
                "kernel": KERNEL_VARIANTS[step_variant], "us_per_launch": dt * 1e6,
                "algorithmic_bytes_per_env_step": B, "envs_per_launch": N, "peak_source": peak_src,
                "note": "per-launch time = steps-only graph of 30 dependent launches / 30 (includes inter-kernel gaps)"}

    state_mb = env.state_words * 4 * N / 1e6
    # ---- same kernel at large N (working set >> L2), rank 0 only -------------------------------------
    roof_large = None
    if rank == 0 and not args.skip_large:
        try:
            roof_large = large_n_roofline(torch, dev, peak)
        except Exception as exc:                             # never lose the headline line to the side measurement
            roof_large = {"error": str(exc)[:200]}

    # ---- end-to-end through the host-buffer ABI (H2D + kernel + D2H + sync per step) ----------------
    e2e = e2e_measure(env, demand_h, actions_h, torch, dev, world, episodes=max(2, min(args.steps, 5)))
    e2e["mode"] = "zero-copy: the step kernel addresses the pinned host buffers directly (default)"
    # the same call with staged copies (cudaMemcpyAsync H2D, kernel, cudaMemcpyAsync D2H on one stream): the copy engine moves
    # the payload a little faster than SM stores over PCIe but adds two copy launches per step; both are measured at every
    # world size and the headline is the better one (the library default is zero-copy; IMX_HOST_ZERO_COPY=0 selects staged)
    os.environ["IMX_HOST_ZERO_COPY"] = "0"
    try:
        env_st = MultiAgentInvManagement(dict(presets.serial4(), num_envs=N, device=str(dev), env_offset=rank * N))
        e2e_staged = e2e_measure(env_st, demand_h, actions_h, torch, dev, world, episodes=max(2, min(args.steps, 5)))
        e2e_staged["mode"] = "staged: cudaMemcpyAsync in, kernel, cudaMemcpyAsync out (IMX_HOST_ZERO_COPY=0)"
        del env_st
    except Exception as exc:
        e2e_staged = {"error": str(exc)[:200]}
    finally:
        os.environ.pop("IMX_HOST_ZERO_COPY", None)
    e2e_modes = {"zero_copy": dict(e2e), "staged_copy_engine": e2e_staged}
    if e2e_staged.get("value", 0.0) > e2e["value"]:
        e2e = dict(e2e_staged)
    # same call with float32 observations (the cast RLlib's preprocessor applies to every observation anyway):
    # 40 % fewer bytes over PCIe; reported beside the float64 drop-in number, never instead of it
    env32 = MultiAgentInvManagement(dict(presets.serial4(), num_envs=N, device=str(dev), env_offset=rank * N, obs_dtype="float32"))
    e2e_f32 = e2e_measure(env32, demand_h, actions_h, torch, dev, world, episodes=max(2, min(args.steps, 5)))
    e2e_f32["api"] += "; obs_f32 = 1"
    del env32

    # ---- the other BASELINE configs at this world size (every rank takes part; rank 0 reports) --------------------------
    other = {}
    if not args.skip_configs:
        del obs_all, obs, rew, ep
        torch.cuda.empty_cache()
        creps = max(5, min(args.steps, 20))
        for key, fn in (("config3_maim8_fused_rollout_1Mi", lambda: config3_fused_rollout(1 << 20, world, rank, dev, torch, dist, creps)),
                        ("config4_div1_262144", lambda: config4_episode_loop("div1", 262144, world, rank, dev, torch, dist, peak, creps)),
                        ("config4_div2_262144", lambda: config4_episode_loop("div2", 262144, world, rank, dev, torch, dist, peak, creps)),
                        ("config5_maim2_cc_observer", lambda: config5_env_plus_observer(ENVS_PER_GPU, world, rank, dev, torch, dist, peak, creps))):
            try:
                other[key] = fn()
            except Exception as exc:                         # a side measurement must never cost the headline line
                other[key] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
            torch.cuda.empty_cache()

    if rank == 0:
        line = {
            "metric": "agent_steps_per_sec", "value": value, "unit": "agent-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": elapsed / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i32 state / f64 obs+reward",
            "data": "synthetic",
            "config": bench_config(world, N),
            "measurement": {"l2": (f"inputs larger than L2: each step streams {T} distinct action/obs/reward buffers "
                                   f"({(T * N * m * (2 + O) * 8) / 1e6:.0f} MB > 126 MB L2); the {state_mb:.1f} MB state stays cached by design"),
                            "timing": "CUDA events around K CUDA-graph replays (reset + 30 step launches) + per-episode return statistics"
                                      + (" + 1 NCCL all-reduce of the batch statistics" if world > 1 else "") + ", max over ranks"},
            "configs": other, "cpu_baseline_reference": reference_timing("config2_maim4_ma6"),
            "roofline": roofline, "roofline_large_n": roof_large, "replay_fused": replay_fused, "cpu_baseline": cpu, "cpu_baseline_1core": cpu_1, "cpu_baseline_c": cpu_c, "e2e": e2e, "e2e_modes": e2e_modes, "e2e_f32_obs": e2e_f32,
            "gpu_launches": int(launches_per_episode * args.steps), "host_cores_bound_to_gpu_numa_node": numa_cores,
            "clocks": clocks,
            "episode_stats": {"n": float(final_stats[0].item()), "mean_return": float((final_stats[1] / final_stats[0]).item())},
        }
        print(json.dumps(line), flush=True)
    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()


DUMP_ENVS = 4096
DUMP_LIMIT_BYTES = 64 << 20


def sample_outputs(obs0, obs_all, rew, stats):
    """Device copies of what the last timed episode returned to its caller: the reset observations, the 30 periods'
    observations and rewards, and the episode statistics accumulated over the timed steps.  Per-env arrays keep a fixed,
    seeded sample of DUMP_ENVS envs (all of them when there are fewer), the same in every run, so that two builds can be
    compared output for output."""
    import torch
    N = obs0.shape[0]
    keep = np.sort(np.random.default_rng(0).choice(N, size=min(N, DUMP_ENVS), replace=False))
    idx = torch.as_tensor(keep, device=obs0.device)
    return {"obs_reset": obs0.index_select(0, idx), "obs": obs_all.index_select(1, idx), "reward": rew.index_select(1, idx),
            "episode_stats": stats.clone()}


def write_outputs(out_dir, sampled):
    """sample_outputs' arrays as float64 DIR/<name>.npy files."""
    arrays = {k: v.double().cpu().numpy() for k, v in sampled.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs would write {total} bytes (limit {DUMP_LIMIT_BYTES})")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def large_n_roofline(torch, dev, peak, N=4 * 1024 * 1024, periods=8):
    from marl_for_im_b200 import presets
    from marl_for_im_b200.envs import MultiAgentInvManagement
    m, T = M_STAGES, T_PERIODS
    env = MultiAgentInvManagement(dict(presets.serial4(), num_envs=N, device=str(dev)))
    O = env.obs_len
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    demand = torch.randint(0, 11, (N, 1, T), dtype=torch.int32, device=dev, generator=g)
    actions = torch.rand((periods, N, m), dtype=torch.float64, device=dev, generator=g) * 2 - 1
    obs = [torch.empty((N, m, O), dtype=torch.float64, device=dev) for _ in range(2)]
    rew = [torch.empty((N, m), dtype=torch.float64, device=dev) for _ in range(2)]
    obs0 = obs[0]
    ep = RawEpisode(env, demand, actions, obs, rew, obs0)
    s = torch.cuda.current_stream().cuda_stream
    ep.reset(s)
    ep.steps(s, periods)                                   # warm-up
    torch.cuda.synchronize()
    env._lib.imx_set_period(env._handle, 0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ep.steps(s, periods)
    e1.record()
    torch.cuda.synchronize()
    dt = e0.elapsed_time(e1) * 1e-3 / periods
    B = algorithmic_bytes_per_env_step(env)
    achieved = B * N / dt / 1e9
    variant = env._lib.imx_kernel_variant(env._handle)
    del env
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "envs_per_launch": N, "us_per_launch": dt * 1e6, "working_set_mb": B * N / 1e6,
            "agent_steps_per_sec": N * m / dt, "algorithmic_bytes_per_launch": B * N,
            "traffic": ncu_traffic("step_kernel_config2_4Mi")[0] if N == 4 * 1024 * 1024 else None,
            "traffic_source": ncu_traffic("step_kernel_config2_4Mi")[1] or "not captured for this kernel revision",
            "kernel": KERNEL_VARIANTS[variant]}


def e2e_measure(env, demand_h, actions_h, torch, dev, world, episodes):
    """Host buffers in, host buffers out, every step: imx_reset_host + 30 x imx_step_host."""
    import torch.distributed as dist
    from marl_for_im_b200 import _lib
    N, m, T, O = env.num_envs, env.num_nodes, T_PERIODS, env.obs_len
    pin = lambda a: torch.as_tensor(a).pin_memory()   # noqa: E731
    dem_p, act_p = pin(demand_h), pin(actions_h)
    obs_bytes = 4 if env.obs_dtype == torch.float32 else 8
    obs_p = torch.empty((N, m, O), dtype=env.obs_dtype).pin_memory()
    rew_p = torch.empty((N, m), dtype=torch.float64).pin_memory()
    lib, h = env._lib, env._handle

    def one_episode():
        _lib.check(lib.imx_reset_host(h, C.c_void_p(dem_p.data_ptr()), None, 0, 7, C.c_void_p(obs_p.data_ptr())))
        for t in range(T):
            _lib.check(lib.imx_step_host(h, C.c_void_p(act_p[t].data_ptr()), C.c_void_p(obs_p.data_ptr()), C.c_void_p(rew_p.data_ptr())))
        return float(rew_p[0, 0])                      # device→host read of the step's result

    one_episode()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(episodes):
        one_episode()
    wall = time.perf_counter() - t0
    if world > 1:
        tmax = torch.tensor([wall], dtype=torch.float64, device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        wall = float(tmax.item())
    h2d = T * N * m * 8 + N * T * 4
    d2h = T * (N * m * O * obs_bytes + N * m * 8) + N * m * O * obs_bytes
    return {"value": world * N * m * T * episodes / wall, "unit": "agent-steps/s",
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "episodes_timed": episodes,
            "api": "imx_reset_host + 30 x imx_step_host on pinned host buffers (wall clock, each call synchronises)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU, help="environments per GPU")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-large", action="store_true")
    ap.add_argument("--skip-configs", action="store_true", help="skip BASELINE configs 3 / 4 / 5 (the `configs` object of the line)")
    ap.add_argument("--large-only", action="store_true", help="only the 4 Mi-env roofline point (used for the ncu capture)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last timed episode's observations, "
                    "rewards and episode statistics (a fixed sample of envs, float64) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.large_only or args.impl == "reference"):
        ap.error("--dump-outputs writes the outputs of the timed GPU path; it does not apply to --large-only or --impl reference")
    if args.large_only:
        import torch
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
        print(json.dumps(large_n_roofline(torch, torch.device("cuda:0"), peak)), flush=True)
    elif args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
