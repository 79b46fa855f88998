#!/usr/bin/env python
"""A GPU-resident rollout loop at kernel rate: policy forward + env.step() captured ONCE as a CUDA graph and replayed per
episode, so no Python runs between the launches (a plain Python loop is host-bound: 9.5 us per step() call against a 6 us
kernel, see benchmarks/bench_python_loop.py).

The "policy" here is a stand-in (a per-agent linear map of the observation squashed to [-1, 1]); swap in any module
whose forward is graph-capturable.  The returns are added up by the step launch itself (env.step_eval).  Prints one JSON
line.  Measured on a B200 (1000 W power limit, 1965 MHz max SM clock) at 65 536 envs: 20.1 us per period, of which the env
step with the returns measured 6.5 us with float64 observations (profiles/r3_step_eval.jsonl) — the four small torch kernels of the stand-in policy are the rest.

    python examples/rl_loop_cuda_graph.py [--envs 65536] [--episodes 20]
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from marl_for_im_b200 import _lib, presets  # noqa: E402
from marl_for_im_b200.envs import MultiAgentInvManagement  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--episodes", type=int, default=20)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    N = args.envs
    env = MultiAgentInvManagement(dict(presets.serial4(), num_envs=N, reuse_buffers=True, obs_dtype="float32"))
    m, O, T = env.num_nodes, env.obs_len, env.num_periods
    torch.manual_seed(0)
    w = torch.randn((m, O), device=dev) * 0.3                       # one weight vector per agent
    actions = torch.empty((N, m), dtype=torch.float64, device=dev)   # the graph's action buffer
    returns = torch.zeros((N, m), dtype=torch.float64, device=dev)   # step_eval restarts it at period 0
    _lib.check(env._lib.imx_prepare(env._handle, _lib.PREPARE_EVAL))  # its kernels are loaded before the capture

    env.reset()
    obs = env.last_obs                                               # the reused [N, m, O] float32 output buffer

    def period():
        actions.copy_(torch.tanh(torch.einsum("nmo,mo->nm", obs, w)))   # policy forward -> actions (float32 -> float64 buffer)
        env.step_eval(actions, returns=returns, want_rewards=False)  # one launch: the reused obs buffer + the returns

    # warm up on a side stream (module loads, allocator), then capture.  An imx_step launch carries its period index
    # (it selects the demand row), so the periods are captured in order, all T of them in one graph.
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        period()
        period()
    torch.cuda.current_stream().wait_stream(s)
    env.reset()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):                                        # the whole episode: T x (policy, step with return accumulation)
        for t in range(T):
            period()

    def episode_exact():
        env.reset()                                                  # fresh Philox demand drawn on the device
        g.replay()
        env._lib.imx_set_period(env._handle, T)                      # host-side period counter (a replay does not advance it)

    episode_exact()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.episodes):
        episode_exact()
    e1.record()
    torch.cuda.synchronize()
    dt = e0.elapsed_time(e1) * 1e-3 / args.episodes
    print(json.dumps({"case": "T x (policy forward + env.step_eval with the returns) captured as one CUDA graph, float32 observations",
                      "envs": N, "ms_per_episode": dt * 1e3, "us_per_period": dt / T * 1e6,
                      "agent_steps_per_sec": N * m * T / dt, "mean_return": float(returns.sum(-1).mean().item())}))


if __name__ == "__main__":
    main()
