"""Vector adapters: one GPU batch behind RLlib's vectorised-env plug points.

The reference registers ONE Python env per rollout worker (``tune.register_env(name, lambda cfg: Env(cfg))``,
MA_inv_management.py:34-36,83-84) and RLlib wraps it.  RLlib's own batched plug points are
``ray.rllib.env.VectorEnv`` (``vector_reset / reset_at / vector_step / get_unwrapped``, single-agent) and
``ray.rllib.env.BaseEnv`` (``poll / send_actions / try_reset``, multi-agent) of ray 1.5.2 — ray is pinned in
the reference's ``poetry.lock`` but not vendored and not installable here, so these classes are duck-typed: same
method names, argument meaning and return structure, no ray import.  They add no arithmetic: every step is one
``imx_step`` launch on the whole batch; the adapters only reshape its outputs.

All envs of a batch run in lock-step (episodes are fixed length, MAIM_env.py:395-397), so every env reports
``done`` at the same step; ``reset_at`` / ``try_reset`` reset the whole batch once and then hand out the cached
observations env by env.

The ``*_tensors`` methods are the zero-copy path for a GPU-resident policy: torch tensors in, torch tensors out,
no per-env Python objects.
"""
from __future__ import annotations

import numpy as np
import torch


def _host(t):
    """numpy copy of a device tensor; bfloat16 (which numpy lacks) as its exact float32 widening."""
    t = t.cpu()
    return (t.float() if t.dtype == torch.bfloat16 else t).numpy()


class _LockStepBatch:
    def __init__(self, env):
        if not env.batched:
            raise ValueError("vector adapters wrap a batched env (construct it with num_envs=N)")
        self.env = env
        self.num_envs = env.num_envs
        self.observation_space = env.observation_space
        self.action_space = env.action_space
        self._reset_pending = False       # the batch finished an episode and has not been reset yet
        self._obs_host = None

    def _batch_reset(self):
        self.env.reset()
        obs = self.env.last_obs           # the packed [N, m, O] tensor the per-agent views point into
        self._obs_dev = obs
        self._obs_host = _host(obs)
        self._reset_pending = False
        return obs

    def get_unwrapped(self):
        """VectorEnv.get_unwrapped: the underlying envs — here ONE batched env stands for all of them."""
        return [self.env]

    def stop(self):
        self.env.close()


class BatchedVectorEnv(_LockStepBatch):
    """``VectorEnv`` surface for the single-agent kinds (InvManagement, InvManagementDiv)."""

    def __init__(self, env):
        super().__init__(env)
        if env.MULTI:
            raise ValueError("BatchedVectorEnv wraps a single-agent env; use BatchedMultiAgentEnv")

    # ---- list surface (what RLlib's sampler calls) ----
    def vector_reset(self):
        self._batch_reset()
        return [self._obs_host[n] for n in range(self.num_envs)]

    def reset_at(self, index):
        if self._reset_pending or self._obs_host is None:
            self._batch_reset()
        return self._obs_host[int(index)]

    def vector_step(self, actions):
        obs, rew, done = self.step_tensors(torch.as_tensor(np.asarray(actions, dtype=np.float64), device=self.env.device))
        o, r = _host(obs), rew.cpu().numpy()
        N = self.num_envs
        return [o[n] for n in range(N)], [np.float64(r[n]) for n in range(N)], [done] * N, [{} for _ in range(N)]

    # ---- tensor surface ----
    def reset_tensors(self):
        return self._batch_reset()

    def step_tensors(self, actions):
        """actions [N, m] → (obs [N, m, O], reward [N], done)."""
        obs, rew, done, _ = self.env.step(actions)
        self._reset_pending = bool(done)
        return obs, rew, bool(done)


class BatchedMultiAgentEnv(_LockStepBatch):
    """``BaseEnv`` surface (``poll`` / ``send_actions`` / ``try_reset``) for the multi-agent kinds: dicts keyed by
    env id, then by agent id (``stage_i`` / ``node_i``), as RLlib's multi-agent sampler consumes them."""

    def __init__(self, env):
        super().__init__(env)
        if not env.MULTI:
            raise ValueError("BatchedMultiAgentEnv wraps a multi-agent env; use BatchedVectorEnv")
        self._agents = list(env.agent_names)
        self._pending = None              # (obs [N,m,O], reward [N,m] or None, done) waiting to be polled
        self._batch_reset()
        self._pending = (self._obs_dev, None, False)

    # ---- dict surface ----
    def poll(self):
        """→ (obs, rewards, dones, infos, off_policy_actions), each ``{env_id: {agent_id: value}}``; rewards are
        empty right after a reset (BaseEnv convention: a fresh observation carries no reward)."""
        if self._pending is None:
            return {}, {}, {}, {}, {}
        obs_d, rew_d, done = self._pending
        self._pending = None
        o = _host(obs_d)
        r = rew_d.cpu().numpy() if rew_d is not None else None
        obs, rewards, dones, infos = {}, {}, {}, {}
        for n in range(self.num_envs):
            obs[n] = {a: o[n, i] for i, a in enumerate(self._agents)}
            rewards[n] = {a: np.float64(r[n, i]) for i, a in enumerate(self._agents)} if r is not None else {}
            dones[n] = {"__all__": done}
            infos[n] = {}
        return obs, rewards, dones, infos, {}

    def send_actions(self, action_dict):
        """action_dict ``{env_id: {agent_id: action}}`` for every env of the batch."""
        N, m = self.num_envs, len(self._agents)
        if len(action_dict) != N:
            raise ValueError(f"a lock-step batch needs actions for all {N} envs (got {len(action_dict)})")
        act = np.empty((N, m), dtype=np.float64)
        for n in range(N):
            row = action_dict[n]
            for i, a in enumerate(self._agents):
                act[n, i] = np.asarray(row[a], dtype=np.float64).reshape(-1)[0]
        self.send_action_tensor(torch.as_tensor(act, device=self.env.device))

    def try_reset(self, env_id):
        """→ ``{agent_id: obs}`` of env ``env_id`` after the (single, batch-wide) reset."""
        if self._reset_pending:
            self._batch_reset()
            self._pending = None          # observations are handed out through try_reset, not poll
        return {a: self._obs_host[int(env_id), i] for i, a in enumerate(self._agents)}

    # ---- tensor surface ----
    def reset_tensors(self):
        self._pending = None
        return self._batch_reset()

    def send_action_tensor(self, actions):
        _, _, done, _ = self.env.step(actions)
        done = bool(done["__all__"])
        self._reset_pending = done
        self._pending = (self.env.last_obs, self.env.last_reward, done)

    def poll_tensors(self):
        """→ (obs [N, m, O], reward [N, m] or None after a reset, done) on the device."""
        p, self._pending = self._pending, None
        return p
