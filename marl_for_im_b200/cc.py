"""Centralised-critic observation function — drop-in for ``central_critic_observer`` and the
opponent-action fill of ``FillInActions`` (models/CC_Model.py:165-214), batched on the GPU.

RLlib flattens the dict observation ``{"own_obs", "opponent_obs", "opponent_action"}`` in sorted key
order, so the model sees ``[opponent_action | opponent_obs | own_obs]``
(``CentralizedCriticModel`` reads ``input[..., -obs_size:]`` as own_obs, CC_Model.py:127).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib


def cc_observe(env, obs, actions=None, clip=(-1.0, 1.0), dtype=torch.float64):
    """obs: [N, m, O] tensor (or the env's dict of [N, O] views / [O] numpy arrays); actions: [N, m]
    tensor, dict, or None (zeros — what the observer emits at sampling time).  Returns the flat
    centralised-critic observation [N, m, W] on the device, W = (m-1)*(1+O) + O."""
    N, m, O = env.num_envs, env.num_nodes, env.obs_len
    if isinstance(obs, dict):
        vals = [obs[n] for n in env.agent_names]
        if isinstance(vals[0], torch.Tensor):
            obs = torch.stack([v.reshape(N, O) for v in vals], dim=1)
        else:
            obs = torch.as_tensor(np.stack([np.asarray(v).reshape(N, O) for v in vals], axis=1), device=env.device)
    obs = obs.to(device=env.device, dtype=env.obs_dtype).reshape(N, m, O).contiguous()   # the element type this env writes
    act = None
    if actions is not None:
        act = env._actions_to_device(actions)
    W = env._lib.imx_cc_obs_len(env._handle)
    out_type = {torch.float64: 0, torch.float32: 1, torch.bfloat16: 2}.get(dtype)    # imx_cc_observe's out_is_f32 codes
    if out_type is None:
        raise ValueError("dtype must be float64, float32 or bfloat16")
    out = torch.empty((N, m, W), dtype=dtype, device=env.device)
    _lib.check(env._lib.imx_cc_observe(env._handle, C.c_void_p(obs.data_ptr()), C.c_void_p(act.data_ptr()) if act is not None else None,
                                       float(clip[0]), float(clip[1]), C.c_void_p(out.data_ptr()), out_type, env._stream()))
    return out


def central_critic_observer(agent_obs, env=None, **kw):
    """Same signature and result as the reference function: dict of per-agent observations in, dict
    of ``{"own_obs", "opponent_obs", "opponent_action"}`` out (opponent actions zero).  Needs the env
    (``env=``) whose observations these are; batched envs get [N, ...] tensors, drop-in envs numpy."""
    if env is None:
        raise TypeError("central_critic_observer(agent_obs, env=<the env>) — the batched observer runs on the env's device")
    m, O = env.num_nodes, env.obs_len
    flat = cc_observe(env, agent_obs)
    out = {}
    for i, name in enumerate(env.agent_names):
        row = flat[:, i, :]
        entry = {"own_obs": row[:, (m - 1) * (1 + O):], "opponent_obs": row[:, m - 1:(m - 1) * (1 + O)], "opponent_action": row[:, :m - 1]}
        if not env.batched:
            entry = {k: v[0].cpu().numpy() for k, v in entry.items()}
        out[name] = entry
    return out
