"""Batched, GPU-resident drop-ins for the four reference environments.

    InvManagement               environments/IM_env.py        (gym.Env surface)
    MultiAgentInvManagement     environments/MAIM_env.py      (RLlib MultiAgentEnv dict surface)
    InvManagementDiv            environments/IM_div_env.py
    MultiAgentInvManagementDiv  environments/MAIM_div_env.py

Same constructor keys, same ``reset(customer_demand=None, noisy_delay=False,
noisy_delay_threshold=0)`` and ``step(action) -> (obs, reward, done, info)``, same attributes
(``inv_max, order_max, demand_max, retailers, period, inv[period, :], ...``).  Two modes:

* **drop-in mode** (no ``num_envs`` key): one environment, numpy in / numpy out, full
  ``info`` dicts and ``[T+1, m]`` float64 history arrays exactly like the reference, demand drawn
  with the reference's own host generator (scipy on the global ``np.random`` stream);
* **batched mode** (``num_envs=N``): N environments advance per call, every array gains a leading
  N axis and lives on the GPU as a torch tensor (float64 obs/rewards, int32 state), demand comes
  from a replayed tensor or the on-device Philox stream.

All arithmetic happens in the sm_100a kernels behind the C ABI (include/imx_b200.h); this module
only parses configs, owns buffers and shapes the results.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _lib
from .spaces import Box
from .topology import check_connections, create_network, get_retailers, get_stage

_I32 = np.int32


class _DevView:
    """Zero-copy torch view of library-owned device memory (via __cuda_array_interface__)."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2, "strides": None}


def _int_vec(x, n, name):
    arr = np.asarray(x, dtype=np.float64).reshape(-1)
    if arr.size != n:
        raise ValueError(f"{name}: expected {n} entries, got {arr.size}")
    if not np.all(arr == np.rint(arr)):
        raise ValueError(f"{name} must hold integral values (state is int32 on the device)")
    return arr.astype(np.int64)


class _History:
    """Batched-mode stand-in for the reference's ``[T+1, m]`` arrays: ``env.inv[env.period, :]``
    (the access pattern of base_restock_policy.py:12) returns the live ``[N, m]`` state tensor."""

    def __init__(self, env, field):
        self._env, self._field = env, field

    def __getitem__(self, idx):
        t = idx[0] if isinstance(idx, tuple) else idx
        if int(t) != self._env.period:
            raise IndexError("batched envs keep only the current period's state "
                             f"(asked for period {int(t)}, current is {self._env.period})")
        v = self._env._state_view(self._field)
        return v[(slice(None),) + tuple(idx[1:])] if isinstance(idx, tuple) and len(idx) > 1 else v


class _ImxEnvBase:
    KIND = ""
    DIV = False
    MULTI = False
    AGENT_PREFIX = "stage_"

    # ------------------------------------------------------------------ construction
    def __init__(self, config):
        self.config = config.copy()
        take = config.get if self.DIV else config.pop        # quirk 11: the serial ctors empty the caller's dict
        self.num_periods = take("num_periods", 50)
        self._parse_structure(config, take)
        m = self.num_nodes
        self.standardise_state = True if self.KIND == "MAIM_div" else take("standardise_state", True)
        self.standardise_actions = True if self.KIND == "MAIM_div" else take("standardise_actions", True)
        if self.KIND == "IM_div":
            self.a, self.b = -1, 1                           # IM_div_env.py:35-36
        else:
            self.a, self.b = take("a", -1), take("b", 1)
        self.time_dependency = take("time_dependency", False)
        self.prev_actions = take("prev_actions", False)
        self.prev_demand = take("prev_demand", False)
        self.prev_length = take("prev_length", 1)
        self.max_delay = int(np.max(self.delay))
        if self.max_delay == 0:
            self.time_dependency = False
        self.stock_cost = np.asarray(take("stock_cost", np.ones(m) * 0.5), dtype=np.float64)
        self.backlog_cost = np.asarray(take("backlog_cost", np.ones(m)), dtype=np.float64)
        self.demand_dist = take("demand_dist", "custom")
        self.SEED = take("seed", 52)
        self.noisy_demand = bool(take("noisy_demand", False)) if self.DIV else False
        self.noisy_demand_threshold = take("noisy_demand_threshold", 0) if self.DIV else 0
        self.noisy_delay = bool(take("noisy_delay", False)) if self.DIV else False
        self.noisy_delay_threshold = take("noisy_delay_threshold", 0) if self.DIV else 0
        self._parse_capacities(config, take)

        # batching / device (extensions; absent keys = drop-in mode)
        n_envs = take("num_envs", None)
        self.batched = n_envs is not None
        self.num_envs = int(n_envs) if self.batched else 1
        self.device = torch.device(take("device", "cuda:0"))
        if self.device.type != "cuda":
            raise _lib.ImxError("marl_for_im_b200 envs run on CUDA devices only (no CPU fallback)")
        self.env_offset = int(take("env_offset", 0))
        self.return_info = bool(take("return_info", not self.batched))
        self.reuse_buffers = bool(take("reuse_buffers", False))
        self.demand_mode = take("demand_mode", "philox" if self.batched else "host")
        obs_dtype = take("obs_dtype", "float64")             # "float32": the cast RLlib applies anyway, half the bytes
        self.obs_dtype = {"float64": torch.float64, "float32": torch.float32, "bfloat16": torch.bfloat16, torch.float64: torch.float64,
                          torch.float32: torch.float32, torch.bfloat16: torch.bfloat16}[obs_dtype]
        # float32 actions: what a reduced-precision policy's output layer emits; results equal float64 actions of the same values
        self.action_dtype = {"float64": torch.float64, "float32": torch.float32, torch.float64: torch.float64,
                             torch.float32: torch.float32}[take("action_dtype", "float64")]
        if not self.batched and (self.obs_dtype == torch.bfloat16 or self.action_dtype == torch.float32):
            raise ValueError("obs_dtype='bfloat16' and action_dtype='float32' are batched-mode options (construct the env with "
                             "num_envs=N): the drop-in env mirrors the reference's float64 numpy surface")
        self.mu = self.config.get("mu", 5)
        if self.demand_dist == "poisson":                    # callers pre-draw test sets with env.dist.rvs (inv_management.py:200)
            from scipy.stats import poisson
            self.dist, self.dist_param = poisson, {"mu": self.mu}
        elif self.demand_dist == "uniform":
            from scipy.stats import randint
            lo_up = self.config.get("lower_upper", (1, 5))
            self.dist, self.dist_param = randint, {"low": lo_up[0], "high": lo_up[1]}
        if not self.batched:
            np.random.seed(seed=int(self.SEED))              # MAIM_env.py:50 — drop-in mode keeps the global-stream semantics

        assert isinstance(self.num_periods, int)             # MAIM_env.py:158
        self.done = set()
        self.state = {} if self.MULTI else None
        self._episode = 0
        self._handle = None
        if take("_config_only", False):                      # build tooling: parse + derive the imx_config, no device work
            self.imx_config = self._build_config(self.noisy_delay)
            return
        self._create_handle(self.noisy_delay)
        self._build_spaces()
        self.reset()

    def _parse_structure(self, config, take):
        raise NotImplementedError

    def _parse_capacities(self, config, take):
        raise NotImplementedError

    # ------------------------------------------------------------------ native handle
    def _build_config(self, with_carry: bool):
        """The C ABI's imx_config for this env (pure host code: no device needed)."""
        m = self.num_nodes
        c = _lib.ImxConfig()
        c.kind = _lib.KIND[self.KIND]
        c.num_nodes, c.num_periods = m, int(self.num_periods)
        c.prev_length = int(self.prev_length)
        c.time_dependency, c.prev_demand, c.prev_actions = int(bool(self.time_dependency)), int(bool(self.prev_demand)), int(bool(self.prev_actions))
        c.standardise_state, c.standardise_actions = int(bool(self.standardise_state)), int(bool(self.standardise_actions))
        c.independent = int(bool(getattr(self, "independent", True)))
        c.share_network = int(bool(getattr(self, "share_network", False)))
        c.noisy_delay = int(bool(with_carry))
        dist = self.demand_dist if self.demand_dist in ("poisson", "uniform") else "replay"
        c.demand_dist = _lib.DIST[dist]
        lower_upper = self.config.get("lower_upper", (1, 5))
        c.uniform_low, c.uniform_high = int(lower_upper[0]), int(lower_upper[1])
        c.device = self.device.index if self.device.index is not None else (torch.cuda.current_device() if torch.cuda.is_available() else 0)
        c.obs_f32 = int(self.obs_dtype == torch.float32)
        c.io_flags = (_lib.IO_OBS_BF16 if self.obs_dtype == torch.bfloat16 else 0) | \
                     (_lib.IO_ACTIONS_F32 if self.action_dtype == torch.float32 else 0)
        c.a, c.b = float(self.a), float(self.b)
        c.mu = float(self.config.get("mu", 5))
        c.noisy_delay_threshold = float(self.noisy_delay_threshold)
        c.noisy_demand_threshold = float(self.noisy_demand_threshold) if (self.DIV and self.noisy_demand) else 0.0
        c.seed = int(self.SEED) & 0xFFFFFFFFFFFFFFFF
        c.num_envs, c.env_offset = self.num_envs, self.env_offset
        inv_init = _int_vec(self.inv_init, m, "init_inv")
        inv_max = _int_vec(self.inv_max, m, "inv_max")
        order_max = _int_vec(self.order_max, m, "order_max")
        delay = _int_vec(self.delay, m, "delay")
        for i in range(m):
            c.inv_init[i], c.inv_max[i], c.order_max[i], c.delay[i] = int(inv_init[i]), int(inv_max[i]), int(order_max[i]), int(delay[i])
            c.inv_target[i] = float(np.asarray(self.inv_target, dtype=np.float64)[i])
            c.stock_cost[i], c.backlog_cost[i] = float(self.stock_cost[i]), float(self.backlog_cost[i])
        if self.DIV:
            for p in range(m):
                ch = list(self.connections.get(p, []) or [])
                if len(ch) > _lib.MAX_CHILDREN:
                    raise ValueError(f"node {p} has {len(ch)} children; at most {_lib.MAX_CHILDREN} are supported")
                c.num_children[p] = len(ch)
                for k, v in enumerate(ch):
                    c.children[p][k] = int(v)
        else:
            price = np.asarray(self.price, dtype=np.float64).reshape(-1)
            for i in range(m + 1):
                c.price[i] = float(price[i])
        return c

    def _create_handle(self, with_carry: bool):
        lib = _lib.load()
        if not torch.cuda.is_available():
            raise _lib.ImxError("no CUDA device — marl_for_im_b200 has no CPU fallback")
        m = self.num_nodes
        c = self._build_config(with_carry)
        if self._handle is not None:
            lib.imx_destroy(self._handle)
            self._handle = None
        h = C.c_void_p()
        _lib.check(lib.imx_create(C.byref(c), C.byref(h)))
        self._handle, self._lib, self._has_carry = h, lib, bool(with_carry)
        self._mail = None                                    # the drop-in mailbox holds pointers into the old handle's state
        self._handle_threshold = float(self.noisy_delay_threshold)
        self._dev_index = c.device
        self.obs_len = lib.imx_obs_len(h)
        self.state_words = lib.imx_state_words(h)
        nret = lib.imx_num_retailers(h)
        buf = (C.c_int32 * max(nret, 1))()
        lib.imx_retailers(h, buf)
        self._retailers = [int(buf[k]) for k in range(nret)]
        dm = (C.c_int32 * m)()
        lib.imx_demand_max(h, dm)
        self._demand_max_lib = np.array([dm[i] for i in range(m)], dtype=np.int64)
        self._views = {}

    def __del__(self):
        try:
            if getattr(self, "_handle", None) is not None:
                self._lib.imx_destroy(self._handle)
                self._handle = None
        except Exception:
            pass

    def close(self):
        self.__del__()

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _state_view(self, field, dtype_str="<i4"):
        if field in self._views:
            return self._views[field]
        ptr, cnt = C.c_void_p(), C.c_int64()
        _lib.check(self._lib.imx_state_field(self._handle, field, C.byref(ptr), C.byref(cnt)))
        if cnt.value == 0:
            return None
        N, m = self.num_envs, self.num_nodes
        shape = {_lib.F_INV: (N, m), _lib.F_BACKLOG: (N, m), _lib.F_ORDER_U: (N, m), _lib.F_CARRY: (N, m),
                 _lib.F_ERROR: (N,)}.get(field, None)
        if shape is None:
            if field == _lib.F_DEMAND:
                shape = (self.num_periods, len(self._retailers), N)
            else:
                shape = (N, cnt.value // N)
        v = torch.as_tensor(_DevView(ptr.value, shape, dtype_str), device=self.device)
        self._views[field] = v
        return v

    def launch_count(self):
        return int(self._lib.imx_launch_count())

    # ------------------------------------------------------------------ helpers with the reference's names
    def rescale(self, val, min_val, max_val, A=-1, B=1):
        """MAIM_env.py:497-507."""
        return A + (((val - min_val) * (B - A)) / (max_val - min_val))

    def rev_scale(self, val_scaled, min_val, max_val, A=-1, B=1):
        """MAIM_env.py:509-519."""
        return (((val_scaled - A) * (max_val - min_val)) / (B - A)) + min_val

    @property
    def agent_names(self):
        return self._agent_names

    @property
    def period(self):
        return self._lib.imx_period(self._handle)

    @property
    def error_flags(self):
        """[N] int32: 0 = ok, 1..4 = the reference's 'Infinite Loop k' watchdog of the divergent split."""
        return self._state_view(_lib.F_ERROR)

    def state_dict(self):
        """Integer state as torch tensors (views): inv, backlog, order_u [N, m]; pipe [N, L]; ..."""
        names = {"inv": _lib.F_INV, "backlog": _lib.F_BACKLOG, "order_u": _lib.F_ORDER_U, "pipe": _lib.F_PIPE,
                 "hist_d": _lib.F_HIST_D, "hist_o": _lib.F_HIST_O, "carry": _lib.F_CARRY, "backlog_to": _lib.F_BACKLOG_TO}
        out = {}
        for k, f in names.items():
            v = self._state_view(f)
            if v is not None:
                out[k] = v
        return out

    # ------------------------------------------------------------------ demand handling
    def _draw_host_demand(self):
        """Reference-identical host draw (MAIM_env.py:199-219 / MAIM_div_env.py:263-295)."""
        from scipy.stats import poisson, randint
        cfg_take = self.config.get if self.DIV else self.config.pop       # quirk 4 (serial kinds pop their parameters)
        T = self.num_periods
        size = (len(self._retailers), T) if self.DIV else T
        if self.demand_dist == "custom":
            default = np.ones((len(self._retailers), T), dtype=np.int16) * 5 if self.DIV else np.ones(T, dtype=np.int16) * 5
            demand = cfg_take("customer_demand", default)
        elif self.demand_dist == "poisson":
            self.mu = cfg_take("mu", 5)
            self.dist, self.dist_param = poisson, {"mu": self.mu}
            demand = self.dist.rvs(size=size, **self.dist_param)
        elif self.demand_dist == "uniform":
            lower, upper = cfg_take("lower_upper", (1, 5))
            self.dist, self.dist_param = randint, {"low": lower, "high": upper}
            if lower >= upper:
                raise Exception("Lower bound cannot be larger than upper bound")
            demand = self.dist.rvs(size=size, **self.dist_param)
        else:
            raise Exception("Unrecognised, Distribution Not Implemented")
        if self.DIV and self.noisy_demand:                                # MAIM_div_env.py:287-295
            for k in range(len(self._retailers)):
                for j in range(T):
                    double_demand = np.random.uniform(0, 1)
                    zero_demand = np.random.uniform(0, 1)
                    if double_demand <= self.noisy_demand_threshold:
                        demand[k, j] = 2 * demand[k, j]
                    if zero_demand <= self.noisy_demand_threshold:
                        demand[k, j] = 0
        return demand

    def _demand_to_device(self, customer_demand):
        N, R, T = self.num_envs, len(self._retailers), self.num_periods
        if isinstance(customer_demand, torch.Tensor):
            d = customer_demand
            if d.dtype.is_floating_point and not bool((d == d.round()).all()):
                raise ValueError("customer_demand must be integral")
            d = d.to(device=self.device, dtype=torch.int32)
        else:
            arr = np.asarray(customer_demand)
            if arr.dtype.kind == "f" and not np.all(arr == np.rint(arr)):
                raise ValueError("customer_demand must be integral")
            d = torch.as_tensor(np.ascontiguousarray(arr.astype(_I32)), device=self.device)
        if d.numel() == R * T:                                            # one trace: shared by every env
            d = d.reshape(1, R, T).expand(N, R, T)
        return d.reshape(N, R, T).contiguous()

    # ------------------------------------------------------------------ reset / step
    def reset(self, customer_demand=None, noisy_delay=False, noisy_delay_threshold=0, delay_mask=None):
        """reset — IM_env.py:164-229, MAIM_env.py:176-240, IM_div_env.py:201-302, MAIM_div_env.py:240-341.

        ``delay_mask`` (extension): replayed noisy-delay outcomes ``[N, T, m]`` / ``[T, m]`` booleans."""
        if noisy_delay:                                                   # sticky, like the reference (quirk 5)
            self.noisy_delay = noisy_delay
            self.noisy_delay_threshold = noisy_delay_threshold
        want_noisy = bool(self.noisy_delay) or delay_mask is not None
        # the carry state exists only in handles created for noisy delays; a device-generated (Philox)
        # mask uses the threshold the handle was created with
        generated_mask = want_noisy and delay_mask is None and self.batched
        if want_noisy and (not self._has_carry or
                           (generated_mask and self._handle_threshold != float(self.noisy_delay_threshold))):
            self._create_handle(True)
        N, m, T = self.num_envs, self.num_nodes, self.num_periods

        demand_dev = None
        if customer_demand is not None:
            self.customer_demand = customer_demand
            demand_dev = self._demand_to_device(customer_demand)
        elif self.demand_mode == "host" or self.demand_dist == "custom":
            self.customer_demand = self._draw_host_demand()
            demand_dev = self._demand_to_device(self.customer_demand)
        else:
            self.customer_demand = None                                   # drawn on the device; see customer_demand_device()

        mask_dev = None
        if want_noisy:
            if delay_mask is None and not self.batched:
                delay_mask = self._draw_host_delay_mask()
            if delay_mask is not None:
                mask_dev = self._mask_to_device(delay_mask)

        obs_buf = self._new_obs()
        self._episode += 1
        _lib.check(self._lib.imx_reset(
            self._handle,
            C.c_void_p(demand_dev.data_ptr()) if demand_dev is not None else None,
            C.c_void_p(mask_dev.data_ptr()) if mask_dev is not None else None,
            int(want_noisy), self._episode, C.c_void_p(obs_buf.data_ptr()), self._stream()))
        self._keepalive = (demand_dev, mask_dev)
        if not self.batched:
            self._alloc_histories()
        self.last_obs, self.last_reward = obs_buf, None       # packed [N, m, O] tensor behind the returned views
        self.state = self._shape_obs(obs_buf)
        return self.state

    def _draw_host_delay_mask(self):
        """Drop-in mode: pre-draw the episode's noisy-delay uniforms on the host stream in the reference's order
        (factory first, eligible stages only — MAIM_env.py:447-468 / MAIM_div_env.py:666-687)."""
        m, T = self.num_nodes, self.num_periods
        order = list(range(m)) if self.DIV else [m - 1] + list(range(m - 1))
        delay_mask = np.zeros((T, m), dtype=bool)
        for t in range(T):
            for i in order:
                if t - int(self.delay[i]) >= 0:
                    delay_mask[t, i] = np.random.uniform(0, 1) <= self.noisy_delay_threshold
        return delay_mask

    def _mask_to_device(self, delay_mask):
        N, m, T = self.num_envs, self.num_nodes, self.num_periods
        mk = torch.as_tensor(np.ascontiguousarray(np.asarray(delay_mask)).astype(np.uint8), device=self.device) \
            if not isinstance(delay_mask, torch.Tensor) else delay_mask.to(device=self.device, dtype=torch.uint8)
        if mk.numel() == T * m:
            mk = mk.reshape(1, T, m).expand(N, T, m)
        return mk.reshape(N, T, m).contiguous()

    def delay_mask_device(self):
        """[T, N, m] uint8 view of this episode's noisy-delay outcomes (None without noisy delays)."""
        ptr, cnt = C.c_void_p(), C.c_int64()
        _lib.check(self._lib.imx_state_field(self._handle, _lib.F_DELAY_MASK, C.byref(ptr), C.byref(cnt)))
        if cnt.value == 0:
            return None
        return torch.as_tensor(_DevView(ptr.value, (self.num_periods, self.num_envs, self.num_nodes), "|u1"), device=self.device)

    def customer_demand_device(self):
        """[T, R, N] int32 view of the episode's demand trace as the kernels read it."""
        return self._state_view(_lib.F_DEMAND)

    def _new_obs(self):
        N, m, O = self.num_envs, self.num_nodes, self.obs_len
        if self.reuse_buffers:
            if getattr(self, "_obs_buf", None) is None:
                self._obs_buf = torch.empty((N, m, O), dtype=self.obs_dtype, device=self.device)
            return self._obs_buf
        return torch.empty((N, m, O), dtype=self.obs_dtype, device=self.device)

    def _new_reward(self):
        shape = (self.num_envs, self.num_nodes) if self.MULTI else (self.num_envs,)
        if self.reuse_buffers:
            if getattr(self, "_rew_buf", None) is None:
                self._rew_buf = torch.empty(shape, dtype=torch.float64, device=self.device)
            return self._rew_buf
        return torch.empty(shape, dtype=torch.float64, device=self.device)

    def _actions_to_device(self, action):
        """[N, m] contiguous CUDA tensor in the handle's action dtype.  With action_dtype='float32' a float64 input is rounded
        to float32 first (round to nearest even), so the env decodes the float32 value, not the float64 one."""
        N, m = self.num_envs, self.num_nodes
        if isinstance(action, dict):
            vals = [action[name] for name in self._agent_names]
            if isinstance(vals[0], torch.Tensor):
                act = torch.stack([v.reshape(N) for v in vals], dim=1)
            else:
                act = np.stack([np.asarray(v, dtype=np.float64).reshape(N) for v in vals], axis=1)
        else:
            act = action
        if isinstance(act, torch.Tensor):
            act = act.to(device=self.device, dtype=self.action_dtype).reshape(N, m)
            return act if act.is_contiguous() else act.contiguous()
        arr = np.ascontiguousarray(np.asarray(act, dtype=np.float64).reshape(N, m))   # np.squeeze semantics of IM_env.py:299
        return torch.as_tensor(arr, device=self.device).to(self.action_dtype)

    def step_packed(self, action):
        """Lean batched step for device-side loops (an RL loop with a GPU policy): ``action`` a contiguous ``[N, m]`` CUDA
        tensor of the env's ``action_dtype`` (anything else is converted like ``step`` does), returns the packed tensors
        ``(obs [N, m, O], reward [N, m] / [N], done)`` — no per-agent dicts, no diagnostics.  With
        ``reuse_buffers=True`` the same two output tensors are overwritten every call and nothing is allocated."""
        if isinstance(action, torch.Tensor) and action.dtype == self.action_dtype and action.is_cuda and action.is_contiguous() \
                and action.numel() == self.num_envs * self.num_nodes:
            act = action
        else:
            act = self._actions_to_device(action)
        obs_buf, rew_buf = self._new_obs(), self._new_reward()
        _lib.check(self._lib.imx_step(self._handle, act.data_ptr(), obs_buf.data_ptr(), rew_buf.data_ptr(), None,
                                      torch.cuda.current_stream(self.device).cuda_stream))
        self.last_obs, self.last_reward = obs_buf, rew_buf
        return obs_buf, rew_buf, self.period >= self.num_periods

    def step_cc(self, action, fill_actions=True, clip=(-1.0, 1.0), want_obs=True):
        """``step_packed`` that also returns the centralised-critic observation rows ``[N, m, W]`` (``W = (m-1)(1+O) + O``:
        opponent actions | opponent observations | own observation — central_critic_observer + FillInActions,
        models/CC_Model.py:165-214), emitted by the step kernel's epilogue from the observation tile it has just built.
        ``fill_actions=False`` leaves the opponent-action slots zero, as the observer does at sampling time.
        Returns ``(obs or None, cc_obs, reward, done)``; cc_obs has the env's observation dtype."""
        if not self.MULTI:
            raise _lib.ImxError("the centralised-critic observation is defined for the multi-agent envs")
        act = self._actions_to_device(action)
        N, m, O = self.num_envs, self.num_nodes, self.obs_len
        obs_buf = self._new_obs() if want_obs else None
        rew_buf = self._new_reward()
        W = (m - 1) * (1 + O) + O
        cc_buf = torch.empty((N, m, W), dtype=self.obs_dtype, device=self.device)
        _lib.check(self._lib.imx_step_cc(self._handle, C.c_void_p(act.data_ptr()), C.c_void_p(obs_buf.data_ptr()) if want_obs else None,
                                         C.c_void_p(cc_buf.data_ptr()), int(bool(fill_actions)), float(clip[0]), float(clip[1]),
                                         C.c_void_p(rew_buf.data_ptr()), self._stream()))
        if want_obs:
            self.last_obs, self.last_reward = obs_buf, rew_buf
            self.state = self._shape_obs(obs_buf)
        return obs_buf, cc_buf, rew_buf, self.period >= self.num_periods

    def _cached_views(self, obs_buf, rew_buf):
        """Per-agent dict views of the packed outputs; built once per buffer pair (reuse_buffers keeps the pair alive)."""
        key = (obs_buf.data_ptr(), rew_buf.data_ptr())
        if getattr(self, "_view_key", None) != key:
            self._view_key, self._view_obs, self._view_rew = key, self._shape_obs(obs_buf), self._shape_reward(rew_buf)
        return self._view_obs, self._view_rew

    # ------------------------------------------------------------------ drop-in mode (N = 1): one launch, one synchronisation
    def _mailbox(self):
        """Pinned host buffer the step kernel reads its actions from and writes every output into directly (the pinned
        allocation is device-addressable at the same address under UVA): observation, reward, the five info fields;
        the three state fields the history arrays record follow by ONE small copy.  A drop-in step is then one kernel
        launch + one copy + one stream synchronisation instead of a dozen device->host reads."""
        if getattr(self, "_mail", None) is not None and self._mail_handle == self._handle.value:
            return self._mail_views
        m, O = self.num_nodes, self.obs_len
        es = 4 if self.obs_dtype == torch.float32 else 8
        ptr = {}
        for f in (_lib.F_INV, _lib.F_BACKLOG, _lib.F_ORDER_U):
            p_, c_ = C.c_void_p(), C.c_int64()
            _lib.check(self._lib.imx_state_field(self._handle, f, C.byref(p_), C.byref(c_)))
            ptr[f] = p_.value
        lo = min(ptr.values())
        span = max(ptr.values()) + m * 4 - lo                         # the three fields sit in one block, 256-byte aligned each
        sizes = [("act", m * 8), ("obs", m * O * es), ("rew", (m if self.MULTI else 1) * 8), ("profit", m * 8), ("demand", m * 4),
                 ("ship", m * 4), ("acq", m * 4), ("order", m * 4), ("state", span), ("err", 4)]
        off, offs = 0, {}
        for name, nbytes in sizes:
            offs[name] = (off, nbytes)
            off += (nbytes + 63) & ~63
        self._mail = torch.zeros(off, dtype=torch.uint8).pin_memory()
        host = self._mail.numpy()
        base = self._mail.data_ptr()
        dt = {"act": np.float64, "obs": np.float32 if es == 4 else np.float64, "rew": np.float64, "profit": np.float64, "demand": np.int32,
              "ship": np.int32, "acq": np.int32, "order": np.int32, "state": np.int32, "err": np.int32}
        v = {k: host[o:o + n].view(dt[k]) for k, (o, n) in offs.items()}
        v["addr"] = {k: base + o for k, (o, n) in offs.items()}
        v["state_dst"] = self._mail[offs["state"][0]:offs["state"][0] + span].view(torch.int32)
        v["state_src"] = torch.as_tensor(_DevView(lo, (span // 4,), "<i4"), device=self.device)
        v["state_idx"] = {f: (ptr[f] - lo) // 4 for f in ptr}
        v["err_dst"] = self._mail[offs["err"][0]:offs["err"][0] + 4].view(torch.int32)
        v["info"] = _lib.ImxInfoOut(v["addr"]["demand"], v["addr"]["ship"], v["addr"]["acq"], v["addr"]["order"], v["addr"]["profit"])
        self._mail_views, self._mail_handle = v, self._handle.value
        return v

    def _step_dropin(self, action):
        m, O = self.num_nodes, self.obs_len
        v = self._mailbox()
        t = self.period
        if isinstance(action, dict):
            for i, name in enumerate(self._agent_names):
                a = action[name]
                v["act"][i] = float(a.item() if isinstance(a, torch.Tensor) else np.asarray(a, dtype=np.float64).reshape(-1)[0])
        else:
            v["act"][:] = (action.detach().cpu().numpy() if isinstance(action, torch.Tensor) else np.asarray(action, dtype=np.float64)).reshape(m)
        stream = torch.cuda.current_stream(self.device)
        _lib.check(self._lib.imx_step(self._handle, v["addr"]["act"], v["addr"]["obs"], v["addr"]["rew"], C.byref(v["info"]), stream.cuda_stream))
        with torch.cuda.stream(stream):
            v["state_dst"].copy_(v["state_src"], non_blocking=True)
            if self.DIV:
                v["err_dst"].copy_(self.error_flags[:1], non_blocking=True)
        stream.synchronize()
        if self.DIV and int(v["err"][0]) != 0:
            raise Exception(f"Infinite Loop {int(v['err'][0])}")             # MAIM_div_env.py:503-505 etc.
        idx = v["state_idx"]
        self.inv[t + 1, :] = v["state"][idx[_lib.F_INV]:idx[_lib.F_INV] + m]
        self.backlog[t + 1, :] = v["state"][idx[_lib.F_BACKLOG]:idx[_lib.F_BACKLOG] + m]
        self.order_u[t + 1, :] = v["state"][idx[_lib.F_ORDER_U]:idx[_lib.F_ORDER_U] + m]
        self.demand[t, :] = v["demand"]
        self.ship[t, :] = v["ship"]
        self.acquisition[t, :] = v["acq"]
        self.order_r[t, :] = v["order"]
        obs = v["obs"].reshape(m, O).copy()
        rew, profit = v["rew"].copy(), v["profit"].copy()
        self.last_obs = torch.as_tensor(obs).unsqueeze(0)
        self.last_reward = torch.as_tensor(rew).reshape((1, m) if self.MULTI else (1,))
        done_flag = (t + 1) >= self.num_periods
        if self.MULTI:
            self.state = {name: obs[i] for i, name in enumerate(self._agent_names)}
            reward = {name: np.float64(rew[i]) for i, name in enumerate(self._agent_names)}
            info = {name: {"period": t + 1, "demand": self.demand[t, i], "ship": self.ship[t, i], "acquisition": self.acquisition[t, i],
                           "actual order": self.order_r[t, i], "profit": np.float64(profit[i])}           # post-increment period (quirk 7)
                    for i, name in enumerate(self._agent_names)}
        else:
            self.state = obs
            reward = np.float64(rew[0])
            info = {"period": t, "demand": self.demand[t, :], "ship": self.ship[t, :],                      # pre-increment period (quirk 7)
                    "acquisition": self.acquisition[t, :], "profit": profit}
        return self.state, reward, self._shape_done(done_flag), (info if self.return_info else {})

    def step(self, action):
        """step — IM_env.py:287-360, MAIM_env.py:330-411, IM_div_env.py:361-549, MAIM_div_env.py:441-630."""
        if not self.batched:
            return self._step_dropin(action)
        if self.batched and not self.return_info:           # fast path: one ctypes call, cached views when buffers are reused
            obs_buf, rew_buf, done_flag = self.step_packed(action)
            if self.reuse_buffers:
                self.state, rew = self._cached_views(obs_buf, rew_buf)
            else:
                self.state, rew = self._shape_obs(obs_buf), self._shape_reward(rew_buf)
            return self.state, rew, self._shape_done(done_flag), {}
        N, m = self.num_envs, self.num_nodes
        t = self.period
        act = self._actions_to_device(action)
        obs_buf, rew_buf = self._new_obs(), self._new_reward()
        info_struct, info_bufs = None, None
        if self.return_info:
            info_bufs = {k: torch.empty((N, m), dtype=torch.int32, device=self.device) for k in ("demand", "ship", "acquisition", "order")}
            info_bufs["profit"] = torch.empty((N, m), dtype=torch.float64, device=self.device)
            info_struct = _lib.ImxInfoOut(info_bufs["demand"].data_ptr(), info_bufs["ship"].data_ptr(),
                                          info_bufs["acquisition"].data_ptr(), info_bufs["order"].data_ptr(),
                                          info_bufs["profit"].data_ptr())
        _lib.check(self._lib.imx_step(self._handle, C.c_void_p(act.data_ptr()), C.c_void_p(obs_buf.data_ptr()),
                                      C.c_void_p(rew_buf.data_ptr()),
                                      C.byref(info_struct) if info_struct is not None else None, self._stream()))
        done_flag = self.period >= self.num_periods
        self.last_obs, self.last_reward = obs_buf, rew_buf    # packed [N, m, O] / [N, m] tensors behind the returned views
        self.state = self._shape_obs(obs_buf)
        return self.state, self._shape_reward(rew_buf), self._shape_done(done_flag), self._shape_info(t, info_bufs)

    def step_many(self, actions, obs_out=None, reward_out=None, want_obs=True, return_info=False):
        """K consecutive ``step()`` calls on a stored plan ``actions [K, N, m]`` (the LP scripts' replay loops,
        DSHLP_4.py:905-925) in one call: returns ``(obs [K, N, m, O] or None, reward [K, N, m] / [K, N], done)``, plus with ``return_info=True`` a
        dict of ``[K, N, m]`` tensors ``demand, ship, acquisition, actual order, profit`` (DSHLP_4.py:918-923).
        Same results as K ``step()`` calls; one launch with the state resident on chip where the batch allows it."""
        if not self.batched:
            raise _lib.ImxError("step_many is a batched-mode call (construct the env with num_envs=N)")
        N, m, O = self.num_envs, self.num_nodes, self.obs_len
        act = actions if isinstance(actions, torch.Tensor) else torch.as_tensor(np.asarray(actions, dtype=np.float64))
        act = act.to(device=self.device, dtype=self.action_dtype).reshape(-1, N, m).contiguous()
        K = act.shape[0]
        if want_obs and obs_out is None:
            obs_out = torch.empty((K, N, m, O), dtype=self.obs_dtype, device=self.device)
        if reward_out is None:
            reward_out = torch.empty((K, N, m) if self.MULTI else (K, N), dtype=torch.float64, device=self.device)
        info_struct, info = None, None
        if return_info:                                        # [K, N, m] blocks: what the LP replay loops record per period
            info = {k: torch.empty((K, N, m), dtype=torch.int32, device=self.device) for k in ("demand", "ship", "acquisition", "actual order")}
            info["profit"] = torch.empty((K, N, m), dtype=torch.float64, device=self.device)
            info_struct = _lib.ImxInfoOut(info["demand"].data_ptr(), info["ship"].data_ptr(), info["acquisition"].data_ptr(),
                                          info["actual order"].data_ptr(), info["profit"].data_ptr())
        _lib.check(self._lib.imx_step_many(self._handle, C.c_void_p(act.data_ptr()), K,
                                           C.c_void_p(obs_out.data_ptr()) if obs_out is not None else None,
                                           C.c_void_p(reward_out.data_ptr()),
                                           C.byref(info_struct) if info_struct is not None else None, self._stream()))
        self._keepalive_many = act
        if obs_out is not None:
            self.last_obs, self.last_reward = obs_out[K - 1], reward_out[K - 1]
            self.state = self._shape_obs(obs_out[K - 1])
        done = self.period >= self.num_periods
        if return_info:
            return obs_out, reward_out, self._shape_done(done), info
        return obs_out, reward_out, (self._shape_done(done))

    def replay_episode(self, actions, customer_demand=None, delay_mask=None, noisy_delay=None, want_obs=False, want_rewards=False,
                       returns=True, stats=None, accumulate=False, eval_acc=False):
        """A whole episode on a stored plan ``actions [T, N, m]``: ``reset(customer_demand)`` + T ``step()`` calls + the episode's
        returns, statistics and evaluation-loop accumulators (the LP scripts' replay loop, DSHLP_4.py:896-928) in one call —
        one kernel launch where the batch allows it, without materialising per-period rewards or observations unless asked.

        customer_demand: [N, R, T] / [N, T] / one trace, or None (Philox, the stream ``reset()`` draws from).  Noisy delays follow
        the env's sticky ``noisy_delay`` flag unless ``noisy_delay`` is given; ``delay_mask`` replays them ([N, T, m] / [T, m]).
        stats: None (not wanted), True (a new vector) or a float64 tensor ``[3 (+ 2m)]`` to write, or with ``accumulate=True``
        to add into.  Returns ``dict(returns, stats, obs [T, N, m, O], rewards [T, N(, m)], eval [N, 4 + m])`` with None for
        what was not asked; ``eval`` is what ``eval_accumulate`` builds over the episode (``eval_stats`` / ``eval_summary``
        take it as is).  Leaves the env at period T with the final state."""
        if not self.batched:
            raise _lib.ImxError("replay_episode is a batched-mode call (construct the env with num_envs=N)")
        N, m, O, T = self.num_envs, self.num_nodes, self.obs_len, self.num_periods
        act = actions if isinstance(actions, torch.Tensor) else torch.as_tensor(np.asarray(actions, dtype=np.float64))
        act = act.to(device=self.device, dtype=self.action_dtype)
        if act.numel() != T * N * m:
            raise ValueError(f"actions must hold a whole episode: [T={T}, N={N}, m={m}]")
        act = act.reshape(T, N, m).contiguous()
        demand_dev = self._demand_to_device(customer_demand) if customer_demand is not None else None
        want_noisy = (bool(self.noisy_delay) if noisy_delay is None else bool(noisy_delay)) or delay_mask is not None
        mask_dev = None
        if want_noisy:
            if not self._has_carry:
                self._create_handle(True)
            if delay_mask is not None:
                mask_dev = self._mask_to_device(delay_mask)
        cols = (m,) if self.MULTI else ()
        f64 = dict(dtype=torch.float64, device=self.device)
        obs = torch.empty((T, N, m, O), dtype=self.obs_dtype, device=self.device) if want_obs else None
        rew = torch.empty((T, N) + cols, **f64) if want_rewards else None
        ret = torch.empty((N,) + cols, **f64) if returns else None
        if stats is True:
            stats = torch.zeros(3 + (2 * m if self.MULTI else 0), **f64)
        elif stats is False:
            stats = None
        if stats is not None and (stats.dtype != torch.float64 or not stats.is_contiguous() or stats.numel() != 3 + (2 * m if self.MULTI else 0)):
            raise ValueError("stats must be a contiguous float64 tensor of 3 (+ 2m for the multi-agent kinds) entries")
        ev = torch.empty((N, 4 + m), **f64) if eval_acc else None
        self._episode += 1
        p = lambda x: C.c_void_p(x.data_ptr()) if x is not None else None   # noqa: E731
        _lib.check(self._lib.imx_replay_episode(self._handle, p(demand_dev), p(mask_dev), int(want_noisy), self._episode, p(act),
                                                p(obs), p(rew), p(ret), p(stats), int(bool(accumulate)), p(ev), self._stream()))
        self._keepalive = (act, demand_dev, mask_dev)
        if obs is not None:
            self.last_obs = obs[T - 1]
            self.state = self._shape_obs(obs[T - 1])
        if rew is not None:
            self.last_reward = rew[T - 1]
        return {"returns": ret, "stats": stats, "obs": obs, "rewards": rew, "eval": ev}

    # ------------------------------------------------------------------ drop-in mode histories
    def _alloc_histories(self):
        T, m = self.num_periods, self.num_nodes
        self.inv = np.zeros([T + 1, m])
        self.order_r = np.zeros([T, m])
        self.order_u = np.zeros([T + 1, m])
        self.ship = np.zeros([T, m])
        self.acquisition = np.zeros([T, m])
        self.backlog = np.zeros([T + 1, m])
        self.demand = np.zeros([T + 1, m])
        self.inv[0, :] = np.asarray(self.inv_init, dtype=np.float64)
        d = np.asarray(self.customer_demand)
        if self.DIV:
            for k, node in enumerate(self._retailers):
                self.demand[0, node] = d[k][0]
        else:
            self.demand[0, 0] = d.reshape(-1)[0]                          # pre-filled unclipped (quirk 8)

    def _record_history(self, t, info_bufs):
        sv = self._state_view
        self.inv[t + 1, :] = sv(_lib.F_INV)[0].cpu().numpy()
        self.backlog[t + 1, :] = sv(_lib.F_BACKLOG)[0].cpu().numpy()
        self.order_u[t + 1, :] = sv(_lib.F_ORDER_U)[0].cpu().numpy()
        if info_bufs is not None:
            self.demand[t, :] = info_bufs["demand"][0].cpu().numpy()
            self.ship[t, :] = info_bufs["ship"][0].cpu().numpy()
            self.acquisition[t, :] = info_bufs["acquisition"][0].cpu().numpy()
            self.order_r[t, :] = info_bufs["order"][0].cpu().numpy()

    # shaping hooks ------------------------------------------------------
    def _shape_obs(self, obs_buf):
        raise NotImplementedError

    def _shape_reward(self, rew_buf):
        raise NotImplementedError

    def _shape_done(self, flag):
        raise NotImplementedError

    def _shape_info(self, t, info_bufs):
        raise NotImplementedError

    # ------------------------------------------------------------------ fused base-stock rollout
    def rollout_basestock(self, z, customer_demand=None, pmf=None, step_rewards=False, write_state=False, delay_mask=None,
                          noisy_delay=None):
        """Whole-episode order-up-to rollout in one kernel (dfo_func's loop, base_restock_policy.py:30-45).

        z: [m] or [N, m] base-stock levels.  customer_demand: [N, R, T] / [N, T] / one trace, or None
        (Philox).  pmf: probabilities of the trace, [N, R, T] / [R, T] / [N, T] / [T].  Noisy delays follow the
        env's sticky ``noisy_delay`` flag (MAIM_env.py:192-194) unless ``noisy_delay`` is given; ``delay_mask``
        replays their outcomes ([N, T, m] / [T, m]), otherwise the drop-in draws them from numpy's global stream in
        the reference's order and a batched env from Philox.
        Returns dict(returns=[N] or [N, m], step_rewards=[T, N(, m)] or None, dfo=[N] or None)."""
        N, m, T, R = self.num_envs, self.num_nodes, self.num_periods, len(self._retailers)
        zt = torch.as_tensor(np.asarray(z, dtype=np.float64), device=self.device) if not isinstance(z, torch.Tensor) \
            else z.to(device=self.device, dtype=torch.float64)
        zt = zt.contiguous()
        if zt.numel() == m:
            stride = 0
        elif zt.numel() == N * m:
            stride = m
        else:
            raise ValueError("z must have m or N*m entries")
        demand_dev = self._demand_to_device(customer_demand) if customer_demand is not None else None
        pmf_dev = None
        if pmf is not None:
            pmf_dev = torch.as_tensor(np.asarray(pmf, dtype=np.float64), device=self.device) if not isinstance(pmf, torch.Tensor) \
                else pmf.to(device=self.device, dtype=torch.float64)
            if pmf_dev.numel() == R * T:
                pmf_dev = pmf_dev.reshape(1, R, T).expand(N, R, T)
            pmf_dev = pmf_dev.reshape(N, R, T).contiguous()
        want_noisy = (bool(self.noisy_delay) if noisy_delay is None else bool(noisy_delay)) or delay_mask is not None
        mask_dev = None
        if want_noisy:
            if not self._has_carry:
                self._create_handle(True)
            if delay_mask is None and not self.batched:
                delay_mask = self._draw_host_delay_mask()
            if delay_mask is not None:
                mask_dev = self._mask_to_device(delay_mask)
        ret = torch.empty((N, m) if self.MULTI else (N,), dtype=torch.float64, device=self.device)
        dfo = torch.empty((N,), dtype=torch.float64, device=self.device) if (pmf_dev is not None and not self.MULTI) else None
        want_sr = step_rewards or dfo is not None            # the objective kernel reads the per-period rewards
        sr = torch.empty((T, N, m) if self.MULTI else (T, N), dtype=torch.float64, device=self.device) if want_sr else None
        self._episode += 1
        p = lambda x: C.c_void_p(x.data_ptr()) if x is not None else None   # noqa: E731
        _lib.check(self._lib.imx_rollout_basestock(self._handle, p(zt), stride, p(demand_dev), p(mask_dev), int(want_noisy),
                                                   self._episode, p(pmf_dev), p(ret), p(sr), p(dfo), int(write_state), self._stream()))
        self._keepalive = (zt, demand_dev, pmf_dev, mask_dev)
        return {"returns": ret, "step_rewards": sr if step_rewards else None, "dfo": dfo}

    def return_stats(self, returns):
        """[n, Σ, Σ², then per agent (Σ, Σ²)] float64 on the device — the payload of the cross-GPU all-reduce."""
        m = self.num_nodes
        out = torch.empty(3 + (2 * m if self.MULTI else 0), dtype=torch.float64, device=self.device)
        _lib.check(self._lib.imx_return_stats(self._handle, C.c_void_p(returns.data_ptr()), C.c_void_p(out.data_ptr()), self._stream()))
        return out

    def episode_stats(self, step_rewards, stats=None, accumulate=False, returns=None):
        """step_rewards [T, N, m] (MAIM kinds) or [T, N] float64 on the device → statistics vector (see
        return_stats); ``accumulate=True`` adds into ``stats`` (evaluation batches, one all-reduce at the end);
        ``returns`` ([N, m] / [N] float64, contiguous) also receives the episode returns (sum over periods in period order)."""
        m = self.num_nodes
        if stats is None:
            stats = torch.zeros(3 + (2 * m if self.MULTI else 0), dtype=torch.float64, device=self.device)
        sr = step_rewards.contiguous()
        if returns is not None and (not returns.is_contiguous() or returns.dtype != torch.float64 or returns.numel() != sr[0].numel()):
            raise ValueError("returns must be a contiguous float64 tensor of one period's reward shape")
        _lib.check(self._lib.imx_episode_stats(self._handle, C.c_void_p(sr.data_ptr()), int(sr.shape[0]),
                                               C.c_void_p(returns.data_ptr()) if returns is not None else None,
                                               C.c_void_p(stats.data_ptr()), int(bool(accumulate)), self._stream()))
        return stats

    # ------------------------------------------------------------------ evaluation-loop accumulators
    EVAL_COLUMNS = ("episode_reward", "total_inventory", "total_backlog", "customer_backlog")

    def eval_accumulate(self, acc, obs, reward, profit=None, reset=False):
        """One step of the scripts' evaluation loop (MA_inv_management.py:568-581, inv_management.py:585-600,
        DSHLP_4.py:908-913) for the whole batch, on the device: ``acc [N, 4 + m]`` float64 rows
        ``{episode_reward, total_inventory, total_backlog, customer_backlog, stage_profit[m]}``.
        ``obs`` / ``reward`` are what ``step()`` returned (dicts or the packed tensors), ``profit`` is
        ``info[...]['profit']`` packed ``[N, m]`` or None.  ``acc=None`` allocates; ``reset=True`` starts an episode."""
        N, m = self.num_envs, self.num_nodes
        if acc is None:
            acc = torch.zeros((N, 4 + m), dtype=torch.float64, device=self.device)
            reset = True
        pack = lambda d, shape: (torch.stack([d[a] for a in self._agent_names], dim=1) if isinstance(d, dict) else d).reshape(shape).contiguous()   # noqa: E731
        o = pack(obs, (N, m, self.obs_len))
        if o.dtype != self.obs_dtype:
            raise TypeError(f"observations must be {self.obs_dtype} (the dtype this env writes)")
        r = pack(reward, (N, m) if self.MULTI else (N,)).to(torch.float64)
        pr = pack(profit, (N, m)).to(torch.float64) if profit is not None else None
        _lib.check(self._lib.imx_eval_accumulate(self._handle, C.c_void_p(o.data_ptr()), C.c_void_p(r.data_ptr()),
                                                 C.c_void_p(pr.data_ptr()) if pr is not None else None,
                                                 C.c_void_p(acc.data_ptr()), int(bool(reset)), self._stream()))
        self._keepalive_eval = (o, r, pr)
        return acc

    def eval_stats(self, acc, stats=None, accumulate=False):
        """``{n, then (Σ, Σ²) per column of acc}`` float64 ``[1 + 2(4 + m)]`` on the device — the inputs of the
        ``np.mean`` / ``np.std`` lines MA_inv_management.py:589-600; add across GPUs with one all-reduce."""
        W = 4 + self.num_nodes
        if stats is None:
            stats = torch.zeros(1 + 2 * W, dtype=torch.float64, device=self.device)
        _lib.check(self._lib.imx_eval_stats(self._handle, C.c_void_p(acc.data_ptr()), C.c_void_p(stats.data_ptr()),
                                            int(bool(accumulate)), self._stream()))
        return stats

    @staticmethod
    def eval_summary(stats, num_nodes):
        """mean / population std (np.std, ddof = 0) per accumulator column from an ``eval_stats`` vector."""
        st = np.asarray(stats.detach().cpu().numpy() if isinstance(stats, torch.Tensor) else stats, dtype=np.float64)
        n = st[0]
        names = list(_ImxEnvBase.EVAL_COLUMNS) + [f"stage_profit_{i}" for i in range(num_nodes)]
        out = {}
        for k, name in enumerate(names):
            mean = st[1 + 2 * k] / n
            out[name] = (mean, float(np.sqrt(max(st[2 + 2 * k] / n - mean * mean, 0.0))))
        return out

    # ------------------------------------------------------------------ spaces
    def _obs_shape_declared(self):
        """Per-agent observation length the reference declares (MAIM_env.py:83-153)."""
        P, D = int(self.prev_length), int(self.max_delay)
        td, pa, pd = bool(self.time_dependency), bool(self.prev_actions), bool(self.prev_demand)
        n = 3 + (D if td else 0) + (P if pa else 0) + (P if pd else 0)
        if self.KIND == "MAIM" and not self.standardise_state:
            n = 3 + (D if td else 0)                                    # quirk 13: declared shape ignores the history slots
        if getattr(self, "share_network", False):
            n += 1
        return n

    def _build_spaces(self):
        m, a, b = self.num_nodes, self.a, self.b
        n = self._obs_shape_declared()
        inv_max_obs = float(np.max(self.inv_max))
        order_max_obs = float(np.max(self.order_max))
        if self.MULTI:
            if self.standardise_actions:
                self.action_space = Box(low=np.ones(1) * a, high=np.ones(1) * b, dtype=np.float64, shape=(1,))
            else:
                self.action_space = Box(low=np.zeros(1), high=np.ones(1) * order_max_obs, dtype=np.int32, shape=(1,))
            if self.standardise_state:
                self.observation_space = Box(low=np.ones(n) * a, high=np.ones(n) * b, dtype=np.float64, shape=(n,))
            else:
                high = np.ones(n) * inv_max_obs
                high[1] = np.inf
                self.observation_space = Box(low=np.zeros(n), high=high, dtype=np.float64, shape=(n,))
        else:
            if self.standardise_actions:
                self.action_space = Box(low=np.ones(m) * a, high=np.ones(m) * b, dtype=np.float64, shape=(m,))
            else:
                self.action_space = Box(low=np.zeros(m), high=np.asarray(self.order_max, dtype=np.float64), dtype=np.int32, shape=(m,))
            if self.standardise_state:
                self.observation_space = Box(low=np.ones((m, n)) * a, high=np.ones((m, n)) * b, dtype=np.float64, shape=(m, n))
            else:
                high = np.ones((m, n)) * inv_max_obs
                high[:, 1] = np.inf
                self.observation_space = Box(low=np.zeros((m, n)), high=high, dtype=np.float64, shape=(m, n))


# ======================================================================================
# serial chains
# ======================================================================================
class _SerialMixin:
    DIV = False
    AGENT_PREFIX = "stage_"

    def _parse_structure(self, config, take):
        if self.MULTI:
            self.independent = take("independent", True)                 # MAIM_env.py:16
        self.num_stages = take("num_stages", 3)
        self.num_nodes = self.num_stages
        m = self.num_stages
        self._agent_names = [self.AGENT_PREFIX + str(i) for i in range(m)]
        if self.MULTI:
            self.stage_names = list(self._agent_names)
            self.num_agents = take("num_agents", m)
        self.inv_init = take("init_inv", np.ones(m) * (100 if self.MULTI else 20))
        self.inv_target = take("inv_target", np.ones(m) * 10)
        self.delay = take("delay", np.ones(m, dtype=np.int8))
        self.price = take("price", np.flip(np.arange(m + 1) + 1))

    def _parse_capacities(self, config, take):
        m = self.num_stages
        self.inv_max = take("inv_max", np.ones(m, dtype=np.int32) * (200 if self.MULTI else 100))
        order_max = np.zeros(m)
        for i in range(m - 1):
            order_max[i] = self.inv_max[i + 1]
        order_max[m - 1] = self.inv_max[m - 1]
        self.order_max = take("order_max", order_max)
        self.demand_max = np.asarray(self.inv_max).copy()
        self.retailers = [0]
        for i in range(len(self.price) - 1):
            assert self.price[i] > self.price[i + 1]                     # MAIM_env.py:167-168
        assert self.order_max[m - 1] <= self.inv_max[m - 1]              # MAIM_env.py:171
        if min(int(d) for d in np.asarray(self.delay).reshape(-1)) < 1:
            raise ValueError("delay must be >= 1 for every stage")


class _DivMixin:
    DIV = True
    AGENT_PREFIX = "node_"

    def _parse_structure(self, config, take):
        if self.MULTI:
            self.independent = take("independent", True)
            self.share_network = take("share_network", False)
        self.num_nodes = take("num_nodes", 3)
        m = self.num_nodes
        self._agent_names = [self.AGENT_PREFIX + str(i) for i in range(m)]
        if self.MULTI:
            self.node_names = list(self._agent_names)
        self.connections = take("connections", {0: [1], 1: [2], 2: []})
        check_connections(self.connections)
        self.network = create_network(self.connections)
        self.order_network = np.transpose(self.network)
        self.retailers = get_retailers(self.network)
        self.non_retailers = [i for i in range(m) if i not in self.retailers]
        self.upstream_node = {i: int(np.where(self.order_network[i] == 1)[0][0]) for i in range(1, m)}
        self.num_stages = get_stage(node=int(m - 1), network=self.network) + 1
        if self.MULTI:
            self.num_agents = take("num_agents", m)
        self.inv_init = take("init_inv", np.ones(m) * (100 if self.MULTI else 20))
        self.inv_target = take("inv_target", np.ones(m) * (0 if self.MULTI else 10))
        self.delay = take("delay", np.ones(m, dtype=np.int8))
        stage_price = np.arange(self.num_stages) + 2                    # MAIM_div_env.py:55-61
        stage_cost = np.arange(self.num_stages) + 1
        self.node_price = np.array([stage_price[get_stage(i, self.network)] for i in range(m)], dtype=np.float64)
        self.node_cost = np.array([stage_cost[get_stage(i, self.network)] for i in range(m)], dtype=np.float64)
        self.price = take("price", np.flip(np.arange(self.num_stages + 1) + 1))   # read but unused, like the reference

    def _parse_capacities(self, config, take):
        m = self.num_nodes
        self.inv_max = take("inv_max", np.ones(m, dtype=np.int16) * 100)
        order_max = np.zeros(m)
        for i in range(1, m):
            order_max[i] = self.inv_max[self.upstream_node[i]]
        order_max[0] = self.inv_max[0]
        self.order_max = take("order_max", order_max)
        self.num_downstream = {i: int(np.sum(self.network[i])) for i in range(m)}
        self.demand_max = np.asarray(self.inv_max).copy()               # MAIM_div_env.py:91-99
        for i in range(m):
            s = sum(self.order_max[j] for j in range(m) if self.network[i][j] == 1)
            if s > self.demand_max[i]:
                self.demand_max[i] = s
        assert self.order_max[0] <= self.inv_max[0]                      # MAIM_div_env.py:235
        if min(int(d) for d in np.asarray(self.delay).reshape(-1)) < 1:
            raise ValueError("delay must be >= 1 for every node")


class _SingleAgentShape:
    """gym.Env surface: obs [m, O] (batched [N, m, O]), scalar reward (batched [N]), bool done,
    info {period, demand, ship, acquisition, profit} (IM_env.py:345-360)."""
    MULTI = False

    def _shape_obs(self, obs_buf):
        return obs_buf if self.batched else obs_buf[0].cpu().numpy()

    def _shape_reward(self, rew_buf):
        return rew_buf if self.batched else np.float64(rew_buf[0].item())

    def _shape_done(self, flag):
        return bool(flag)

    def _shape_info(self, t, bufs):
        if bufs is None:
            return {}
        if self.batched:
            return {"period": t, "demand": bufs["demand"], "ship": bufs["ship"], "acquisition": bufs["acquisition"],
                    "actual order": bufs["order"], "profit": bufs["profit"]}
        return {"period": t, "demand": self.demand[t, :], "ship": self.ship[t, :],          # pre-increment period (quirk 7)
                "acquisition": self.acquisition[t, :], "profit": bufs["profit"][0].cpu().numpy()}


class _MultiAgentShape:
    """RLlib MultiAgentEnv surface: dicts keyed by agent id (MAIM_env.py:395-411)."""
    MULTI = True

    def _shape_obs(self, obs_buf):
        if self.batched:
            return dict(zip(self._agent_names, obs_buf.unbind(1)))          # m views from one call
        host = obs_buf[0].cpu().numpy()
        return {name: host[i].copy() for i, name in enumerate(self._agent_names)}

    def _shape_reward(self, rew_buf):
        if self.batched:
            return dict(zip(self._agent_names, rew_buf.unbind(1)))
        host = rew_buf[0].cpu().numpy()
        return {name: np.float64(host[i]) for i, name in enumerate(self._agent_names)}

    def _shape_done(self, flag):
        return {"__all__": bool(flag)}

    def _shape_info(self, t, bufs):
        if bufs is None:
            return {}
        info = {}
        if self.batched:
            for i, name in enumerate(self._agent_names):
                info[name] = {"period": t + 1, "demand": bufs["demand"][:, i], "ship": bufs["ship"][:, i],
                              "acquisition": bufs["acquisition"][:, i], "actual order": bufs["order"][:, i],
                              "profit": bufs["profit"][:, i]}
            return info
        profit = bufs["profit"][0].cpu().numpy()
        for i, name in enumerate(self._agent_names):
            info[name] = {"period": t + 1, "demand": self.demand[t, i], "ship": self.ship[t, i],   # post-increment (quirk 7)
                          "acquisition": self.acquisition[t, i], "actual order": self.order_r[t, i],
                          "profit": np.float64(profit[i])}
        return info


class _BatchedHistoryMixin:
    """In batched mode ``env.inv / env.order_u / env.backlog`` are period-indexed proxies."""

    def _install_batched_histories(self):
        self.inv = _History(self, _lib.F_INV)
        self.backlog = _History(self, _lib.F_BACKLOG)
        self.order_u = _History(self, _lib.F_ORDER_U)


def _finish_init(env):
    if env.batched:
        env._install_batched_histories()


class InvManagement(_SerialMixin, _SingleAgentShape, _BatchedHistoryMixin, _ImxEnvBase):
    """Drop-in for environments/IM_env.py:6 ``InvManagement(gym.Env)``."""
    KIND = "IM"

    def __init__(self, config):
        super().__init__(config)
        _finish_init(self)


class MultiAgentInvManagement(_SerialMixin, _MultiAgentShape, _BatchedHistoryMixin, _ImxEnvBase):
    """Drop-in for environments/MAIM_env.py:7 ``MultiAgentInvManagement(MultiAgentEnv)``."""
    KIND = "MAIM"

    def __init__(self, config):
        super().__init__(config)
        _finish_init(self)


class InvManagementDiv(_DivMixin, _SingleAgentShape, _BatchedHistoryMixin, _ImxEnvBase):
    """Drop-in for environments/IM_div_env.py:8 ``InvManagementDiv(gym.Env)``."""
    KIND = "IM_div"

    def __init__(self, config):
        super().__init__(config)
        _finish_init(self)


class MultiAgentInvManagementDiv(_DivMixin, _MultiAgentShape, _BatchedHistoryMixin, _ImxEnvBase):
    """Drop-in for environments/MAIM_div_env.py:8 ``MultiAgentInvManagementDiv(MultiAgentEnv)``."""
    KIND = "MAIM_div"

    def __init__(self, config):
        super().__init__(config)
        _finish_init(self)


ENV_CLASSES = {"IM": InvManagement, "MAIM": MultiAgentInvManagement, "IM_div": InvManagementDiv,
               "MAIM_div": MultiAgentInvManagementDiv}
