"""ctypes binding of the C ABI declared in include/imx_b200.h (libimx_b200.so).

There is deliberately no fallback: if the shared library is missing, fails to load or lacks a
symbol, ``load()`` raises, and so does every env constructor.
"""
from __future__ import annotations

import ctypes as C
import os

MAX_NODES, MAX_CHILDREN, MAX_DELAY, MAX_HIST = 32, 8, 8, 8
ABI_VERSION = 3          # IMX_ABI_VERSION of include/imx_b200.h this binding mirrors
KIND = {"IM": 0, "MAIM": 1, "IM_div": 2, "MAIM_div": 3}
DIST = {"replay": 0, "custom": 0, "poisson": 1, "uniform": 2}
PREPARE_EPISODE = 32    # IMX_PREPARE_EPISODE: imx_replay_episode's kernels and scratch (imx_prepare)
IO_OBS_BF16, IO_ACTIONS_F32 = 1, 2   # imx_config.io_flags: bfloat16 observations, float32 actions
F_INV, F_BACKLOG, F_ORDER_U, F_PIPE, F_HIST_D, F_HIST_O, F_CARRY, F_BACKLOG_TO, F_ERROR, F_DEMAND, F_DELAY_MASK = range(11)

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libimx_b200.so")


class ImxConfig(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("num_nodes", C.c_int32), ("num_periods", C.c_int32), ("prev_length", C.c_int32),
        ("time_dependency", C.c_int32), ("prev_demand", C.c_int32), ("prev_actions", C.c_int32),
        ("standardise_state", C.c_int32), ("standardise_actions", C.c_int32), ("independent", C.c_int32),
        ("share_network", C.c_int32), ("noisy_delay", C.c_int32), ("demand_dist", C.c_int32),
        ("uniform_low", C.c_int32), ("uniform_high", C.c_int32), ("device", C.c_int32),
        ("obs_f32", C.c_int32), ("io_flags", C.c_int32),
        ("a", C.c_double), ("b", C.c_double), ("mu", C.c_double), ("noisy_delay_threshold", C.c_double), ("noisy_demand_threshold", C.c_double),
        ("seed", C.c_uint64), ("num_envs", C.c_int64), ("env_offset", C.c_int64),
        ("inv_init", C.c_int32 * MAX_NODES), ("inv_max", C.c_int32 * MAX_NODES),
        ("order_max", C.c_int32 * MAX_NODES), ("delay", C.c_int32 * MAX_NODES),
        ("inv_target", C.c_double * MAX_NODES), ("stock_cost", C.c_double * MAX_NODES),
        ("backlog_cost", C.c_double * MAX_NODES), ("price", C.c_double * (MAX_NODES + 1)),
        ("num_children", C.c_int32 * MAX_NODES), ("children", (C.c_int32 * MAX_CHILDREN) * MAX_NODES),
    ]


class ImxInfoOut(C.Structure):
    _fields_ = [("demand_dev", C.c_void_p), ("ship_dev", C.c_void_p), ("acquisition_dev", C.c_void_p),
                ("order_dev", C.c_void_p), ("profit_dev", C.c_void_p)]


# every symbol include/imx_b200.h declares: (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "imx_last_error": (C.c_char_p, []),
    "imx_abi_version": (C.c_int, []),
    "imx_config_size": (C.c_int, []),
    "imx_create": (C.c_int, [C.POINTER(ImxConfig), C.POINTER(_P)]),
    "imx_destroy": (C.c_int, [_P]),
    "imx_obs_len": (C.c_int, [_P]),
    "imx_state_words": (C.c_int, [_P]),
    "imx_num_retailers": (C.c_int, [_P]),
    "imx_pipe_words": (C.c_int, [_P]),
    "imx_ledger_words": (C.c_int, [_P]),
    "imx_retailers": (C.c_int, [_P, C.POINTER(C.c_int32)]),
    "imx_demand_max": (C.c_int, [_P, C.POINTER(C.c_int32)]),
    "imx_node_price": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "imx_state_field": (C.c_int, [_P, C.c_int, C.POINTER(_P), C.POINTER(C.c_int64)]),
    "imx_period": (C.c_int, [_P]),
    "imx_set_period": (C.c_int, [_P, C.c_int]),
    "imx_reset": (C.c_int, [_P, _P, _P, C.c_int, C.c_uint64, _P, _P]),
    "imx_step": (C.c_int, [_P, _P, _P, _P, C.POINTER(ImxInfoOut), _P]),
    "imx_step_many": (C.c_int, [_P, _P, C.c_int, _P, _P, C.POINTER(ImxInfoOut), _P]),
    "imx_replay_episode": (C.c_int, [_P, _P, _P, C.c_int, C.c_uint64, _P, _P, _P, _P, _P, C.c_int, _P, _P]),
    "imx_rollout_basestock": (C.c_int, [_P, _P, C.c_int, _P, _P, C.c_int, C.c_uint64, _P, _P, _P, _P, C.c_int, _P]),
    "imx_prepare": (C.c_int, [_P, C.c_int]),
    "imx_step_cc": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_double, C.c_double, _P, _P]),
    "imx_return_stats": (C.c_int, [_P, _P, _P, _P]),
    "imx_reset_host": (C.c_int, [_P, _P, _P, C.c_int, C.c_uint64, _P]),
    "imx_step_host": (C.c_int, [_P, _P, _P, _P]),
    "imx_poisson_cdf": (C.c_int, [_P, C.POINTER(C.c_double), C.c_int]),
    "imx_episode_stats": (C.c_int, [_P, _P, C.c_int, _P, _P, C.c_int, _P]),
    "imx_eval_len": (C.c_int, [_P]),
    "imx_eval_accumulate": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, _P]),
    "imx_eval_stats": (C.c_int, [_P, _P, _P, C.c_int, _P]),
    "imx_cc_obs_len": (C.c_int, [_P]),
    "imx_cc_observe": (C.c_int, [_P, _P, _P, C.c_double, C.c_double, _P, C.c_int, _P]),
    "imx_kernel_variant": (C.c_int, [_P]),
    "imx_jit_log": (C.c_char_p, []),
    "imx_jit_compile_check": (C.c_int, [C.POINTER(ImxConfig), C.c_int, C.c_char_p, C.c_int]),
    "imx_round_bf16": (C.c_int, [_P, _P, C.c_int64]),
    "imx_launch_count": (C.c_int64, []),
}

_lib = None


class ImxError(RuntimeError):
    pass


def load():
    """dlopen libimx_b200.so and bind every declared symbol; raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImxError(f"{LIB_PATH} not found — run `python __graft_entry__.py` (nvcc, sm_100a) first; "
                       "there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.imx_config_size() != C.sizeof(ImxConfig):
        raise ImxError(f"imx_config layout mismatch: C {lib.imx_config_size()} vs ctypes {C.sizeof(ImxConfig)}")
    if lib.imx_abi_version() != ABI_VERSION:
        raise ImxError(f"unexpected ABI version {lib.imx_abi_version()}")
    _lib = lib
    return lib


def check(rc: int):
    if rc < 0:
        msg = load().imx_last_error().decode("utf-8", "replace")
        if rc == -5:
            raise Exception(msg)              # 'Not Implemented' — same exception type the reference raises
        if rc == -6:
            raise IndexError(msg)             # stepping past the episode end (reference: IndexError on its arrays)
        raise ImxError(msg)
    return rc
