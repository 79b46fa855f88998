"""TEST INFRASTRUCTURE — loader for the UNMODIFIED reference envs (only works where a checkout of the
reference is present: IMX_REFERENCE_ROOT, default oracle/_ref, which git ignores).

The reference (MarwanMousa/MARL-for-IM) is pure Python and needs `gym` and
`ray.rllib` only for two base classes and `gym.spaces.Box`; neither package is
installed here.  This module registers ~25 lines of stand-in modules in
``sys.modules`` and then imports ``environments/*.py``, ``utils.py`` and
``base_restock_policy.py`` straight from the read-only reference tree.  Nothing is
copied; the reference code runs as is.

Used by: ``tests/golden/make_golden.py`` (fixture generation) and the
``test_oracle_vs_reference`` tests (skipped when the tree is absent).
Never imported by the product package.
"""
from __future__ import annotations

import os
import sys
import types
import warnings

REFERENCE_ROOT = os.environ.get("IMX_REFERENCE_ROOT", os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref"))


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "environments", "MAIM_env.py"))


class _Box:
    """Stand-in for gym.spaces.Box: stores what the reference passes in."""

    def __init__(self, low=None, high=None, dtype=None, shape=None):
        self.low, self.high, self.dtype, self.shape = low, high, dtype, shape


def _install_stubs() -> None:
    if "gym" not in sys.modules:
        gym = types.ModuleType("gym")
        spaces = types.ModuleType("gym.spaces")
        spaces.Box = _Box
        gym.spaces = spaces
        gym.Env = type("Env", (), {})
        sys.modules["gym"] = gym
        sys.modules["gym.spaces"] = spaces
    if "ray" not in sys.modules:
        ray = types.ModuleType("ray")
        rllib = types.ModuleType("ray.rllib")
        agents = types.ModuleType("ray.rllib.agents")
        rllib.MultiAgentEnv = type("MultiAgentEnv", (), {})
        rllib.agents = agents
        ray.rllib = rllib
        sys.modules["ray"] = ray
        sys.modules["ray.rllib"] = rllib
        sys.modules["ray.rllib.agents"] = agents


_cache = {}


def load_reference():
    """Returns a namespace with the four reference env classes and the base-stock helpers."""
    if "ns" in _cache:
        return _cache["ns"]
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    _install_stubs()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from environments.IM_env import InvManagement
        from environments.MAIM_env import MultiAgentInvManagement
        from environments.IM_div_env import InvManagementDiv
        from environments.MAIM_div_env import MultiAgentInvManagementDiv
        import base_restock_policy as brp
        import utils as ref_utils
    ns = types.SimpleNamespace(
        InvManagement=InvManagement,
        MultiAgentInvManagement=MultiAgentInvManagement,
        InvManagementDiv=InvManagementDiv,
        MultiAgentInvManagementDiv=MultiAgentInvManagementDiv,
        base_stock_policy=brp.base_stock_policy,
        dfo_func=brp.dfo_func,
        create_network=ref_utils.create_network,
        get_stage=ref_utils.get_stage,
        get_retailers=ref_utils.get_retailers,
        check_connections=ref_utils.check_connections,
    )
    _cache["ns"] = ns
    return ns


def load_reference_cc_observer():
    """central_critic_observer from models/CC_Model.py, imported unmodified.  The module pulls in a
    dozen RLlib names at import time; they are stubbed (the observer itself is pure numpy)."""
    if "cc" in _cache:
        return _cache["cc"]
    _install_stubs()
    import torch

    def mod(name, **attrs):
        m = sys.modules.get(name) or types.ModuleType(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m
        return m

    sys.modules["gym.spaces"].Box = _Box
    mod("ray.rllib.agents.callbacks", DefaultCallbacks=type("DefaultCallbacks", (), {}))
    mod("ray.rllib.models", ModelCatalog=type("ModelCatalog", (), {}))
    mod("ray.rllib.policy")
    mod("ray.rllib.policy.sample_batch", SampleBatch=type("SampleBatch", (), {"CUR_OBS": "obs", "ACTIONS": "actions"}))
    mod("ray.rllib.models.torch")
    mod("ray.rllib.models.torch.torch_modelv2", TorchModelV2=type("TorchModelV2", (), {}))
    mod("ray.rllib.utils")
    mod("ray.rllib.utils.framework", try_import_torch=lambda: (torch, torch.nn))
    mod("ray.rllib.models.torch.fcnet", FullyConnectedNetwork=type("FullyConnectedNetwork", (), {}))
    mod("ray.rllib.models.torch.recurrent_net", RecurrentNetwork=type("RecurrentNetwork", (), {}))
    mod("ray.rllib.utils.annotations", override=lambda cls: (lambda f: f))
    mod("ray.rllib.models.modelv2", ModelV2=type("ModelV2", (), {}))
    mod("ray.rllib.models.preprocessors", get_preprocessor=lambda *a, **k: None)
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from models.CC_Model import central_critic_observer
    _cache["cc"] = central_critic_observer
    return central_critic_observer
