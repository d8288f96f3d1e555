"""Stubs that let the UNMODIFIED reference shells import and run in this container
(TEST INFRASTRUCTURE; used by tests/golden/make_shell_golden.py and tests/test_reference_live.py).

The reference's shells need ``tkinter``, ``gym``, ``ray.rllib.env.multi_agent_env``, ``rvo2`` and
``time.clock`` (collision_avoidance/envs/collision_avoidence_env.py:5-16,414,486;
collision_avoidance/ALAN/ALAN_true.py:5-6), none of which exist here (SURVEY F2, Q10).  ``install``
puts inert stand-ins into ``sys.modules`` and binds ``rvo2.PyRVOSimulator`` to whatever
PyRVOSimulator-compatible class the caller passes (the CPU oracle, a recording proxy, or
``collision_avoidance_b200.rvo2_compat`` on a GPU box).  Nothing in the reference is edited:
it is imported as it lies from the checkout named by ``$COLLISION_AVOIDANCE_REFERENCE``.
"""
from __future__ import annotations

import importlib
import os
import sys
import time
import time as _time_mod
import types

import numpy as np

# a checkout of the reference project (navallo/collision_avoidance); the repository does not vendor it
REFERENCE_ROOT = os.environ.get("COLLISION_AVOIDANCE_REFERENCE", "")
REGISTRY = {}          # gym.envs.registration.register(id=..., entry_point=...) calls seen


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, "collision_avoidance"))


class _Widget:
    """Tk / Canvas stand-in: every method exists, does nothing and returns 0."""

    def __init__(self, *a, **k):
        pass

    def __getattr__(self, name):
        return lambda *a, **k: 0


class Box:
    """gym.spaces.Box stand-in keeping what the env passes (collision_avoidence_env.py:52-53)."""

    def __init__(self, low, high, shape=None, dtype=np.float32):
        self.low, self.high, self.shape, self.dtype = low, high, shape, dtype


def _module(name, **attrs):
    m = types.ModuleType(name)
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m
    return m


def install(sim_cls):
    """Install the stubs and bind ``rvo2.PyRVOSimulator = sim_cls``.  Idempotent."""
    _module("tkinter", Tk=_Widget, Canvas=_Widget, LAST="last", __all__=["Tk", "Canvas", "LAST"])
    spaces = _module("gym.spaces", Box=Box)
    seeding = _module("gym.utils.seeding", np_random=lambda seed=None: (np.random.RandomState(seed), seed))
    gutils = _module("gym.utils", seeding=seeding)
    reg = _module("gym.envs.registration",
                  register=lambda id, entry_point=None, **k: REGISTRY.__setitem__(id, entry_point))
    genvs = _module("gym.envs", registration=reg)
    _module("gym", Env=type("Env", (), {}), spaces=spaces, utils=gutils, envs=genvs)
    mae = _module("ray.rllib.env.multi_agent_env", MultiAgentEnv=type("MultiAgentEnv", (), {}))
    renv = _module("ray.rllib.env", multi_agent_env=mae)
    rllib = _module("ray.rllib", env=renv)
    _module("ray", rllib=rllib)
    _module("rvo2", PyRVOSimulator=sim_cls)
    if not hasattr(time, "clock"):      # removed in Python 3.8 (SURVEY Q10)
        time.clock = time.perf_counter
    for p in (REFERENCE_ROOT, os.path.join(REFERENCE_ROOT, "collision_avoidance", "ALAN")):
        if p not in sys.path:
            sys.path.insert(0, p)


def bind_simulator(sim_cls):
    """Point the already imported reference modules at another simulator class."""
    sys.modules["rvo2"].PyRVOSimulator = sim_cls


class _QuietTime:
    """``time`` as the reference modules see it: no sleeping between frames
    (collision_avoidence_env.py:567, ALAN_true.py:699)."""
    clock = staticmethod(_time_mod.perf_counter)
    perf_counter = staticmethod(_time_mod.perf_counter)
    time = staticmethod(_time_mod.time)

    @staticmethod
    def sleep(_s):
        return None


def load_reference(sim_cls):
    """Returns (ALAN_true module, collision_avoidence_env module, Train_ALAN_action_space module)."""
    if not reference_available():
        raise RuntimeError("the reference tree is not present on this machine")
    install(sim_cls)
    alan = importlib.import_module("collision_avoidance.ALAN.ALAN_true")
    env = importlib.import_module("collision_avoidance.envs.collision_avoidence_env")
    sys.modules.setdefault("ALAN_true", alan)        # Train_ALAN_action_space.py:1 imports it flat
    train = importlib.import_module("Train_ALAN_action_space")
    for m in (alan, env):
        m.time = _QuietTime
    bind_simulator(sim_cls)
    return alan, env, train
