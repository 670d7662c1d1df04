"""Import stubs that let the UNMODIFIED reference (the original project, a checkout of which SSD_REFERENCE_ROOT names)
be imported here.

TEST INFRASTRUCTURE (oracle/).  The reference needs gym 0.21, ray 2.2 and matplotlib, none
of which this project depends on (SURVEY.md §8c).  Only the tiny surface the hot path touches is
stubbed; nothing here re-implements reference logic.  Nothing under `-m gpu`, `smoke()` or
`bench.py`'s GPU arm uses it; the tests that run the reference skip when SSD_REFERENCE_ROOT is not set.
"""
import os
import sys
import types

import numpy as np

# a checkout of the original project (its `environments/`, `contract/`, `utils/` at the top level), or None
REFERENCE_ROOT = os.environ.get("SSD_REFERENCE_ROOT") or None
# `oracle/stage_reference.py` (run by __graft_entry__.build()) copies the unmodified reference modules the path needs into
# this git-ignored directory, so that bench.py's CPU-baseline arm can time the REAL reference on a machine that has a built
# tree but no reference checkout.  Parity tests never use the staged copy.
STAGED_ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def live_reference():
    """REFERENCE_ROOT when it holds the reference tree, else None (what the parity tests run against)."""
    if REFERENCE_ROOT and os.path.isdir(os.path.join(REFERENCE_ROOT, "environments")):
        return REFERENCE_ROOT
    return None


def reference_root():
    """The reference checkout when present, else the staged copy, else None."""
    if live_reference():
        return REFERENCE_ROOT
    return STAGED_ROOT if os.path.isdir(os.path.join(STAGED_ROOT, "environments")) else None


class Space:
    def __init__(self, shape=None, dtype=None):
        self.shape = None if shape is None else tuple(shape)
        self.dtype = None if dtype is None else np.dtype(dtype)


class Box(Space):
    # gym 0.21 Box: low/high are stored as arrays of `dtype` (float32 by default) — this matters
    # for np.random.uniform(low, high) at two_stage_train.py:164 (high = float32(0.2)).
    def __init__(self, low, high, shape=None, dtype=np.float32):
        if shape is None:
            shape = np.broadcast(np.asarray(low), np.asarray(high)).shape
        super().__init__(shape, dtype)
        self.low = np.broadcast_to(np.asarray(low, dtype=dtype), self.shape).copy()
        self.high = np.broadcast_to(np.asarray(high, dtype=dtype), self.shape).copy()

    def sample(self):
        return np.random.uniform(self.low, self.high).astype(self.dtype)


class Discrete(Space):
    def __init__(self, n):
        self.n = n
        super().__init__((), np.int64)

    def sample(self):
        return int(np.random.randint(self.n))


class MultiDiscrete(Space):
    def __init__(self, nvec):
        self.nvec = np.asarray(nvec, dtype=np.int64)
        super().__init__(self.nvec.shape, np.int64)


class Dict(Space):
    def __init__(self, spaces):
        self.spaces = dict(spaces)
        super().__init__(None, None)

    def keys(self):
        return self.spaces.keys()

    def __getitem__(self, k):
        return self.spaces[k]


def _mod(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def install(root=None):
    """Put the stub modules in sys.modules and the reference root on sys.path."""
    root = root or REFERENCE_ROOT
    if not root or not os.path.isdir(root):
        raise RuntimeError("reference tree %r not present: set SSD_REFERENCE_ROOT to a checkout of the original project" % root)
    if "gym" not in sys.modules:
        spaces = _mod("gym.spaces", Space=Space, Box=Box, Discrete=Discrete,
                      MultiDiscrete=MultiDiscrete, Dict=Dict)
        _mod("gym", spaces=spaces, Env=object)
    if "ray" not in sys.modules:
        class MultiAgentEnv:  # ray.rllib.env.MultiAgentEnv: empty base class is all the path needs
            pass

        class DefaultCallbacks:
            pass

        class TaskSettableEnv:
            pass

        ray = _mod("ray")
        rllib = _mod("ray.rllib")
        env = _mod("ray.rllib.env", MultiAgentEnv=MultiAgentEnv)
        _mod("ray.rllib.env.apis")
        _mod("ray.rllib.env.apis.task_settable_env", TaskSettableEnv=TaskSettableEnv)
        _mod("ray.rllib.algorithms")
        _mod("ray.rllib.algorithms.callbacks", DefaultCallbacks=DefaultCallbacks)
        agents = _mod("ray.rllib.agents")
        agents.ppo = _mod("ray.rllib.agents.ppo", PPOTrainer=None)
        _mod("ray.rllib.utils")
        _mod("ray.rllib.utils.framework",
             try_import_tf=lambda: (None, None, None), try_import_torch=lambda: (None, None))
        _mod("ray.tune")
        _mod("ray.tune.registry", register_env=lambda name, fn: None)
        ray.rllib = rllib
        rllib.env = env
    if "matplotlib" not in sys.modules:
        plt = _mod("matplotlib.pyplot", close=lambda *a, **k: None, cla=lambda *a, **k: None,
                   imshow=lambda *a, **k: None, show=lambda *a, **k: None,
                   savefig=lambda *a, **k: None)
        _mod("matplotlib", pyplot=plt)
    if root not in sys.path:
        sys.path.insert(0, root)
