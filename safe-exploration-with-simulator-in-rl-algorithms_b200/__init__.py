"""B200-native batched Coulom swimmer + Augmented Random Search hot path.

Reference-shaped plugin surface (drop-in names):
    SwimmerEnv                      envs/gym_swimmer/swimmer/remy_swimmer_env.py
    Environment                     ars/environment.py
    ARSAgent, EnvParam, ARSParam, Threshold, Database, Estimator, Experiment     ars/*.py
    Basic_ARS, Safe_ARS             safe_ars/ars.py
    RlglueArsExperiment             rlglue/agent/SwimmerAgent.py + rlglue/experiment/SwimmerExperiment.cpp
New batched surface: ops.step_batched / ops.rollout / ArsEngine (see include/swimmer_ars.h).
All arithmetic runs in libswimmer_ars.so (hand-written sm_100a CUDA); there is no CPU fallback.
"""
from . import _lib, ops  # noqa: F401
from ._lib import (ARS_AGENT, ARS_RLGLUE, ARS_TOPB, DELTA_01, DELTA_PM1, GYM, KERNEL_AUTO, KERNEL_LANES,  # noqa: F401
                   KERNEL_LANES2, KERNEL_LANES3, KERNEL_THREAD, RLGLUE, SwimmerLibError, build_library, make_params)
from .ars_agent import ARSAgent  # noqa: F401
from .database import Database, pick_sub_database  # noqa: F401
from .engine import ArsEngine  # noqa: F401
from .environment import Environment  # noqa: F401
from .estimator import Estimator  # noqa: F401
from .experiment import Experiment, SeedFanout  # noqa: F401
from .parameters import ARSParam, EnvParam, Threshold  # noqa: F401
from .rlglue_agent import RlglueArsExperiment, read_parameters  # noqa: F401
from .safe_ars import Basic_ARS, MaxAffineCost, Safe_ARS, builtin_cost  # noqa: F401
from .swimmer_env import SwimmerEnv  # noqa: F401

__version__ = "0.1.0"

# gym registration id of the reference (envs/gym_swimmer/register.py:5-11)
GYM_ID = "LeonSwimmer-v0"
GYM_KWARGS = {"direction": [1., 0.], "n": 5, "max_u": 5., "l_i": 1., "k": 10., "m_i": 1., "h": 0.001}


def make(env_id=GYM_ID, **overrides):
    """gym.make-style constructor for the registered id (register.py: n=5, max_episode_steps=1000)."""
    if env_id != GYM_ID:
        raise ValueError("unknown environment id %r" % (env_id,))
    kw = dict(GYM_KWARGS)
    kw.update(overrides)
    return SwimmerEnv(envName=env_id, **kw)
