"""ppx -- B200-native learner hot path of BoogaQ/PPO-exploration (package dir: ppo-exploration_b200/).

Import as ``import ppo_exploration_b200 as ppx`` (the root-level shim maps the hyphenated directory
name onto an importable module name).  Everything here calls hand-written sm_100a kernels through
the C ABI in include/ppx.h; there is no CPU fallback.
"""
from . import _lib
from . import logger
from .buffer import BaseBuffer, RolloutStorage, IntrinsicStorage, CountTable, discount_with_dones
from .models import Policy, RndNetwork, IntrinsicCuriosityModule, ActionConverter, ConvTrunk, ParamBank
from .util import RunningMeanStd, normalize_obs
from .algorithms import BaseAlgorithm, PPO, PPO_RND, PPO_ICM
from .evolution_strategies import EvolutionStrategy
from .spaces import Box, Discrete, SyntheticVecEnv
from .env import VecNormalize
from .classic_control import ClassicControlVecEnv, EpisodeMonitor, ToNumpy, make_env

__all__ = ["BaseBuffer", "RolloutStorage", "IntrinsicStorage", "CountTable", "discount_with_dones", "Policy",
           "RndNetwork", "IntrinsicCuriosityModule", "ActionConverter", "RunningMeanStd", "normalize_obs",
           "BaseAlgorithm", "PPO", "PPO_RND", "PPO_ICM", "EvolutionStrategy", "Box", "Discrete", "SyntheticVecEnv", "logger", "VecNormalize", "ConvTrunk", "ParamBank",
           "ClassicControlVecEnv", "EpisodeMonitor", "ToNumpy", "make_env"]
