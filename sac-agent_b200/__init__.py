"""boatenv-b200: B200-native batched BoatEnv step path behind the reference's gym-style API.

    from sac_agent_b200 import BatchedBoatEnv, BoatEnv, ReplayBuffer, load_config

Everything that computes runs in hand-written sm_100a CUDA kernels inside
``libboatenv.so`` (C ABI: ``include/boatenv.h``).  There is no CPU fallback: importing
the env classes works anywhere, constructing one without the library or without a GPU
raises.
"""
from .config import AttrDict, load_config, params_from_config  # noqa: F401
from ._lib import BoatEnvError, lib, library_path  # noqa: F401
from .boat_env import BatchedBoatEnv, BoatEnv, Box, TERM_NAMES  # noqa: F401
from .buffer import PrioritizedReplayBuffer, ReplayBuffer  # noqa: F401
from .toy_envs import ToyCar, ToyParachute  # noqa: F401
from .csv_export import BatchedRecorder, DeviceRecorder  # noqa: F401
from .sharding import all_reduce_counters, make_sharded_env, shard_range  # noqa: F401
from .experiment import Experiment, HPTuner, get_experiment_config, info_from_counters  # noqa: F401
from . import population  # noqa: F401
from .population import AgentPopulation  # noqa: F401

__all__ = ["AttrDict", "load_config", "params_from_config", "BoatEnvError", "lib", "library_path",
           "BatchedBoatEnv", "BoatEnv", "Box", "TERM_NAMES", "PrioritizedReplayBuffer", "ReplayBuffer", "ToyCar", "ToyParachute",
           "BatchedRecorder", "DeviceRecorder", "all_reduce_counters", "make_sharded_env", "shard_range",
           "Experiment", "HPTuner", "get_experiment_config", "info_from_counters", "AgentPopulation",
           "ContinuousAgent", "SACLearner", "SAC2Learner", "OverlappedActorLearner"]


def __getattr__(name):  # the agent pulls in torch.nn / torch.optim: imported on first use only
    if name in ("ContinuousAgent", "SACLearner", "SAC2Learner", "OverlappedActorLearner"):
        from . import continuous_agent
        return getattr(continuous_agent, name)
    raise AttributeError(name)
