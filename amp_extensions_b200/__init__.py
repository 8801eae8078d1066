"""amp_extensions_b200 — B200-native batched learned-dynamics env step of gym-simenv / MILO.

Host-side mirror of the reference's plugin surface for this one hot path:

  DynamicsEnsemble / DynamicsModel   (reference milo/milo/dynamics.py)
  RBFLinearCost / MLPCost            (reference milo/milo/linear_cost.py)
  GAILCost (evaluation side)         (reference milo/milo/gail_cost.py)
  AmpDataset                         (reference milo/milo/datasets.py)
  SimEnv / VecSimEnv                 (reference gym-simenv/gym_simenv/envs/sim_env.py)
  ImitationReward                    (reference DeepMimicCore/scenes/SceneImitate.cpp)
  sampler.get_samples / sample_points (reference milo/milo/sampler.py, batched on the device)
  MLPBaseline / DeviceMLPBaseline     (reference mjrl/mjrl/baselines/mlp_baseline.py)
  BC / DeviceBC                       (reference mjrl/mjrl/algos/behavior_cloning.py)

All compute goes through libsimstep.so (include/simstep.h); there is no CPU fallback.
"""
__version__ = "0.1.0"

from .datasets import AmpDataset  # noqa: F401
from .dynamics import DynamicsEnsemble, DynamicsModel  # noqa: F401
from .engine import Engine, HumanoidTermination  # noqa: F401
from .linear_cost import MLPCost, RBFLinearCost  # noqa: F401
from .gail_cost import GAILCost  # noqa: F401
from .sim_env import SimEnv, VecSimEnv  # noqa: F401
from .character import Character, humanoid3d  # noqa: F401
from .imitation import ImitationReward  # noqa: F401
from .motion import MotionClip  # noqa: F401
from . import sampler  # noqa: F401
from .baseline import DeviceMLPBaseline, MLPBaseline  # noqa: F401
from .bc import BC, DeviceBC  # noqa: F401


def register_gym(env_id="simenv-v0"):
    """Register this package's SimEnv under the reference's gym id (gym-simenv/gym_simenv/__init__.py:3-6), so that
    `gym.make('simenv-v0', deepmimic_args=..., dynamic_ensemble=..., reset_args=...)` (run.py:120) builds the B200
    plugin.  gym (or gymnasium) is the caller's dependency: raises ImportError when neither is installed."""
    try:
        from gym.envs.registration import register
    except ImportError:
        from gymnasium.envs.registration import register
    register(id=env_id, entry_point="amp_extensions_b200.sim_env:SimEnv")
    return env_id
