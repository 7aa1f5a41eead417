"""B200-native batched environment engine for the environment-step hot path of
HKPolyU-UAV/ReinforcementLearningPlatform (see DESIGN.md, include/b200env.h)."""
from . import _lib  # noqa: F401
from . import compat, dist, episodes, gae, normalization, policy, rollout  # noqa: F401
from .episodes import EpisodeTracker  # noqa: F401
from .policy import GaussianPolicy  # noqa: F401
from . import ppo2  # noqa: F401
from .ppo2 import VecPPO2  # noqa: F401
from . import ppo  # noqa: F401
from .ppo import VecPPO  # noqa: F401
from . import dqn  # noqa: F401
from .dqn import VecDQN  # noqa: F401
from .compat import SingleEnv, single  # noqa: F401
from .normalization import Normalization  # noqa: F401
from .rollout import RolloutBuffer  # noqa: F401
from .vec_env import VecEnvBase  # noqa: F401
from .envs.cartpole import CartPole, CartPoleAngleOnly  # noqa: F401
from .envs.simple import (BallBalancer1D, Flight_Attitude_Simulator, FlightAttitudeSimulatorDiscrete, SecondOrderIntegration,  # noqa: F401
                          TwoLinkManipulator, UGVBidirectional, UGVForward, UGVForwardObstacleAvoidance)
from .envs.uavrobust import uav_hover, uav_hover_outer_loop, uav_inner_loop, uav_tracking_outer_loop  # noqa: F401
from .envs.uav import UavAttCtrlRL, UavPosCtrlRL, uav_param, fntsmc_param  # noqa: F401

__all__ = ["VecEnvBase", "RolloutBuffer", "EpisodeTracker", "Normalization", "GaussianPolicy", "VecPPO2", "VecPPO", "VecDQN", "SingleEnv", "single", "CartPole", "CartPoleAngleOnly", "UavAttCtrlRL", "UavPosCtrlRL", "uav_param", "fntsmc_param",
           "Flight_Attitude_Simulator", "FlightAttitudeSimulatorDiscrete", "SecondOrderIntegration", "BallBalancer1D", "TwoLinkManipulator", "UGVForward",
           "UGVBidirectional", "UGVForwardObstacleAvoidance", "uav_hover", "uav_hover_outer_loop",
           "uav_inner_loop", "uav_tracking_outer_loop"]
