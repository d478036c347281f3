"""
gym_copter_b200 -- B200-native (sm_100a CUDA) batched implementation of gym-copter's physics
and env step, behind the reference's reset/step API.  See DESIGN.md.

The compute path is libcopter_b200.so (gym_copter_b200/csrc, C ABI in include/copter_b200.h);
build it with `python -m gym_copter_b200.build`.  There is no CPU fallback.
"""

from ._lib import CopterError, CopterParams, default_params, load as load_library   # noqa: F401
from .envs import (CopterVecEnv, LanderVec, Lander3DVec, Lander2DVec, Lander1DVec,     # noqa: F401
                   Hover3DVec, Hover2DVec, Hover1DVec, TakeoffVec, Lander, Lander3D, Lander2D,
                   Lander1D, Hover3D, Hover2D, Hover1D, Takeoff, SingleEnv, make)
from .dynamics import Dynamics                                                         # noqa: F401
from .sharding import shard_range, make_sharded_env, all_reduce_stats                  # noqa: F401
from .rollout import (FusedMLPPolicy, FusedMLPValue, FusedPolicyRollout, PolicyRollout, PlanarLinear,   # noqa: F401
                      gae, mlp_policy)
from .gym_compat import register_envs, make_vector_env                                 # noqa: F401
from .export import CsvTrajectoryWriter                                                # noqa: F401

__version__ = '0.1.0'
