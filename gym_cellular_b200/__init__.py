"""gym_cellular_b200 -- B200-native batched environment step for the gym-cellular environments.

Host code is Python; the hot path is hand-written CUDA for sm_100a behind a C ABI
(include/gym_cellular_b200.h, libgymcellular_b200.so) called through ctypes.  See DESIGN.md.
"""
from ._gym import gym  # noqa: F401  (real gymnasium, or the structural stand-in)
from . import tables
from .tables import right_polarizing, multiple_optima, nonlinear, nonlinear_right_polarizing
from .vector_env import CellularVectorEnv, Counts, Transitions, make_vector_env
from .packed_env import PackedCellularVectorEnv
from .plan import Plan, value_iteration
from .device_codec import encode_mixed, decode_mixed
from .codec import (generalized_cellular2tabular, generalized_tabular2cellular, cellular2tabular,
                    tabular2cellular)
from .envs import (Cells3States3Actions3Env, Cells2Rest3Env, Cells3ResetVDeadlockEnv, GridWorldEnv,
                   DebugEnv, DeepPlanningDebugEnv, DeepExplorationDebugEnv, PriorKnowledge,
                   GridWorldPriorKnowledge)
from . import registration  # noqa: F401  (registers the gym_cellular/<Name>-v0 ids)
from .alias import install_alias

__all__ = ["CellularVectorEnv", "PackedCellularVectorEnv", "Transitions", "Counts", "make_vector_env", "tables", "right_polarizing", "multiple_optima",
           "nonlinear", "nonlinear_right_polarizing", "Cells3States3Actions3Env", "Cells2Rest3Env",
           "Cells3ResetVDeadlockEnv", "GridWorldEnv", "PriorKnowledge", "GridWorldPriorKnowledge",
           "generalized_cellular2tabular", "generalized_tabular2cellular", "cellular2tabular", "tabular2cellular",
           "DebugEnv", "DeepPlanningDebugEnv", "DeepExplorationDebugEnv", "install_alias", "encode_mixed", "decode_mixed",
           "Plan", "value_iteration"]
__version__ = "0.1.0"
