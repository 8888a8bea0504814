"""Convenience re-exports, mirroring irs_lqr/all.py:5-11 of the reference."""
from .dynamical_system import *  # noqa: F401,F403
from .dynamical_system import CudaDynamicalSystem, DynamicalSystem  # noqa: F401
from .irs_lqr import (IrsLqr, IrsLqrExact, IrsLqrFirstOrder, IrsLqrParameters,  # noqa: F401
                      IrsLqrZeroOrder)
from .batched import BatchedIrsLqrZeroOrder  # noqa: F401
from .cem import CemParameters, CrossEntropyMethod  # noqa: F401
from .sampling import GaussianSampling  # noqa: F401
from .systems import (BicycleDynamics, MlpDynamics, PendulumDynamics, QuadrotorDynamics,  # noqa: F401
                      ThreeCartDynamics)
from .tv_lqr import get_solver, solve_tvlqr  # noqa: F401
from .user_system import CudaSourceDynamics  # noqa: F401
