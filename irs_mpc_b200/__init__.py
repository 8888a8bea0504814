"""irs_mpc_b200 — B200-native implementation of the iRS-MPC smoothing + TVLQR hot path.

Host side: Python, same call surface as hjsuh94/irs_mpc (`DynamicalSystem`, `IrsLqrParameters`,
`IrsLqrExact/FirstOrder/ZeroOrder`, `solve_tvlqr`).  Device side: hand-written sm_100a CUDA in
`csrc/`, reached through the C ABI of `include/irs_mpc_b200.h` (ctypes, `_lib.py`).
"""
from . import _lib  # noqa: F401

__all__ = ["all", "dynamical_system", "irs_lqr", "sampling", "smoothing", "systems", "tv_lqr", "user_system"]
