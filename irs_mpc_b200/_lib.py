"""ctypes binding of the C ABI in include/irs_mpc_b200.h (libirs_mpc_b200.so, built in-tree).

There is deliberately no fallback: if the shared library is missing or CUDA is unavailable the
product path raises instead of computing anything on the CPU.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("IRS_MPC_B200_LIB") or os.path.join(_HERE, "libirs_mpc_b200.so")   # env: tuning builds
CSRC = os.path.join(_HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(_HERE), "include")

ABI_VERSION = 4      # IRS_ABI_VERSION of include/irs_mpc_b200.h this binding was written against

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]


def sources():
    return [os.path.join(CSRC, "api.cu")]


def _stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "irs_mpc_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile the CUDA library for sm_100a with nvcc (cross-compiles without a GPU)."""
    if not force and not _stale():
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + ["-I", INCLUDE, "-o", LIB_PATH] + sources()
    if verbose:
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)
    return LIB_PATH


_c_double_p = ctypes.POINTER(ctypes.c_double)
_vp = ctypes.c_void_p
_ll = ctypes.c_longlong
_ull = ctypes.c_ulonglong
_i = ctypes.c_int
_u = ctypes.c_uint

# name -> argtypes (restype is int unless listed in _RESTYPES); mirrors include/irs_mpc_b200.h
SIGNATURES = {
    "irs_abi_version": [],
    "irs_last_error": [],
    "irs_set_gram_engine": [_i],
    "irs_system_dims": [_i, ctypes.POINTER(_i), ctypes.POINTER(_i), ctypes.POINTER(_i)],
    "irs_partial_width": [_i, _i],
    "irs_smooth_plan": [_i, _i, _i, _ll, _ll, ctypes.POINTER(_i), ctypes.POINTER(_ll)],
    "irs_smooth_zero_order_accumulate": [_i, _c_double_p, _i, _i, _vp, _vp, _i, _ll, _vp, _vp,
                                         _ull, _u, _u, _u, _ull, _i, _ll, _vp, _vp],
    "irs_smooth_first_order_accumulate": [_i, _c_double_p, _i, _i, _vp, _vp, _i, _ll, _vp, _vp,
                                          _ull, _u, _u, _u, _ull, _i, _ll, _vp, _vp],
    "irs_smooth_reduce_chunks": [_i, _i, _vp, _i, _i, _vp, _vp],
    "irs_smooth_finalize_peer": [_i, _c_double_p, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _ll, _i,
                                 _i, _i, ctypes.c_double, ctypes.c_double, _i, _vp, _vp, _vp, _vp, _vp],
    "irs_smooth_finalize_peer_capacity": [_i, _i, ctypes.POINTER(_i)],
    "irs_smooth_finalize_gather": [_i, _c_double_p, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _ll, _i, _i,
                                   _i, _i, ctypes.c_double, ctypes.c_double, _i, _vp, _vp],
    "irs_smooth_finalize": [_i, _c_double_p, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _i, _ll,
                            ctypes.c_double, _i, _vp, _vp, _vp, _vp, _vp],
    "irs_exact_linearize": [_i, _c_double_p, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp],
    "irs_philox_dump": [_i, _ll, _i, _vp, _ull, _u, _u, _u, _ull, _i, _vp, _vp, _vp],
    "irs_dynamics_batch_f32": [_i, _c_double_p, _i, _i, _vp, _vp, _vp, _ll, _vp],
    "irs_dynamics_batch_f64": [_i, _c_double_p, _i, _i, _vp, _vp, _vp, _ll, _vp],
    "irs_jacobian_xu_batch_f32": [_i, _c_double_p, _i, _vp, _vp, _vp, _ll, _vp],
    "irs_jacobian_xu_batch_f64": [_i, _c_double_p, _i, _vp, _vp, _vp, _ll, _vp],
    "irs_project_batch_f64": [_i, _c_double_p, _i, _vp, _ll, _vp],
    "irs_tvlqr_riccati": [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _i, _i, _vp, _vp, _vp, _vp],
    "irs_tvlqr_riccati_segment": [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "irs_tvlqr_riccati_ex": [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp],
    "irs_mlp_register": [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "irs_mlp_release": [_i],
    "irs_user_arrays_register": [_vp, _ll, ctypes.POINTER(_i)],
    "irs_user_arrays_update": [_i, _ll, _vp, _ll, _vp],
    "irs_user_arrays_release": [_i],
    "irs_cem_refit": [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp],
    "irs_gram_block_f64": [_i, _i, _vp, _vp, _ll, _vp, _vp],
    "irs_tvlqr_plan_rows": [_i, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp],
    "irs_tvlqr_plan_check": [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, ctypes.c_double, _i, _i, _i,
                             _vp, _vp, _vp],
    "irs_tvlqr_box_solve": [_i, _c_double_p, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _vp, _vp,
                            _vp, _vp, _vp, _vp, _ll, _ll, _vp, _vp, _vp, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                            _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp],
    "irs_tvlqr_linear_rollout": [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp],
    "irs_tvlqr_any_limits": [ctypes.POINTER(_i), ctypes.POINTER(_i)],
    "irs_tvlqr_riccati_any": [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp],
    "irs_tvlqr_linear_rollout_any": [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp],
    "irs_tvlqr_box_qp_any": [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _vp, _vp, _vp, _vp, _vp,
                             _vp, _ll, _ll, _vp, ctypes.c_double, ctypes.c_double, _i, _i, _i, _vp, _vp, _vp, _vp,
                             _vp],
    "irs_rollout_closed_loop": [_i, _c_double_p, _i, _vp, _vp, _vp, _vp, _ll, _vp, _vp, _i, _i,
                                _vp, _vp, _vp, _vp],
    "irs_rollout_open_loop": [_i, _c_double_p, _i, _vp, _vp, _vp, _ll, _vp, _vp, _i, _i,
                              _vp, _vp, _vp],
    "irs_fp32_fma_peak": [_i, _vp, _ll, _c_double_p, _vp],
    "irs_evaluate_cost": [_i, _i, _vp, _vp, _vp, _ll, _vp, _vp, _i, _i, _vp, _vp],
    "irs_graph_begin": [_vp],
    "irs_graph_end": [_vp, ctypes.POINTER(_vp)],
    "irs_graph_update_smoothing": [_vp, _vp, _ull, _u, _u],
    "irs_graph_launch": [_vp, _vp],
    "irs_graph_destroy": [_vp],
}
_RESTYPES = {"irs_last_error": ctypes.c_char_p}


class IrsCudaError(RuntimeError):
    pass


class Library:
    """One build of the C ABI: the main library, or the library of a user-written system
    (user_system.py), which exports the same entry points.  Loaded on first use."""

    _by_path = {}

    def __init__(self, path):
        self.path = path
        self._handle = None

    @classmethod
    def at(cls, path):
        """The one Library object of `path` (one dlopen per library and process)."""
        path = os.path.abspath(path)
        if path not in cls._by_path:
            cls._by_path[path] = cls(path)
        return cls._by_path[path]

    def handle(self):
        """Load (once) and return the ctypes handle.  Raises if the library has not been built."""
        if self._handle is None:
            if not os.path.exists(self.path):
                raise ImportError(
                    "irs_mpc_b200: %s not found. Build it with `python -c 'import __graft_entry__ as g; "
                    "g.build()'` (needs nvcc). There is no CPU fallback." % self.path)
            handle = ctypes.CDLL(self.path)
            for name, argtypes in SIGNATURES.items():
                fn = getattr(handle, name)
                fn.argtypes = argtypes
                fn.restype = _RESTYPES.get(name, ctypes.c_int)
            if handle.irs_abi_version() != ABI_VERSION:
                raise ImportError("irs_mpc_b200: ABI version mismatch in %s" % self.path)
            self._handle = handle
        return self._handle

    def call(self, name, *args):
        """Invoke an entry point; translate a non-zero status into IrsCudaError(message)."""
        handle = self.handle()
        rc = getattr(handle, name)(*args)
        if rc != 0:
            raise IrsCudaError("%s failed: %s" % (name, handle.irs_last_error().decode()))
        return rc


MAIN = Library.at(LIB_PATH)


def lib():
    """Load (once) and return the ctypes handle of the main library."""
    return MAIN.handle()


def call(name, *args):
    """Invoke an entry point of the main library."""
    return MAIN.call(name, *args)


def params_array(values):
    arr = (ctypes.c_double * len(values))(*[float(v) for v in values])
    return arr, len(values)
