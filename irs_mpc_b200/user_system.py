"""User-written dynamics: a DynamicalSystem given as CUDA C++ source, compiled for sm_100a on first use.

    sys = CudaSourceDynamics(
        dim_x=4, dim_u=1, h=0.02, params=[1.0, 0.1, 0.5, 9.81],
        step='''
            R s, c; Math<R>::sincos(x[1], s, c);
            ...
            o[0] = x[0] + h * x[2];  ...
        ''',
        jacobian=None,      # optional: a body writing J[N*D], row-major, columns [x | u]
        autodiff=False,     # or True: the Jacobian of the step body by forward-mode dual numbers
        arrays=None,        # optional: {name: array} read by the bodies from device memory
        name="cartpole")

The bodies are C++ over the scalar type R, instantiated as float (the sample work of the smoothing kernels)
and as double (rollouts, fits, exact linearization).  They see the inputs `x[N]`, `u[M]`, the output `o[N]`
(or `J[N*D]`), the step `h`, the parameters `p[0..]` (already in R), the dimensions N, M, D and `Math<R>`
(sincos, rcp, div: fast intrinsics in float, libdevice in double).

The library wraps them in a functor with the interface of the built-in systems (csrc/systems.cuh) and compiles
csrc/api.cu once more around it, with IRS_USER_SYSTEM defined: a shared library of its own that exports the same
C ABI, in which the user system has id 5 (kUser).  Every kernel of the hot path — sampling and Gram
accumulation, fits, Riccati, rollouts, the bounded descent — is then the one the built-in systems run.  The
library is cached under a hash of everything it is built from (IRS_USER_CACHE, default: _user_cache/ next to
this file); constructing the same system again loads it without compiling.

autodiff=True derives the Jacobian from the step body alone (no jacobian body; giving both is a ValueError).  The
body is then also evaluated over irs::ad::Dual<R, K> (csrc/dual.cuh): a value and K tangent lanes, packed FP32
pairs in float.  jac_var seeds unit tangents on K consecutive columns of [x | u] per pass, P = ceil(D / 8) passes
of K = ceil(D / P), and reads J off the tangents of o.  In such a body R is the dual type where it is
differentiated, while h and p[] stay plain float / double.  Supported: construction from int, float, double and R;
unary -; + - * / and += -= *= /= with R or a number on either side; comparisons (on the values); Math<R>::sincos /
rcp / div (the values are Math<float>'s fast intrinsics or Math<double>'s); sqrt, exp, log, sin, cos, tan, asin,
acos, atan, atan2, sinh, cosh, tanh, fabs, fmin, fmax, and pow with a constant exponent.  There is no conversion
back to float, double or int: a body that drops the derivative (`float t = x[0];`) does not compile.  At kinks:
branches follow the values; fabs at 0 takes the + branch; fmin / fmax take the derivative of the argument they
select, the first one on a tie; sqrt at 0 gives the infinite derivative that math gives.  The Jacobian is checked
against central differences at construction, as a hand-written body is.

arrays={name: values} gives the bodies read-only arrays in device memory: matrices, lookup tables, network weights.
Each is real, finite and non-empty with 1 to 3 dimensions; all of them together hold at most 2^24 elements
(MAX_ARRAY_ELEMENTS).  In a body, `name[i]` reads it flat (row-major), `name(i, j)` and `name(i, j, k)` by
dimension, and `name_n0`, `name_n1`, `name_n2` are its extents (1 for a missing dimension) as compile-time
constants.  Elements are in the base type, like h and p[]: float in the fp32 sample kernels, double elsewhere; they
carry no tangents under autodiff.  An element is returned by value, so writing to an array does not compile.
Only the names and shapes enter the generated source: systems that differ in array values share one library,
and `set_array(name, values)` replaces one array's values (same shape) in place, without recompiling and without
re-capturing a CUDA graph.  Names must be C identifiers that are neither C++ keywords nor names a body already
sees (RESERVED_NAMES), and must not start with `irs` or `__`.
"""
import ctypes
import functools
import hashlib
import os
import re
import shutil
import subprocess
import tempfile
import time

import numpy as np

from . import _device, _lib
from .dynamical_system import CudaDynamicalSystem

USER_SYSTEM_ID = 5
MAX_REGRESSORS = 16         # kMaxRegressors (csrc/smooth.cuh): n + m
MAX_PARAMS = 9              # SysParams::v[10] (csrc/common.cuh) holds h and nine more
BUILTIN_PAIRS = ((2, 1), (5, 2), (12, 4), (6, 2))      # (n, m) with compile-time LQR kernels (api.cu)
AUTODIFF_MAX_LANES = 8      # tangent lanes of one forward-mode pass (DESIGN.md 3.10.1)
MAX_ARRAY_ELEMENTS = 1 << 24        # IRS_USER_ARRAYS_MAX_ELEMS (include/irs_mpc_b200.h): int indices in a body
# names a body already sees, the generated functor's members, and the math functions a body calls: an array
# of such a name would shadow them
RESERVED_NAMES = frozenset("""
    x u o J h p R B N M D Math
    NJ Rebind kHasJacobian kTrigAhead kHasProjection kPasses kLanes BATCH DR
    step eval jac_var jac_assemble project UserStep UserSystem SysParams ArrayView prm user_arrays ad irs std
    sqrt exp log sin cos tan asin acos atan atan2 sinh cosh tanh fabs fmin fmax pow floor ceil round trunc
    fmod abs min max sincos rcp div
""".split())
CPP_KEYWORDS = frozenset("""
    alignas alignof and and_eq asm auto bitand bitor bool break case catch char char8_t char16_t char32_t class
    compl concept const consteval constexpr constinit const_cast continue co_await co_return co_yield decltype
    default delete do double dynamic_cast else enum explicit export extern false float for friend goto if inline
    int long mutable namespace new noexcept not not_eq nullptr operator or or_eq private protected public
    register reinterpret_cast requires return short signed sizeof static static_assert static_cast struct switch
    template this thread_local throw true try typedef typeid typename union unsigned using virtual void volatile
    wchar_t while xor xor_eq
""".split())
_IDENTIFIER = re.compile(r"[A-Za-z_][A-Za-z0-9_]*\Z")


def _check_array(name, values):
    """values as a C-contiguous float64 array; ValueError naming the array unless real, finite, non-empty and
    of 1 to 3 dimensions."""
    try:
        a = np.asarray(values)
        if np.iscomplexobj(a):
            raise TypeError("complex")
        a = np.asarray(a, dtype=np.float64)
    except (TypeError, ValueError):
        raise ValueError("array %r must hold real numbers" % (name,)) from None
    if not 1 <= a.ndim <= 3:
        raise ValueError("array %r has %d dimensions; arrays have 1 to 3" % (name, a.ndim))
    a = np.ascontiguousarray(a)
    if a.size == 0:
        raise ValueError("array %r is empty" % (name,))
    if not np.all(np.isfinite(a)):
        raise ValueError("array %r holds a value that is not finite" % (name,))
    return a


def check_arrays(arrays):
    """The arrays of a user system, validated -> [(name, float64 array)] in the mapping's order (see the module
    docstring for the rules).  Every violation is a ValueError naming the array."""
    if arrays is None:
        return []
    if not hasattr(arrays, "items"):
        raise ValueError("arrays must be a mapping from name to array, got %s" % type(arrays).__name__)
    out, total = [], 0
    for name, values in arrays.items():
        if not isinstance(name, str) or not _IDENTIFIER.match(name):
            raise ValueError("array name %r is not a C identifier" % (name,))
        if name in RESERVED_NAMES or name in CPP_KEYWORDS:
            raise ValueError("array name %r is taken: a body already sees that name" % name)
        if name.startswith("irs") or name.startswith("__"):
            raise ValueError("array name %r starts with a reserved prefix (irs, __)" % name)
        out.append((name, _check_array(name, values)))
        total += out[-1][1].size
        if total > MAX_ARRAY_ELEMENTS:
            raise ValueError("array %r brings the arrays to %d elements, more than the limit of %d"
                             % (name, total, MAX_ARRAY_ELEMENTS))
    extents = {"%s_n%d" % (name, k) for name, _ in out for k in range(3)}
    for name, _ in out:
        if name in extents:
            raise ValueError("array name %r is the name of another array's extent" % name)
    return out


def _array_lines(arrays, scalar="R"):
    """Members of the functor for checked arrays: extents, then one view per array into the copy in `scalar`."""
    lines = []
    for name, a in arrays:
        n0, n1, n2 = tuple(a.shape) + (1,) * (3 - a.ndim)
        lines.append("    static constexpr int %s_n0 = %d, %s_n1 = %d, %s_n2 = %d;" % (name, n0, name, n1, name, n2))
        lines.append("    ArrayView<%s, %d, %d, %d, %d> %s;" % (scalar, a.ndim, n0, n1, n2, name))
    return lines


def _array_init_lines(arrays, prefix):
    lines, off = [], 0
    for name, a in arrays:
        lines.append("        %s%s.data = user_arrays<R>(sp) + %d;" % (prefix, name, off))
        off += a.size
    return lines


def cache_dir():
    return os.environ.get("IRS_USER_CACHE") or os.path.join(_lib._HERE, "_user_cache")


def _nvcc():
    return os.environ.get("NVCC", "nvcc")


@functools.lru_cache(maxsize=None)
def _nvcc_version(nvcc):
    """`nvcc --version`, or None when there is no such compiler."""
    if shutil.which(nvcc) is None:
        return None
    out = subprocess.run([nvcc, "--version"], capture_output=True, text=True)
    return out.stdout if out.returncode == 0 else None


def _build_inputs_digest():
    """Hash of every file the user library is compiled from besides the generated source, and the flags."""
    h = hashlib.sha256()
    for f in sorted(os.listdir(_lib.CSRC)):
        h.update(f.encode())
        with open(os.path.join(_lib.CSRC, f), "rb") as fh:
            h.update(fh.read())
    with open(os.path.join(_lib.INCLUDE, "irs_mpc_b200.h"), "rb") as fh:
        h.update(fh.read())
    h.update(" ".join(_lib.NVCC_FLAGS).encode())
    return h.hexdigest()


def autodiff_passes(d):
    """(P, K) of a forward-mode Jacobian over d columns: P passes of K tangent lanes, K at most 8."""
    p = -(-d // AUTODIFF_MAX_LANES)
    return p, -(-d // p)


def _array_defines(arrays, nparams):
    """The defines of a unit with arrays: the handle is one more parameter after h and p[]."""
    if not arrays:
        return ["#define IRS_USER_NPARAMS %d" % nparams]
    return ["#define IRS_USER_NPARAMS %d" % (nparams + 1),
            "#define IRS_USER_ARRAYS 1",
            "#define IRS_USER_ARRAY_ELEMS %d" % sum(a.size for _, a in arrays)]


def generate_source(dim_x, dim_u, nparams, step, jacobian=None, autodiff=False, arrays=None):
    """The translation unit of a user library: the functor around the bodies, then csrc/api.cu.
    nparams counts h.  #line directives make the compiler's diagnostics point into the bodies.  arrays: the
    mapping of CudaSourceDynamics; only names and shapes enter the source (the handle of the array set follows
    the scalar parameters)."""
    arrays = check_arrays(arrays)
    if autodiff:
        return _generate_autodiff_source(dim_x, dim_u, nparams, step, arrays)
    n, m = dim_x, dim_u
    d = n + m
    lines = [
        "// generated by irs_mpc_b200/user_system.py: a user-written system around csrc/api.cu",
        "#define IRS_USER_SYSTEM 1",
        "#define IRS_USER_N %d" % n,
        "#define IRS_USER_M %d" % m,
    ] + _array_defines(arrays, nparams) + [
        '#include "systems.cuh"',
    ] + (['#include "user_arrays.cuh"'] if arrays else []) + [
        "",
        "namespace irs {",
        "template <typename R>",
        "struct UserSystem {",
        "    template <typename S> using Rebind = UserSystem<S>;",
        "    static constexpr int N = %d, M = %d, D = %d, NJ = %d;" % (n, m, d, n * d),
        "    static constexpr bool kHasJacobian = %s;" % ("true" if jacobian is not None else "false"),
        "    static constexpr int kTrigAhead = 0;",
        "    static constexpr bool kHasProjection = false;",
        "    R h;",
        "    R p[%d];" % max(1, nparams - 1),
    ] + _array_lines(arrays) + [
        "    __device__ explicit UserSystem(const SysParams& sp) : h(prm<R>(sp, 0)) {",
        "#pragma unroll",
        "        for (int i = 0; i < %d; ++i) p[i] = i + 1 < %d ? prm<R>(sp, i + 1) : R(0);" % (max(1, nparams - 1), nparams),
    ] + _array_init_lines(arrays, "") + [
        "    }",
        "    template <bool BATCH>",
        "    __device__ __forceinline__ void step(const R* x, const R* u, R* o) const {",
    ]

    def body(text, label):
        lines.append('#line 1 "%s"' % label)
        lines.extend(text.splitlines() or [""])
        lines.append('#line %d "user_system.cu"' % (len(lines) + 2))

    body(step, "step")
    lines += ["    }",
              "    // the whole Jacobian varies: jac_var writes it, jac_assemble copies it",
              "    __device__ __forceinline__ void jac_var(const R* x, const R* u, R* J) const {"]
    if jacobian is not None:
        body(jacobian, "jacobian")
    lines += ["    }",
              "    __device__ __forceinline__ void jac_assemble(const R* v, R* J) const {",
              "#pragma unroll",
              "        for (int i = 0; i < N * D; ++i) J[i] = v[i];",
              "    }",
              "    __device__ __forceinline__ void project(R*) const {}",
              "};",
              "}  // namespace irs",
              "",
              '#include "api.cu"',
              ""]
    return "\n".join(lines)


def _generate_autodiff_source(dim_x, dim_u, nparams, step, arrays):
    """generate_source with autodiff: the step body is written once, in UserStep<B>::eval over any scalar type
    R, and UserSystem<B> derives from UserStep<B>.  step<BATCH> evaluates it over B; jac_var evaluates step<false>
    over irs::ad::Dual<B, K> in P passes, each seeding unit tangents on K consecutive columns of [x | u]."""
    n, m = dim_x, dim_u
    d = n + m
    np_ = max(1, nparams - 1)
    passes, lanes = autodiff_passes(d)
    lines = [
        "// generated by irs_mpc_b200/user_system.py: a user-written system around csrc/api.cu, its Jacobian by",
        "// forward-mode dual numbers (csrc/dual.cuh)",
        "#define IRS_USER_SYSTEM 1",
        "#define IRS_USER_AUTODIFF 1",
        "#define IRS_USER_N %d" % n,
        "#define IRS_USER_M %d" % m,
    ] + _array_defines(arrays, nparams) + [
        '#include "systems.cuh"',
        '#include "dual.cuh"',
    ] + (['#include "user_arrays.cuh"'] if arrays else []) + [
        "",
        "namespace irs {",
        "// the step body over any scalar R; h and p[] stay in the base type B (parameters carry no tangents)",
        "template <typename B>",
        "struct UserStep {",
        "    static constexpr int N = %d, M = %d, D = %d;" % (n, m, d),
        "    B h;",
        "    B p[%d];" % np_,
    ] + _array_lines(arrays, "B") + [
        "    template <bool BATCH, typename R>",
        "    __device__ __forceinline__ void eval(const R* x, const R* u, R* o) const {",
    ]
    lines.append('#line 1 "step"')
    lines.extend(step.splitlines() or [""])
    lines.append('#line %d "user_system.cu"' % (len(lines) + 2))
    lines += [
        "    }",
        "};",
        "",
        "template <typename R>",
        "struct UserSystem : UserStep<R> {",
        "    template <typename S> using Rebind = UserSystem<S>;",
        "    static constexpr int N = %d, M = %d, D = %d, NJ = %d;" % (n, m, d, n * d),
        "    static constexpr bool kHasJacobian = true;",
        "    static constexpr int kTrigAhead = 0;",
        "    static constexpr bool kHasProjection = false;",
        "    // jac_var: P passes of K tangent lanes (P = ceil(D / 8), K = ceil(D / P))",
        "    static constexpr int kPasses = %d, kLanes = %d;" % (passes, lanes),
        "    __device__ explicit UserSystem(const SysParams& sp) {",
        "        this->h = prm<R>(sp, 0);",
        "#pragma unroll",
        "        for (int i = 0; i < %d; ++i) this->p[i] = i + 1 < %d ? prm<R>(sp, i + 1) : R(0);" % (np_, nparams),
    ] + _array_init_lines(arrays, "this->") + [
        "    }",
        "    template <bool BATCH>",
        "    __device__ __forceinline__ void step(const R* x, const R* u, R* o) const {",
        "        this->template eval<BATCH, R>(x, u, o);",
        "    }",
        "    // the whole Jacobian of step<false> varies: jac_var writes it, jac_assemble copies it",
        "    __device__ __forceinline__ void jac_var(const R* x, const R* u, R* J) const {",
        "        using DR = ad::Dual<R, kLanes>;",
        "#pragma unroll",
        "        for (int pass = 0; pass < kPasses; ++pass) {",
        "            const int c0 = pass * kLanes;",
        "            DR xd[N], ud[M], od[N];",
        "#pragma unroll",
        "            for (int q = 0; q < N; ++q) xd[q] = DR::seed(x[q], q - c0);",
        "#pragma unroll",
        "            for (int q = 0; q < M; ++q) ud[q] = DR::seed(u[q], N + q - c0);",
        "            this->template eval<false, DR>(xd, ud, od);",
        "#pragma unroll",
        "            for (int i = 0; i < N; ++i)",
        "#pragma unroll",
        "                for (int k = 0; k < kLanes; ++k)",
        "                    if (c0 + k < D) J[i * D + c0 + k] = od[i].tangent(k);",
        "        }",
        "    }",
        "    __device__ __forceinline__ void jac_assemble(const R* v, R* J) const {",
        "#pragma unroll",
        "        for (int i = 0; i < N * D; ++i) J[i] = v[i];",
        "    }",
        "    __device__ __forceinline__ void project(R*) const {}",
        "};",
        "}  // namespace irs",
        "",
        '#include "api.cu"',
        "",
    ]
    return "\n".join(lines)


def _compile(src_path, out_path):
    """nvcc with the main library's flags; RuntimeError with the compiler's diagnostics on failure."""
    cmd = [_nvcc()] + _lib.NVCC_FLAGS + ["-I", _lib.INCLUDE, "-I", _lib.CSRC, "-o", out_path, src_path]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("compiling the user system failed:\n" + (res.stderr or res.stdout))


def build_library(dim_x, dim_u, nparams, step, jacobian=None, name="user", autodiff=False, arrays=None):
    """Compile (or find in the cache) the library of one user system -> (path, seconds spent compiling,
    source hash).  seconds is 0.0 on a cache hit.  autodiff: derive the Jacobian from the step body.
    arrays: {name: values}; only the names and shapes select the library."""
    if autodiff and jacobian is not None:
        raise ValueError("give a jacobian body or autodiff=True, not both")
    src = generate_source(dim_x, dim_u, nparams, step, jacobian, autodiff, arrays)
    src_digest = hashlib.sha256((src + _build_inputs_digest()).encode()).hexdigest()[:24]
    tag = re.sub(r"[^A-Za-z0-9_]", "_", str(name))[:40] or "user"
    root = cache_dir()
    version = _nvcc_version(_nvcc())
    if version is None:
        # no compiler: a library built from the same sources by any compiler version will do
        found = sorted(f for f in (os.listdir(root) if os.path.isdir(root) else [])
                       if f.startswith("lib%s_%s_" % (tag, src_digest)) and f.endswith(".so"))
        if not found:
            raise RuntimeError("no CUDA compiler found (set $NVCC or put nvcc on PATH) and no cached library "
                               "for user system %r in %s; there is no fallback" % (name, root))
        return os.path.join(root, found[-1]), 0.0, src_digest
    ver_digest = hashlib.sha256(version.encode()).hexdigest()[:8]
    path = os.path.join(root, "lib%s_%s_%s.so" % (tag, src_digest, ver_digest))
    if os.path.exists(path):
        return path, 0.0, src_digest
    os.makedirs(root, exist_ok=True)
    t0 = time.perf_counter()
    with tempfile.TemporaryDirectory(dir=root) as tmp:
        cu = os.path.join(tmp, "user_system.cu")
        with open(cu, "w") as fh:
            fh.write(src)
        out = os.path.join(tmp, "lib.so")
        _compile(cu, out)
        os.replace(out, path)       # atomic: a concurrent build of the same system writes the same bytes
    return path, time.perf_counter() - t0, src_digest


class CudaSourceDynamics(CudaDynamicalSystem):
    """A DynamicalSystem whose dynamics are CUDA C++ source (see the module docstring).

    dim_x, dim_u: N and M, with N + M <= 16.  h: the step, visible as `h`.  params: at most nine further
    finite numbers, visible as p[0..]; `self.params` may be changed later (same count), which re-captures
    the solvers' CUDA graphs.  step: body computing o = f(x, u).  jacobian: optional body writing
    J = d f / d(x, u) [N x (N+M)] row-major.  autodiff: derive J from the step body by forward-mode dual
    numbers instead (not together with jacobian).  Either Jacobian is checked against central differences of
    the fp64 step at a few seeded points (this needs the GPU) and a mismatch is refused.  Without one, the
    Jacobian methods, IrsLqrFirstOrder and IrsLqrExact raise NotImplementedError.  arrays: {name: values} the
    bodies read from device memory (module docstring), registered on the current device; set_array replaces
    one array's values.  Changing the source, or an array's shape, means a new object."""

    system_id = USER_SYSTEM_ID
    _array_handle = -1

    def __init__(self, dim_x, dim_u, h, params=(), step=None, jacobian=None, autodiff=False, name="user",
                 arrays=None):
        super().__init__()
        if int(dim_x) != dim_x or int(dim_u) != dim_u or dim_x < 1 or dim_u < 1:
            raise ValueError("dim_x and dim_u must be positive integers, got %r and %r" % (dim_x, dim_u))
        dim_x, dim_u = int(dim_x), int(dim_u)
        if dim_x + dim_u > MAX_REGRESSORS:
            raise ValueError("dim_x + dim_u = %d exceeds the limit of %d regressors (kMaxRegressors)"
                             % (dim_x + dim_u, MAX_REGRESSORS))
        params = [float(v) for v in params]
        if len(params) > MAX_PARAMS:
            raise ValueError("%d parameters given: at most %d besides h fit the kernels' parameter block"
                             % (len(params), MAX_PARAMS))
        if not np.all(np.isfinite([float(h)] + params)):
            raise ValueError("h and the parameters must be finite")
        if not isinstance(step, str) or not step.strip():
            raise ValueError("step must be the C++ body of the dynamics")
        if jacobian is not None and (not isinstance(jacobian, str) or not jacobian.strip()):
            raise ValueError("jacobian must be a C++ body or None")
        arrays = check_arrays(arrays)
        self.h = float(h)
        self.dim_x, self.dim_u = dim_x, dim_u
        self.params = params
        self.system_name = str(name)
        self.autodiff = bool(autodiff)
        self.has_jacobian = jacobian is not None or self.autodiff
        self.riccati_segments = (dim_x, dim_u) in BUILTIN_PAIRS
        self._nparams = 1 + len(params)
        path, self.build_seconds, self.source_hash = build_library(dim_x, dim_u, self._nparams, step, jacobian,
                                                                   name, self.autodiff, dict(arrays))
        self.cache_hit = self.build_seconds == 0.0
        self.library_path = path
        self.lib = _lib.Library.at(path)
        n, m = ctypes.c_int(), ctypes.c_int()
        self.lib.call("irs_system_dims", USER_SYSTEM_ID, ctypes.byref(n), ctypes.byref(m), None)
        if (n.value, m.value) != (dim_x, dim_u):
            raise RuntimeError("library %s holds a (%d, %d) system, expected (%d, %d)"
                               % (path, n.value, m.value, dim_x, dim_u))
        # name -> (offset of its first element in the array set, current values)
        self._arrays, offset = {}, 0
        for aname, a in arrays:
            self._arrays[aname] = (offset, a)
            offset += a.size
        if arrays:
            _device.require_cuda()
            handle = ctypes.c_int(-1)
            flat = np.concatenate([a.ravel() for _, a in arrays])
            self.lib.call("irs_user_arrays_register", flat.ctypes.data, flat.size, ctypes.byref(handle))
            self._array_handle = handle.value
        if self.has_jacobian:
            self._check_jacobian()

    @property
    def system_key(self):
        return (USER_SYSTEM_ID, self.source_hash)

    def device_params(self):
        if len(self.params) != self._nparams - 1:
            raise ValueError("system %r was built with %d parameters, now has %d"
                             % (self.system_name, self._nparams - 1, len(self.params)))
        prm = [self.h] + [float(v) for v in self.params]
        if self._arrays:
            prm.append(float(self._array_handle))     # in the graph keys: systems with other values never share
        return prm

    @property
    def arrays(self):
        """{name: a read-only view of the current values (float64)}."""
        out = {}
        for name, (_, a) in self._arrays.items():
            v = a.view()
            v.flags.writeable = False
            out[name] = v
        return out

    def set_array(self, name, values):
        """Replace the values of array `name` (same shape).  The copy is ordered on the current stream: the next
        call sees the new values, eager or replayed from a CUDA graph; nothing recompiles or re-captures."""
        if name not in self._arrays:
            raise ValueError("system %r has no array %r (it has %s)" % (self.system_name, name, sorted(self._arrays)))
        offset, old = self._arrays[name]
        a = _check_array(name, values)
        if a.shape != old.shape:
            raise ValueError("array %r has shape %s, got values of shape %s" % (name, old.shape, a.shape))
        self.lib.call("irs_user_arrays_update", self._array_handle, offset, a.ctypes.data, a.size,
                      _device.stream_ptr())
        self._arrays[name] = (offset, a)

    def __del__(self):
        try:
            if self._array_handle >= 0:
                self.lib.call("irs_user_arrays_release", self._array_handle)
        except Exception:      # interpreter shutdown: the library may be gone already
            pass

    def jacobian_xu_batch(self, x, u, *args, **kw):
        if not self.has_jacobian:
            raise NotImplementedError("user system %r was built without a Jacobian body or autodiff=True"
                                      % self.system_name)
        return super().jacobian_xu_batch(x, u, *args, **kw)

    def jacobian_xu(self, x, u):
        return self.jacobian_xu_batch(np.asarray(x)[None, :], np.asarray(u)[None, :])[0]

    def _check_jacobian(self, points=4, seed=0):
        """Refuse a Jacobian (a body, or the dual-number derivative) that disagrees with central differences of
        the fp64 step."""
        n, m = self.dim_x, self.dim_u
        d = n + m
        rng = np.random.default_rng(seed)
        xu = 0.5 * rng.standard_normal((points, d))
        J = self.jacobian_xu_batch(xu[:, :n], xu[:, n:])
        eps = 1e-6 * np.maximum(1.0, np.abs(xu))                      # [points, d]
        plus = np.repeat(xu[:, None, :], d, axis=1) + np.eye(d)[None] * eps[:, None, :]
        minus = np.repeat(xu[:, None, :], d, axis=1) - np.eye(d)[None] * eps[:, None, :]
        both = np.concatenate((plus, minus)).reshape(-1, d)
        f = self._run_dynamics(both[:, :n], both[:, n:], False).reshape(2, points, d, n)
        fd = ((f[0] - f[1]) / (2.0 * eps[:, :, None])).transpose(0, 2, 1)   # [points, n, d]
        err = np.abs(J - fd)
        tol = 1e-5 * max(1.0, float(np.abs(fd).max()))
        if not np.all(err <= tol):
            p, i, j = np.unravel_index(int(np.argmax(err)), err.shape)
            raise ValueError("the Jacobian of %r disagrees with central differences of its step: "
                             "J[%d][%d] = %.6g at point %d, differences give %.6g"
                             % (self.system_name, i, j, J[p, i, j], p, fd[p, i, j]))
