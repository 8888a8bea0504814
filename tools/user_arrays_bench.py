"""What reading arrays from device memory (CudaSourceDynamics(..., arrays=...)) costs.

    python tools/user_arrays_bench.py --registers [--out FILE]   # no GPU needed: ptxas registers / spills, loads
    python tools/user_arrays_bench.py [--out FILE]               # GPU: the timings below

--registers compiles every test library of tests/test_user_arrays.py (and the linear plant with its coefficients
written into the body as literals) with -Xptxas -v.  It reports the registers, spill stores and spill loads of
each accumulate kernel the library instantiates, and counts the global loads in its SASS by form: LDG.E.CONSTANT
is the non-coherent read-only path that the arrays' __ldg loads take.

GPU timings (iterations/s of local_descent + evaluate_cost through the public numpy API, the variants alternated
over several rounds so that all see the same machine state), with the mean device time of the accumulate kernel
from torch.profiler:
  * the reference's pendulum network, T=200, N=1e4, zero order: MlpDynamics on its tcgen05 kernel, MlpDynamics on
    its per-thread functor (IRS_MLP_ENGINE=0), and the network written as a source body reading its weights as
    arrays;
  * the same network, first order: MlpDynamics's Jacobian against the source body with autodiff;
  * the (12, 4) linear plant, T=100, N=1e4, zero order and first order (autodiff): A, B, c as arrays against the
    same numbers written into the body as literals.
The card's name and power limit are read in the same run and stored with the numbers.
"""
import argparse
import collections
import concurrent.futures
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import example_configs as ec                                     # noqa: E402
from oracle import user_arrays as ua                                         # noqa: E402
import test_user_arrays as tua                                               # noqa: E402  (the test systems)
from irs_mpc_b200 import _lib, user_system                                   # noqa: E402

ACCUMULATE = ("smooth_zero_order_kernel", "smooth_zero_order_tc_kernel", "smooth_first_order_kernel")


def literal_spec():
    return (12, 4, 0.0, [], ua.linear_literal_step(tua.LIN), None, True)


# ------------------------------------------------------------------------------------------------
# --registers
# ------------------------------------------------------------------------------------------------
def ptxas_report(src, tmp):
    """-> {kernel: {registers, spill_stores, spill_loads, loads: {LDG form: count}}} of the accumulate kernels."""
    cu, so = os.path.join(tmp, "user_system.cu"), os.path.join(tmp, "lib.so")
    with open(cu, "w") as fh:
        fh.write(src)
    cmd = [user_system._nvcc()] + _lib.NVCC_FLAGS + ["-Xptxas", "-v", "-I", _lib.INCLUDE, "-I", _lib.CSRC,
                                                     "-o", so, cu]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(res.stderr)

    def kernel_of(mangled):
        if "UserSystemIfE" not in mangled:
            return None
        return next((k + mangled[mangled.index(k) + len(k):][:40] for k in ACCUMULATE
                     if re.search(r"\d%s" % k + "I", mangled)), None)
    out, current = {}, None
    for line in res.stderr.splitlines():
        m = re.search(r"(?:Compiling entry function|Function properties for) '?(\w+)'?", line)
        if m:
            current = kernel_of(m.group(1))
            continue
        if current is None:
            continue
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m:
            out.setdefault(current, {}).update(spill_stores=int(m.group(1)), spill_loads=int(m.group(2)))
        m = re.search(r"Used (\d+) registers", line)
        if m:
            out.setdefault(current, {})["registers"] = int(m.group(1))
    sass = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True).stdout
    current = None
    for line in sass.splitlines():
        m = re.search(r"Function : (\w+)", line)
        if m:
            current = kernel_of(m.group(1))
        elif current is not None:
            for form in re.findall(r"\b(LDG\.E[\.\w]*)", line):
                out.setdefault(current, {}).setdefault("loads", collections.Counter())[form] += 1
    return out


def registers():
    cases = dict(tua.specs())
    cases["linear_literal"] = literal_spec()
    out = {}
    with tempfile.TemporaryDirectory() as tmp, concurrent.futures.ThreadPoolExecutor(os.cpu_count() or 4) as pool:
        futs = {}
        for i, (name, (n, m, h, prm, step, arrays, ad)) in enumerate(cases.items()):
            d = os.path.join(tmp, str(i))
            os.makedirs(d)
            src = user_system.generate_source(n, m, 1 + len(prm), step, None, ad, arrays)
            futs[name] = pool.submit(ptxas_report, src, d)
        for name, f in futs.items():
            n, m, h, prm, step, arrays, ad = cases[name]
            entry = {"n": n, "m": m, "autodiff": ad,
                     "array_elements": int(sum(np.size(a) for a in (arrays or {}).values())),
                     "kernels": {k: dict(v, loads=dict(v.get("loads", {}))) for k, v in f.result().items()}}
            out[name] = entry
            print(name, json.dumps(entry), flush=True)
    return {"registers": out}


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
def source_system(name):
    n, m, h, prm, step, arrays, ad = literal_spec() if name == "linear_literal" else tua.specs()[name]
    return user_system.CudaSourceDynamics(n, m, h, prm, step=step, autodiff=ad, name=name, arrays=arrays)


def make_solver(api, cls, system, cfg, N):
    n = system.dim_x
    p = api.IrsLqrParameters()
    for key in ("Q", "Qd", "R", "x0", "xd_trj", "u_trj_initial"):
        setattr(p, key, cfg[key])
    sampler = api.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], N, power=0.5, seed=7)
    return cls(system, p, sampler)


def iterations_per_s(solver, K):
    import torch
    x, u = solver.x_trj, solver.u_trj
    for _ in range(5):
        solver.local_descent(x, u)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(K):
        xn, un = solver.local_descent(x, u)
        solver.evaluate_cost(xn, un)
    return K / (time.perf_counter() - t0)


def accumulate_kernel_ms(solver, reps=10):
    """Mean device time of the accumulate kernel over `reps` linearizations (torch.profiler)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    x, u = solver.x_trj, solver.u_trj
    solver.get_TV_matrices(x, u)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            solver.get_TV_matrices(x, u)
        torch.cuda.synchronize()
    total, count = 0.0, 0
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA and \
                ("smooth_zero_order" in ev.name or "smooth_first_order" in ev.name):
            total += ev.device_time
            count += 1
    return total / reps / 1000.0 if count else None


class MlpEngine:
    """IRS_MLP_ENGINE for the duration of a with-block (read by the library per launch; a captured graph keeps
    the kernel it was captured with)."""

    def __init__(self, value):
        self.value = value

    def __enter__(self):
        self.old = os.environ.get("IRS_MLP_ENGINE")
        if self.value is not None:
            os.environ["IRS_MLP_ENGINE"] = self.value

    def __exit__(self, *exc):
        if self.old is None:
            os.environ.pop("IRS_MLP_ENGINE", None)
        else:
            os.environ["IRS_MLP_ENGINE"] = self.old


def gpu_run(rounds=3, K=50):
    import torch
    import irs_mpc_b200.all as api
    assert torch.cuda.is_available(), "the timings need a GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = {"gpu": smi[0] if smi else "unknown", "rounds": rounds, "iterations_per_round": K, "cases": {}}
    mlp = api.MlpDynamics([(w, b) for w, b in zip(tua.golden_weights()[0::2], tua.golden_weights()[1::2])])
    pcfg = ec.pendulum_nn(T=200)
    lcfg = tua.linear_cfg(100)
    mlp_src, mlp_ad = source_system("mlp_src"), source_system("mlp_src_ad")
    lin, lit = source_system("linear"), source_system("linear_literal")
    cases = [
        ("pendulum_network_zero_order_T200_N1e4", pcfg, api.IrsLqrZeroOrder,
         [("MlpDynamics_tcgen05", mlp, "1"), ("MlpDynamics_per_thread", mlp, "0"), ("source_arrays", mlp_src, None)]),
        ("pendulum_network_first_order_T200_N1e4", pcfg, api.IrsLqrFirstOrder,
         [("MlpDynamics", mlp, None), ("source_arrays_autodiff", mlp_ad, None)]),
        ("linear_12x4_zero_order_T100_N1e4", lcfg, api.IrsLqrZeroOrder,
         [("arrays", lin, None), ("literals", lit, None)]),
        ("linear_12x4_first_order_T100_N1e4", lcfg, api.IrsLqrFirstOrder,
         [("arrays", lin, None), ("literals", lit, None)]),
    ]
    for label, cfg, cls, systems in cases:
        solvers = [(tag, make_solver(api, cls, s, cfg, 10000), eng) for tag, s, eng in systems]
        rates = {tag: [] for tag, _, _ in solvers}
        for _ in range(rounds):
            for tag, solver, eng in solvers:
                with MlpEngine(eng):
                    rates[tag].append(iterations_per_s(solver, K))
        res = {tag: {"median_iterations_per_s": float(np.median(r)), "min": float(np.min(r)),
                     "max": float(np.max(r))} for tag, r in rates.items()}
        for tag, solver, eng in solvers:
            with MlpEngine(eng):
                res[tag]["accumulate_kernel_ms"] = accumulate_kernel_ms(solver)
        out["cases"][label] = res
        print(label, json.dumps(res), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--registers", action="store_true")
    args = ap.parse_args()
    res = registers() if args.registers else gpu_run()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
