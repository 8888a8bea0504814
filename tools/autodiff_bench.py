"""What forward-mode Jacobians (CudaSourceDynamics(..., autodiff=True)) cost, against hand-written and built-in ones.

    python tools/autodiff_bench.py --registers [--out FILE]   # no GPU needed: ptxas registers / spills, packed SASS
    python tools/autodiff_bench.py [--out FILE]               # GPU: the timings below

--registers compiles every autodiff test library of tests/test_user_autodiff.py and its hand-Jacobian twin with
-Xptxas -v and reports the registers, spill stores and spill loads of smooth_first_order_kernel<UserSystem<float>>
(the first-order accumulate) and jac_batch_kernel<double, UserSystem<double>>.  It also counts the packed FP32
instructions (FFMA2 / FMUL2 / FADD2) in the accumulate kernel's SASS.

GPU timings (iterations/s of local_descent + evaluate_cost through the public numpy API, the variants alternated
over several rounds so that all see the same machine state):
  * bicycle, first order, BASELINE.json configs[1] sizes (T=100, N=1e4): built-in, source with the hand-written
    Jacobian, source with autodiff;
  * cart-pole, first order, T=100, N=1e4: hand-written Jacobian against autodiff;
  * quadrotor, first order at T=100, N=1e4, and exact at T=100: built-in against source with autodiff;
and the mean time of the first-order accumulate kernel in each first-order case, from torch.profiler.  The
card's name and power limit are read in the same run and stored with the numbers.
"""
import argparse
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
import test_user_autodiff as ta                                              # noqa: E402  (the test systems)
import test_user_dynamics as td                                              # noqa: E402
from irs_mpc_b200 import _lib, user_system                                   # noqa: E402

KERNELS = {"smooth_first_order_kernel<UserSystem<float>>": "smooth_first_order_kernelINS_10UserSystemIfEE",
           "jac_batch_kernel<double, UserSystem<double>>": "jac_batch_kernelIdNS_10UserSystemIdEE"}
PACKED = ("FFMA2", "FMUL2", "FADD2")


# ------------------------------------------------------------------------------------------------
# --registers
# ------------------------------------------------------------------------------------------------
def ptxas_report(src, tmp):
    """-> ({kernel: {registers, spill_stores, spill_loads}}, SASS counts of PACKED in the accumulate kernel)."""
    cu, so = os.path.join(tmp, "user_system.cu"), os.path.join(tmp, "lib.so")
    with open(cu, "w") as fh:
        fh.write(src)
    cmd = [user_system._nvcc()] + _lib.NVCC_FLAGS + ["-Xptxas", "-v", "-I", _lib.INCLUDE, "-I", _lib.CSRC,
                                                     "-o", so, cu]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(res.stderr)
    out, current = {}, None
    for line in res.stderr.splitlines():
        m = re.search(r"(?:Compiling entry function|Function properties for) '?(\w+)'?", line)
        if m:
            current = next((k for k, pat in KERNELS.items() if pat in m.group(1)), None)
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
    counts, inside = {k: 0 for k in PACKED}, False
    for line in sass.splitlines():
        if "Function :" in line:
            inside = KERNELS["smooth_first_order_kernel<UserSystem<float>>"] in line
        elif inside:
            for k in PACKED:
                counts[k] += len(re.findall(r"\b%s\b" % k, line))
    return out, counts


def registers():
    cases = []
    for name, (n, m, h, prm, step) in ta.AD_SPECS.items():
        cases.append((name, "autodiff", user_system.generate_source(n, m, 1 + len(prm), step, None, True)))
        twin = ta.TWIN_OF.get(name) or (name.replace("grid_ad_", "grid_") if name.startswith("grid_ad_") else None)
        if twin is not None:
            n2, m2, h2, prm2, step2, jac2 = ta.HAND_SPECS[twin]
            cases.append((twin, "hand", user_system.generate_source(n2, m2, 1 + len(prm2), step2, jac2)))
    out = {}
    with tempfile.TemporaryDirectory() as tmp, concurrent.futures.ThreadPoolExecutor(os.cpu_count() or 4) as pool:
        futs = {}
        for i, (name, kind, src) in enumerate(cases):
            d = os.path.join(tmp, str(i))
            os.makedirs(d)
            futs[(name, kind)] = pool.submit(ptxas_report, src, d)
        for (name, kind), f in futs.items():
            kern, packed = f.result()
            n, m = (ta.AD_SPECS.get(name) or ta.HAND_SPECS[name])[:2]
            entry = {"n": n, "m": m, "jacobian": kind, "kernels": kern}
            if kind == "autodiff":
                entry["passes_lanes"] = list(user_system.autodiff_passes(n + m))
                entry["accumulate_packed_fp32_sass"] = packed
            out[name] = entry
            print(name, json.dumps(entry), flush=True)
    return {"registers": out}


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
def source_system(name):
    if name in ta.AD_SPECS:
        n, m, h, prm, step = ta.AD_SPECS[name]
        return user_system.CudaSourceDynamics(n, m, h, prm, step=step, autodiff=True, name=name)
    n, m, h, prm, step, jac = td.SPECS[name]
    return user_system.CudaSourceDynamics(n, m, h, prm, step=step, jacobian=jac, name=name)


def make_solver(api, cls, system, cfg, N):
    n = system.dim_x
    p = api.IrsLqrParameters()
    for key in ("Q", "Qd", "R", "x0", "xd_trj", "u_trj_initial"):
        setattr(p, key, cfg[key])
    if cls is api.IrsLqrExact:
        return cls(system, p)
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


def accumulate_kernel_ms(solver, reps=20):
    """Mean device time of the first-order accumulate kernel over `reps` linearizations (torch.profiler)."""
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
        if "smooth_first_order_kernel" in ev.name and ev.device_type == torch.autograd.DeviceType.CUDA:
            total += ev.device_time
            count += 1
    return total / count / 1000.0 if count else None


def gpu_run(rounds=5, K=100):
    import torch
    import irs_mpc_b200.all as api
    assert torch.cuda.is_available(), "the timings need a GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = {"gpu": smi[0] if smi else "unknown", "rounds": rounds, "iterations_per_round": K, "cases": {}}
    qcfg = ec.quadrotor(T=100)
    cases = [
        ("bicycle_first_order_T100_N1e4", ec.bicycle(T=100), 10000, api.IrsLqrFirstOrder,
         [("builtin", api.BicycleDynamics(0.1)), ("source_hand", source_system("bicycle_src")),
          ("source_autodiff", source_system("bicycle_ad"))]),
        ("cartpole_first_order_T100_N1e4", td.cartpole_cfg(100), 10000, api.IrsLqrFirstOrder,
         [("source_hand", source_system("cartpole")), ("source_autodiff", source_system("cartpole_ad"))]),
        ("quadrotor_first_order_T100_N1e4", qcfg, 10000, api.IrsLqrFirstOrder,
         [("builtin", api.QuadrotorDynamics(qcfg["h"])), ("source_autodiff", source_system("quadrotor_ad"))]),
        ("quadrotor_exact_T100", qcfg, 0, api.IrsLqrExact,
         [("builtin", api.QuadrotorDynamics(qcfg["h"])), ("source_autodiff", source_system("quadrotor_ad"))]),
    ]
    for label, cfg, N, cls, systems in cases:
        solvers = [(tag, make_solver(api, cls, s, cfg, N)) for tag, s in systems]
        rates = {tag: [] for tag, _ in solvers}
        for _ in range(rounds):
            for tag, solver in solvers:
                rates[tag].append(iterations_per_s(solver, K))
        res = {tag: {"median_iterations_per_s": float(np.median(r)), "min": float(np.min(r)),
                     "max": float(np.max(r))} for tag, r in rates.items()}
        if cls is api.IrsLqrFirstOrder:
            for tag, solver in solvers:
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
