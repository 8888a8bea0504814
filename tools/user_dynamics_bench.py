"""User-written dynamics (CudaSourceDynamics) against the built-in systems, on one B200.

    python tools/user_dynamics_bench.py [--out FILE]          # GPU: the three timings below
    python tools/user_dynamics_bench.py --construction        # no GPU needed: cold and cached construction

GPU timings (iterations/s of local_descent + evaluate_cost through the public numpy API, built-in and source
alternated over several rounds so that both see the same machine state):
  * pendulum as source against the built-in pendulum, zero order, BASELINE.json configs[0] sizes (T=200, N=1000);
  * bicycle as source against the built-in bicycle, first order, configs[1] sizes (T=100, N=1e4);
  * the cart-pole of tests/test_user_dynamics.py, zero order, T=100, N=1e4.
The card's name and power limit are read in the same run and stored with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import example_configs as ec                                     # noqa: E402
import test_user_dynamics as td                                              # noqa: E402  (the test systems)
from irs_mpc_b200 import user_system                                         # noqa: E402


def source_system(name):
    n, m, h, prm, step, jac = td.SPECS[name]
    return user_system.CudaSourceDynamics(n, m, h, prm, step=step, jacobian=jac, name=name)


def make_solver(api, cls, system, cfg, N):
    n = system.dim_x
    sampler = api.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], N, power=0.5, seed=7)
    p = api.IrsLqrParameters()
    for key in ("Q", "Qd", "R", "x0", "xd_trj", "u_trj_initial"):
        setattr(p, key, cfg[key])
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


def gpu_run(rounds=5, K=200):
    import irs_mpc_b200.all as api
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = {"gpu": smi[0] if smi else "unknown", "rounds": rounds, "iterations_per_round": K, "cases": {}}
    cases = [
        ("pendulum_zero_order_T200_N1000", ec.pendulum(T=200), 1000, api.IrsLqrZeroOrder,
         [("builtin", api.PendulumDynamics(0.05)), ("source", source_system("pendulum_src"))]),
        ("bicycle_first_order_T100_N1e4", ec.bicycle(T=100), 10000, api.IrsLqrFirstOrder,
         [("builtin", api.BicycleDynamics(0.1)), ("source", source_system("bicycle_src"))]),
        ("cartpole_zero_order_T100_N1e4", td.cartpole_cfg(100), 10000, api.IrsLqrZeroOrder,
         [("source", source_system("cartpole"))]),
    ]
    for label, cfg, N, cls, systems in cases:
        solvers = [(tag, make_solver(api, cls, s, cfg, N)) for tag, s in systems]
        rates = {tag: [] for tag, _ in solvers}
        for _ in range(rounds):
            for tag, solver in solvers:
                rates[tag].append(iterations_per_s(solver, K))
        out["cases"][label] = {tag: {"median_iterations_per_s": float(np.median(r)),
                                     "min": float(np.min(r)), "max": float(np.max(r))} for tag, r in rates.items()}
        print(label, json.dumps(out["cases"][label]), flush=True)
    return out


def construction_times():
    """Cold (empty cache: compiles) and cached construction of the cart-pole without a Jacobian body."""
    import shutil
    n, m, h, prm, step, _ = td.SPECS["cartpole_nojac"]
    with tempfile.TemporaryDirectory() as tmp:
        os.environ["IRS_USER_CACHE"] = tmp
        times = []
        for _ in range(2):
            t0 = time.perf_counter()
            user_system.CudaSourceDynamics(n, m, h, prm, step=step, name="cartpole_cold")
            times.append(time.perf_counter() - t0)
        cpus = os.cpu_count()
        nvcc = shutil.which(os.environ.get("NVCC", "nvcc"))
    return {"cold_s": times[0], "cached_s": times[1], "cpus": cpus, "nvcc": nvcc}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--construction", action="store_true")
    args = ap.parse_args()
    res = {"construction": construction_times()} if args.construction else gpu_run()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
