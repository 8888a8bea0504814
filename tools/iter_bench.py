"""iRS-LQR iterations/s at BASELINE.json configs[2] (quadrotor, T=100, N=1e5): local_descent +
evaluate_cost through the public numpy API, for a few pipeline settings (tuning aid).

    python tools/iter_bench.py
"""
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from irs_mpc_b200 import example_configs as ec, irs_lqr as mod                      # noqa: E402
from irs_mpc_b200.all import (GaussianSampling, IrsLqrParameters, IrsLqrZeroOrder,  # noqa: E402
                              QuadrotorDynamics)

cfg = ec.quadrotor(T=100)
CASES = [("auto", True, 0)]
for segs in (3, 4, 5, 6):
    CASES.append(("%d equal" % segs, True, segs))
CASES += [("one pass", False, 0), ("auto", True, 0)]
for label, pipeline, segs in CASES:
    mod._USE_PIPELINE, mod._PIPELINE_SEGMENTS = pipeline, segs
    system = QuadrotorDynamics(cfg["h"])
    params = IrsLqrParameters()
    for key in ("Q", "Qd", "R", "x0", "xd_trj", "u_trj_initial", "xbound", "ubound"):
        setattr(params, key, cfg[key])
    sampler = GaussianSampling(cfg["sigma"][:12], cfg["sigma"][12:], 100000, power=0.5, seed=7)
    solver = IrsLqrZeroOrder(system, params, sampler)
    x, u = solver.x_trj, solver.u_trj
    for _ in range(6):
        solver.local_descent(x, u)
    K = 100
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(K):
        xn, un = solver.local_descent(x, u)
        c = solver.evaluate_cost(xn, un)
    dt = (time.perf_counter() - t0) / K
    print("%-9s %s: %.1f us per descent + cost = %.0f iterations/s (cost %.6f)"
          % (label, solver._pipeline_segments(), dt * 1e6, 1 / dt, c), flush=True)
