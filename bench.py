#!/usr/bin/env python
"""Benchmark of the iRS-MPC hot path (BASELINE.json: smoothed-dynamics samples/s and iRS-LQR
iterations/s at 1/2/4/8 B200 vs the numpy CPU path).

    python bench.py --gpus N --steps K --warmup W            (torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR

--dump-outputs DIR writes what the last timed step returned (At, Bt, ct and the per-point fit status, all
float64) as DIR/<name>.npy.  The inputs depend only on the arguments, so two builds run with the same
arguments can be compared output for output.

Workload (config.workload): BASELINE.json configs[2] — quadrotor 12-state, IrsLqrZeroOrder,
T=100, N=1e5 samples/step per GPU.  A "step" is one full smoothing linearization
(IrsLqrZeroOrder.get_TV_matrices: T x N perturbed dynamics evaluations + least-squares fits).
For N GPUs the SAMPLE axis is sharded (weak scaling: every GPU draws 1e5 samples per step, the
global fit uses N*1e5); the per-step fp64 Gram blocks are exchanged by the chunk-reduction kernel
itself through peer memory (NCCL all-gather as fallback).

One JSON line on stdout (rank 0); everything else goes to stderr.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

T_STEPS = 100
N_SAMPLES = 100000
FLOPS_PER_SAMPLE = 838        # SURVEY.md section 8(d): quadrotor zero-order, algorithmic, FMA = 2
FP32_NOMINAL_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12
SEED0 = 0x1255 + 3
DRAM_BYTES_PER_LAUNCH = 64512   # ncu capture of the dominant kernel, see roofline.traffic_source


def log(*a):
    print(*a, file=sys.stderr, flush=True)


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons every 50 ms from process start; the report uses
    the samples that arrived inside the load windows (timed regions + a sustained repeat of the
    same step, because K steps of this workload last only a few milliseconds)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.windows = index, [], None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception as e:       # nvidia-smi missing: report it, do not fail the bench
            log("clock sampler unavailable:", e)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def window(self, t0, t1):
        self.windows.append((t0, t1))

    def samples_in_windows(self):
        return sum(1 for t, _ in self.rows if any(a <= t <= b for a, b in self.windows))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, r in self.rows:
            if not any(a <= t <= b for a, b in self.windows):
                continue
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for k, name in enumerate(names):
                    if r[4 + k].lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "how": "nvidia-smi -lms 50; samples inside the timed regions and a >=1.5 s sustained repeat "
                       "of the same step"}


def _reference_timing_note():
    """The committed timing of the unmodified reference (build container; it cannot travel to the GPU box)."""
    try:
        t = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_timing.json")))["cases"]
        return "; ".join("%s T=%d N=%d: %.3g samples/s" % (k, v["T"], v["N"], v["samples_per_s"]) for k, v in t.items())
    except Exception:
        return "unavailable"


def dump_outputs(out_dir, arrays):
    """arrays: name -> numpy array, written as out_dir/<name>.npy in float64 (the fit status as 0.0 / 1.0 / 2.0)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))
    log("outputs of the last timed step written to", out_dir)


def quadrotor_problem(for_cpu=False):
    if for_cpu:
        from oracle import example_configs as ec          # CPU baseline leg only
    else:
        from irs_mpc_b200 import example_configs as ec
    return ec.quadrotor(T=T_STEPS)


# ------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the float64 numpy port of the reference path (oracle), timed on
# the host cores.  The unmodified reference cannot travel to the GPU box (pure Python tree at
# /root/reference, needs pydrake) -> kind "port".
# ------------------------------------------------------------------------------------------------
def _cpu_chunk(args):
    t0, t1, n_samples, seed = args
    from oracle import cpu_restatement as cr
    cfg = quadrotor_problem(for_cpu=True)
    orc = cr.QuadrotorOracle(cfg["h"])
    x_trj = cr.rollout(orc, cfg["x0"], cfg["u_trj_initial"])
    rng = np.random.default_rng(seed + t0)
    # the reference draws its normals inside the timed loop too (sampling closure)
    deltas = rng.standard_normal((t1 - t0, n_samples, 16)) * cfg["sigma"]
    cr.zero_order_tv_matrices(orc, x_trj[t0:t1 + 1], cfg["u_trj_initial"][t0:t1], deltas)
    return (t1 - t0) * n_samples


def cpu_pass(n_samples, procs, seed=0, pool=None):
    """One smoothing pass (T=100 timesteps x n_samples) on `procs` host processes, sharded by
    timestep like the reference's ZeroMQ task farm.  Returns (samples, seconds)."""
    bounds = np.linspace(0, T_STEPS, procs + 1).astype(int)
    jobs = [(int(bounds[i]), int(bounds[i + 1]), n_samples, seed) for i in range(procs)
            if bounds[i + 1] > bounds[i]]
    t = time.perf_counter()
    if pool is None:
        done = sum(_cpu_chunk(j) for j in jobs)
    else:
        done = sum(pool.map(_cpu_chunk, jobs))
    return done, time.perf_counter() - t


def run_reference(args, rank, world):
    if rank != 0:
        return
    import multiprocessing as mp
    procs = max(1, min(os.cpu_count() or 1, T_STEPS))
    n_samples = 20000          # bounded sample of the 1e5-samples/step workload (per-sample cost is flat in N)
    # one BLAS thread per worker process (the workers already cover every core)
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = "1"
    ctx = mp.get_context("spawn")
    with ctx.Pool(procs) as pool:
        for _ in range(max(1, min(args.warmup, 1))):
            cpu_pass(2000, procs, pool=pool)
        total, secs = 0, 0.0
        for k in range(args.steps):
            done, dt = cpu_pass(n_samples, procs, seed=k, pool=pool)
            total += done
            secs += dt
    value = total / secs
    sample = ("float64 numpy port (oracle/cpu_restatement.py) of IrsLqrZeroOrder.get_TV_matrices, quadrotor "
              "T=100, N=%d samples/step (bounded from 1e5; cost per sample is flat in N), %d host processes "
              "sharded by timestep; the UNMODIFIED reference's get_TV_matrices timed in the build container "
              "(tests/golden/reference_timing.json): %s" % (n_samples, procs, _reference_timing_note()))
    out = {
        "impl": "reference", "metric": "smoothed_dynamics_samples_per_s", "value": value, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "quadrotor zero-order T=100 N=%d/step (CPU sample of cfg3)" % n_samples},
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": procs, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_gpu(args, rank, local_rank, world):
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from irs_mpc_b200 import _device, _lib, smoothing
    from irs_mpc_b200.all import (GaussianSampling, IrsLqrParameters, IrsLqrZeroOrder,
                                  QuadrotorDynamics)
    from irs_mpc_b200.distributed import ShardedLinearizer

    cfg = quadrotor_problem()
    system = QuadrotorDynamics(cfg["h"])
    params = IrsLqrParameters()
    for key in ("Q", "Qd", "R", "x0", "xd_trj", "u_trj_initial", "xbound", "ubound"):
        setattr(params, key, cfg[key])
    sampler = GaussianSampling(cfg["sigma"][:12], cfg["sigma"][12:], N_SAMPLES, power=cfg["power"], seed=SEED0)
    solver = IrsLqrZeroOrder(system, params, sampler)
    x_host, u_host = solver.x_trj, solver.u_trj
    x_nom = _device.to_device(x_host[:T_STEPS])
    u_nom = _device.to_device(u_host)
    sigma = sampler.sigma(1)
    ws = smoothing.Workspace(system, smoothing.ZERO_ORDER, T_STEPS, N_SAMPLES)
    sharded = ShardedLinearizer(system, smoothing.ZERO_ORDER) if world > 1 else None
    # ours per step: accumulate + finalize; when sample-sharded the finalize kernel itself reduces, exchanges
    # (peer-memory stores over NVLink + per-point arrival flags) and fits, so the count does not change
    # (NCCL fallback: + chunk reduction, and the all-gather is NCCL's)
    launches_per_step = 2

    def step_device(k):
        """Inputs resident in HBM; the seed changes every step so nothing can be cached."""
        if world == 1:
            smoothing.accumulate(system, smoothing.ZERO_ORDER, x_nom, u_nom, N_SAMPLES, ws, sigma=sigma,
                                 seed=SEED0 + k, it=1, flags=sampler.flags())
            return smoothing.finalize(system, smoothing.ZERO_ORDER, x_nom, u_nom, ws, N_SAMPLES)
        return sharded.linearize_n(x_nom, u_nom, N_SAMPLES, sigma=sigma, seed=SEED0 + k, it=1, flags=sampler.flags())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    tick = torch.zeros((1,), dtype=torch.float32, device="cuda")

    def timed(fn, steps, warmup, outputs=None):
        """Device time of `steps` calls after `warmup` untimed ones.  `outputs` (a list) receives host copies
        of the tensors the last timed call returned, taken after the end event."""
        for k in range(warmup):
            fn(k)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if world > 1:
            # the host threads leave the barrier up to ~0.2 ms apart, which the first exchange of the timed steps
            # would pay as a one-time wait (7 us per step at 30 steps): align the ranks ON THE DEVICE with a
            # stream-ordered collective right before the start event — no host sync, the timed launches queue behind it
            dist.all_reduce(tick)
        e0.record()
        for k in range(steps):
            last = fn(warmup + k)
        e1.record()
        barrier()
        if outputs is not None:
            outputs.extend(_device.to_numpy(t) for t in last)
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # 1. headline: device-resident throughput of the whole smoothing pass
    t_w0 = time.time()
    last_step = [] if args.dump_outputs and rank == 0 else None
    ms = timed(step_device, args.steps, args.warmup, outputs=last_step)
    if last_step is not None:
        dump_outputs(args.dump_outputs, dict(zip(("At", "Bt", "ct", "status"), last_step)))
    samples_per_step = world * T_STEPS * N_SAMPLES
    value = samples_per_step * args.steps / (ms * 1e-3)

    # 2. dominant kernel alone (accumulate), CUDA events on the launching stream
    def only_accumulate(k):
        smoothing.accumulate(system, smoothing.ZERO_ORDER, x_nom, u_nom, N_SAMPLES, ws, sigma=sigma,
                             seed=SEED0 + 1000 + k, it=1, flags=sampler.flags())
    ms_kernel = timed(only_accumulate, args.steps, 1) / args.steps
    clocks.window(t_w0, time.time())
    # sustained repeat of the same step so that the 50 ms sampler sees the clocks under this load
    t_l0 = time.time()
    n_load = int(min(200000, max(100, 2000.0 / max(ms / args.steps, 1e-3))))   # ~2 s, same count on all ranks
    for k in range(n_load):
        step_device(100000 + k)
        if k % 256 == 255:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    clocks.window(t_l0, time.time())
    barrier()
    clock_info = clocks.stop() if rank == 0 else None

    # 2b. the same kernel in replay mode (pre-generated noise streamed from HBM, the parity path):
    #     64 B/sample of algorithmic traffic; buffer (640 MB) is far larger than the 126 MB L2
    replay = None
    if world == 1:
        noise = torch.empty((T_STEPS, N_SAMPLES, 16), dtype=torch.float32, device="cuda").normal_(0.0, 0.1)

        def only_replay(k):
            smoothing.accumulate(system, smoothing.ZERO_ORDER, x_nom, u_nom, N_SAMPLES, ws, noise=noise)
        ms_replay = timed(only_replay, args.steps, 2) / args.steps
        gbs = T_STEPS * N_SAMPLES * 64 / (ms_replay * 1e-3) / 1e9
        del noise
        torch.cuda.empty_cache()

    # 3. measured FP32 FMA peak (roofline denominator), best of 5
    scratch = _device.empty((148 * 8 * 256,), torch.float32)
    import ctypes
    flops = ctypes.c_double(0.0)
    best = 0.0
    for _ in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.call("irs_fp32_fma_peak", 20000, _device.ptr(scratch), scratch.numel(), ctypes.byref(flops),
                  _device.stream_ptr())
        e1.record()
        torch.cuda.synchronize()
        best = max(best, flops.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    achieved_tflops = T_STEPS * N_SAMPLES * FLOPS_PER_SAMPLE / (ms_kernel * 1e-3) / 1e12

    # 4. end to end through the public API: numpy in -> get_TV_matrices -> numpy out
    if world == 1:
        def step_e2e(k):
            sampler.seed = SEED0 + 5000 + k
            return solver.get_TV_matrices(x_host, u_host)
    else:
        def step_e2e(k):
            # numpy in, numpy out through the sharded public call: one pinned H2D, one D2H per step
            return sharded.linearize_n_numpy(x_host[:T_STEPS], u_host, N_SAMPLES, sigma=sigma,
                                             seed=SEED0 + 5000 + k, it=1, flags=sampler.flags())
    ms_e2e = timed(step_e2e, args.steps, min(args.warmup, 3))
    e2e_value = samples_per_step * args.steps / (ms_e2e * 1e-3)
    n, m = 12, 4
    if world == 1:
        h2d, d2h = solver._io_bytes()            # counted from the buffers the API copies
    else:
        h2d, d2h = sharded._ws.h2d_bytes(), sharded._ws.d2h_bytes()

    # 5. iRS-LQR iterations/s: local_descent (smoothing + Riccati + closed-loop rollout) + evaluate_cost,
    #    teacher-forced from the initial trajectory, through the public numpy API (replicated per rank)
    def one_iteration(k):
        sampler.seed = SEED0 + 9000 + k
        xn, un = solver.local_descent(x_host, u_host)
        return solver.evaluate_cost(xn, un)
    it_steps = max(3, min(args.steps, 20))
    ms_iter = timed(one_iteration, it_steps, 4)      # the call sequence is captured into a CUDA graph on its 3rd call
    iters_per_s = it_steps / (ms_iter * 1e-3)

    # 5b. BASELINE.json configs[4]: 4096 independent quadrotor MPC instances (T=100, N=1e3 samples/step as
    #     in examples/quadrotor/quadrotor_zero_order.py:44), instances sharded over the ranks, no
    #     collective on the data path.  One step = one local_descent of every instance, device resident.
    batched = None
    if not args.no_batched:
        from irs_mpc_b200.all import BatchedIrsLqrZeroOrder
        I_total = 4096
        lo, hi = rank * I_total // world, (rank + 1) * I_total // world
        # instance b tracks the example's helix with phase 2 pi b / 4096 and starts on it plus noise from
        # default_rng(5000 + b) (example_configs.quadrotor_batch; tests/test_full_size_parity.py uses the same)
        from irs_mpc_b200 import example_configs as gec5
        x0b, xdb = gec5.quadrotor_batch(lo, hi, T=T_STEPS, total=I_total)
        smp = GaussianSampling(cfg["sigma"][:12], cfg["sigma"][12:], 1000, power=cfg["power"], seed=SEED0 + 77)
        bat = BatchedIrsLqrZeroOrder(system, cfg["Q"], cfg["Qd"], cfg["R"], x0b, xdb, cfg["u_trj_initial"], smp,
                                     instance_offset=lo)

        def batched_step(k):
            smp.seed = SEED0 + 77 + k
            return bat.local_descent()
        b_steps = max(3, min(args.steps, 5))
        ms_b = timed(batched_step, b_steps, 2) / b_steps
        bat.check()
        batched = {"workload": "BASELINE.json configs[4]: 4096 quadrotor MPC instances, T=100, N=1000 samples/step, "
                               "zero-order smoothing + Riccati + closed-loop rollout per step",
                   "instances": I_total, "instances_per_gpu": hi - lo, "ms_per_batch_iteration": ms_b,
                   "instance_iterations_per_s": I_total / (ms_b * 1e-3),
                   "samples_per_s": I_total * T_STEPS * 1000 / (ms_b * 1e-3)}
        del bat

    # 5c. the other BASELINE.json configs, device resident (parity-test cases; reported for orientation)
    other = None
    if world == 1 and not args.no_other_configs:
        from irs_mpc_b200 import example_configs as gec
        from irs_mpc_b200.systems import SYSTEM_CLASSES
        other = {}
        for label, name, order, Tn, Nn, proj in (
                ("configs[0] pendulum zero-order T=200 N=1e3", "pendulum", smoothing.ZERO_ORDER, 200, 1000, False),
                ("configs[1] bicycle first-order T=100 N=1e4", "bicycle", smoothing.FIRST_ORDER, 100, 10000, False),
                ("configs[3] three_cart zero-order T=100 N=1e6, in-kernel projection", "three_cart",
                 smoothing.ZERO_ORDER, 100, 1000000, True)):
            c2 = gec.CONFIGS[name](T=Tn)
            sys2 = SYSTEM_CLASSES[name](c2["h"])
            xn2 = _device.to_device(np.zeros((Tn, sys2.dim_x)) + c2["x0"])
            un2 = _device.to_device(c2["u_trj_initial"])
            ws2 = smoothing.Workspace(sys2, order, Tn, Nn)

            def step2(k, sys2=sys2, order=order, xn2=xn2, un2=un2, ws2=ws2, c2=c2, Nn=Nn, proj=proj):
                smoothing.accumulate(sys2, order, xn2, un2, Nn, ws2, sigma=c2["sigma"], seed=SEED0 + k, it=1,
                                     flags=(2 if proj else 0) | sampler.flags())
                smoothing.finalize(sys2, order, xn2, un2, ws2, Nn)
            ms2 = timed(step2, max(5, min(args.steps, 20)), 3) / max(5, min(args.steps, 20))
            other[label] = {"ms_per_linearization": ms2, "samples_per_s": Tn * Nn / (ms2 * 1e-3)}
            del ws2
            # the same linearization end to end through the public API (numpy in -> get_TV_matrices -> numpy out)
            try:
                from irs_mpc_b200.all import IrsLqrFirstOrder
                p2 = IrsLqrParameters()
                for key in ("Q", "Qd", "R", "x0", "xd_trj", "u_trj_initial", "xbound", "ubound"):
                    setattr(p2, key, c2[key])
                smp2 = GaussianSampling(c2["sigma"][:sys2.dim_x], c2["sigma"][sys2.dim_x:], Nn, power=c2["power"],
                                        seed=SEED0 + 31, projection="absolute" if proj else None)
                cls2 = IrsLqrZeroOrder if order == smoothing.ZERO_ORDER else IrsLqrFirstOrder
                sol2 = cls2(sys2, p2, smp2)
                xh2, uh2 = sol2.x_trj, sol2.u_trj

                def e2e2(k, sol2=sol2, smp2=smp2, xh2=xh2, uh2=uh2):
                    smp2.seed = SEED0 + 31 + k
                    return sol2.get_TV_matrices(xh2, uh2)
                reps2 = max(5, min(args.steps, 20))
                other[label]["e2e_ms_per_linearization"] = timed(e2e2, reps2, 4) / reps2
                del sol2
            except Exception as e:
                other[label]["e2e_error"] = repr(e)
        # learned dynamics (SURVEY.md 8(f)-4; the reference's examples/pendulum/pendulum_nn.py: 3-100-100-2 ReLU network,
        # T=200, N=1e4 samples per step): hidden layer of the network on tcgen05; committed weights of a network
        # trained the way the script trains it (tests/golden/mlp_pendulum.npz, oracle/make_mlp_fixture.py)
        try:
            from irs_mpc_b200.all import MlpDynamics
            gw = np.load(os.path.join(ROOT, "tests", "golden", "mlp_pendulum.npz"))
            net = MlpDynamics([(gw["W1"], gw["b1"]), (gw["W2"], gw["b2"]), (gw["W3"], gw["b3"])])
            c3 = gec.pendulum_nn(T=200)
            xn3 = _device.to_device(np.cumsum(0.02 * np.ones((200, 2)), axis=0))
            un3 = _device.to_device(c3["u_trj_initial"])
            ws3 = smoothing.Workspace(net, smoothing.ZERO_ORDER, 200, 10000)

            def acc3(k):
                smoothing.accumulate(net, smoothing.ZERO_ORDER, xn3, un3, 10000, ws3, sigma=c3["sigma"], seed=SEED0 + k,
                                     it=1, flags=sampler.flags())

            def step3(k):
                acc3(k)
                smoothing.finalize(net, smoothing.ZERO_ORDER, xn3, un3, ws3, 10000)
            reps3 = max(5, min(args.steps, 20))
            ms3 = timed(step3, reps3, 3) / reps3
            ms3k = timed(acc3, reps3, 3) / reps3
            net_flops = 2 * (3 * 100 + 100 * 100 + 100 * 2)
            tf = 200 * 10000 * net_flops / (ms3k * 1e-3) / 1e12
            bf16_peak = None
            try:
                bf16_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops")
            except Exception:
                pass
            other["learned dynamics (pendulum_nn.py network 3-100-100-2) zero-order T=200 N=1e4"] = {
                "ms_per_linearization": ms3, "samples_per_s": 200 * 10000 / (ms3 * 1e-3),
                "kernel": "smooth_zero_order_mlp_kernel (first + hidden layer: tcgen05 UMMA 128x112x16, bf16-split x3)",
                "kernel_ms": ms3k, "network_tflops_algorithmic": tf,
                "tensor_peak_bf16_tflops": bf16_peak,
                "frac_of_tensor_peak": (3.0 * 2 * (16 * 112 + 112 * 112) / float(net_flops) * tf / bf16_peak) if bf16_peak else None,
                "frac_note": "EXECUTED tensor flops (3 split products; first layer K = 16, hidden layer on operands padded to "
                             "112 x 112) over the measured bf16 peak; the kernel is a chain of UMMA / TMEM latencies per tile, "
                             "no pipe is saturated (profiles/r2_mlp_tc_full.txt)"}
            del ws3, net
        except Exception as e:      # the headline line must not depend on the optional leg
            other["learned dynamics"] = {"error": repr(e)}

    # 5d. STRONG scaling of the named configs: the TOTAL sample count of BASELINE.json configs[2] (N = 1e5 per
    #     step) and configs[3] (three_cart, N = 1e6 per step) split over the ranks — sample axis (fused peer
    #     exchange inside the finalize kernel) and, for configs[2], the north star's timestep axis (each rank
    #     linearizes T / W timesteps, NCCL all-gather of the packed [A|B|c] blocks, 81.6 KB).  At world == 1 the
    #     same calls give the single-GPU times the ratios refer to.  ms per step, max over ranks.
    strong = None
    if not args.no_strong:
        from irs_mpc_b200 import example_configs as gec
        from irs_mpc_b200.systems import SYSTEM_CLASSES
        strong = {"note": "total work fixed, split over n_gpus ranks; ms per linearization step (device time, max "
                          "over ranks); efficiency = t(1 GPU) / (n_gpus * t(n_gpus)) with the 1-GPU run of this bench"}
        st_steps = max(5, min(args.steps, 20))

        def strong_case(name, Tn, N_total, proj_flag, with_t_axis):
            c2 = gec.CONFIGS[name](T=Tn)
            sys2 = SYSTEM_CLASSES[name](c2["h"])
            xn2 = _device.to_device(np.zeros((Tn, sys2.dim_x)) + c2["x0"]) if name != "quadrotor" else x_nom
            un2 = _device.to_device(c2["u_trj_initial"]) if name != "quadrotor" else u_nom
            fl = proj_flag | sampler.flags()
            out = {"T": Tn, "N_total": N_total, "N_per_gpu": N_total // world}
            if world == 1:
                ws2 = smoothing.Workspace(sys2, smoothing.ZERO_ORDER, Tn, N_total)

                def f1(k):
                    smoothing.accumulate(sys2, smoothing.ZERO_ORDER, xn2, un2, N_total, ws2, sigma=c2["sigma"],
                                         seed=SEED0 + k, it=1, flags=fl)
                    smoothing.finalize(sys2, smoothing.ZERO_ORDER, xn2, un2, ws2, N_total)
                t1 = timed(f1, st_steps, 3) / st_steps
                out["sample_axis_ms"] = t1
                if with_t_axis:
                    out["timestep_axis_ms"] = t1
                del ws2
            else:
                sh2 = ShardedLinearizer(sys2, smoothing.ZERO_ORDER)
                n_loc = N_total // world

                def fn(k):
                    sh2.linearize_n(xn2, un2, n_loc, sigma=c2["sigma"], seed=SEED0 + k, it=1, flags=fl)
                out["sample_axis_ms"] = timed(fn, st_steps, 4) / st_steps
                out["sample_axis_exchange"] = "peer memory, fused into the finalize kernel" if sh2._px is not None \
                    else "NCCL all_gather"
                if with_t_axis:
                    def ft(k):
                        sh2.linearize_t(xn2, un2, N_total, sigma=c2["sigma"], seed=SEED0 + k, it=1, flags=fl)
                    out["timestep_axis_ms"] = timed(ft, st_steps, 3) / st_steps
            out["samples_per_s_sample_axis"] = Tn * N_total / (out["sample_axis_ms"] * 1e-3)
            return out
        strong["configs[2] quadrotor T=100 N=1e5 total"] = strong_case("quadrotor", T_STEPS, N_SAMPLES, 0, True)
        strong["configs[3] three_cart T=100 N=1e6 total, in-kernel projection"] = strong_case(
            "three_cart", 100, 1000000, 2, False)

    # 6. CPU baseline on this box's host cores (rank 0, single GPU run only), bounded sample
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_pass(2000, 1)
        done, secs = cpu_pass(N_SAMPLES, 1)
        cpu = {"value": done / secs, "unit": "samples/s", "cores": 1, "kind": "port",
               "sample": "float64 numpy port (oracle) of IrsLqrZeroOrder.get_TV_matrices, quadrotor T=100 N=1e5 "
                         "(one full step, %.1f s, single process; numpy elementwise is single-threaded, only "
                         "lstsq may use BLAS threads).  The UNMODIFIED reference's get_TV_matrices, timed in the "
                         "build container (tests/golden/reference_timing.json, oracle/make_script_fixtures.py): "
                         "%s" % (secs, _reference_timing_note())}

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        out = {
            "metric": "smoothed_dynamics_samples_per_s", "value": value, "unit": "samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "quadrotor zero-order T=100 N=1e5/step/GPU (BASELINE.json configs[2])",
                       "system": "quadrotor n=12 m=4", "mode": "zero_order", "T": T_STEPS,
                       "samples_per_step_per_gpu": N_SAMPLES, "noise": "Philox4x32-7 + Box-Muller in-kernel, antithetic pairs x +- z "
                                                                     "(GaussianSampling default; one draw per pair)",
                       "sharding": "none" if world == 1 else (
                           "sample axis; fp64 Gram blocks exchanged inside the finalize kernel (peer-memory "
                           "stores over NVLink + per-point arrival flags), no NCCL on the data path" if sharded._px is not None else
                           "sample axis, NCCL all_gather of fp64 Gram blocks"),
                       "l2": "no per-sample HBM input (noise generated in registers); seed changes every step"},
            "iters_per_s": iters_per_s, "ms_per_iteration": ms_iter / it_steps,
            "batched_mpc": batched,
            "other_configs": other,
            "strong_scaling": strong,
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches_per_step * args.steps,
            "roofline": {"bound": "fp32", "kernel": "smooth_zero_order_tc_kernel<Quadrotor<float>,1,kTcPaired,false>",
                         "achieved": achieved_tflops, "peak": best, "unit": "TFLOP/s",
                         "frac": achieved_tflops / best if best > 0 else None,
                         "peak_source": "measured on this box: dependent-chain FFMA microbenchmark (irs_fp32_fma_peak); "
                                        "nominal 148 SM x 128 lanes x 2 x 1.965 GHz = %.1f" % FP32_NOMINAL_TFLOPS,
                         "frac_of_nominal": achieved_tflops / FP32_NOMINAL_TFLOPS,
                         "flops_per_sample": FLOPS_PER_SAMPLE, "kernel_ms": ms_kernel,
                         "traffic": DRAM_BYTES_PER_LAUNCH,
                         "traffic_source": "ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum of one launch "
                                           "(profiles/r2_smooth_tc_paired_full.txt): the kernel reads the nominal points and "
                                           "writes 3.3 MB of packed Gram blocks that stay in L2",
                         "bound_note": "Philox mode has no per-sample HBM stream, so the kernel is bounded by FP32 "
                                       "issue, not by HBM or the tensor pipe (DESIGN.md 3.1)",
                         "achieved_note": "ALGORITHMIC flops (SURVEY.md 8(d): 838 per fitted sample, of which 656 are the "
                                          "Gram update) over the measured kernel time.  The kernel executes fewer: the "
                                          "Gram runs on the tensor cores, and an antithetic pair x +- z contributes ONE "
                                          "rank-1 update (2 z z^T, z (f+ - f-)^T) for two fitted samples; what the "
                                          "CUDA cores issue is 296 instructions per sample (ncu, "
                                          "profiles/r2_smooth_tc_paired_full.txt: issue slots 70 % busy)",
                         "hbm_gbs_measured_peak": peaks.get("hbm_gbs")},
            "roofline_replay_mode": None if world > 1 else {
                "bound": "hbm", "kernel": "smooth_zero_order_tc_kernel<Quadrotor<float>,1,kTcReplay,false> (noise replayed from HBM)",
                "achieved": gbs, "peak": peaks.get("hbm_gbs"), "unit": "GB/s",
                "frac": gbs / peaks["hbm_gbs"] if peaks.get("hbm_gbs") else None,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)", "bytes_per_sample": 64,
                "kernel_ms": ms_replay, "samples_per_s": T_STEPS * N_SAMPLES / (ms_replay * 1e-3),
                "note": "parity/compat path; still bounded by FP32 issue, not by HBM"},
            "cpu_baseline": cpu,
            "clocks": clock_info,
        }
        result_line = json.dumps(out)
    else:
        result_line = None
    if world > 1:
        dist.destroy_process_group()
    return result_line


class StdoutGuard:
    """Everything written to fd 1 while active goes to stderr (NCCL prints its version banner to
    stdout; native libraries may too) so that stdout carries exactly the one JSON line."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-batched", action="store_true", help="skip the 4096-instance leg (configs[4])")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the pendulum/bicycle/three_cart legs")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (GPU arm only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs the GPU arm (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        log("note: warmup raised to 3 (timing rules)")
        args.warmup = 3
    with StdoutGuard():
        line = run_gpu(args, rank, local_rank, world)
    if line is not None:
        print(line, flush=True)


if __name__ == "__main__":
    main()
