"""Where the time of the few-point zero-order fit kernel (finalize_zero_order_kernel) goes, at the bench
shape: quadrotor, P = 100 nominal points, N = 1e5 samples per point (C = 25 chunks), partials from one
real accumulate.

A copy of the library built with -DIRS_FINALIZE_PHASES stamps the SM clock and the global timer at each
phase boundary of block 0 (the shipped library has no stamps): start, chunk sums done (thread 0), Gram in
shared memory (after the barrier), nominal done (thread 32, from the Gram barrier on), factor done and
solves done (warp 0), outputs written (thread 0).  The fit is launched --launches times and the stamps are
read back after each; the table gives the median of every phase next to the kernel time from CUDA events
(launches of the shipped build, and of the stamped one, captured in a CUDA graph).

    python tools/finalize_phases.py [--launches 200] [--csrc DIR | --phase-lib SO] [--out FILE]

--csrc builds the stamped library from another source tree; --phase-lib takes one built already.  The
kernel before the stamps existed is measured by checking out the commit before the one that added this
tool and applying tools/finalize_phases_parent.patch there (the same stamps at the same phase
boundaries, nothing else), then passing that tree's irs_mpc_b200/csrc with --csrc.  Needs a GPU.

The tool also reports, from the SASS of the shipped library (cuobjdump), how many partial loads a thread
of the quadrotor kernel issues before its first conversion to fp64: the chunk sum is fast only while the
compiler keeps them together (96 at three entries x 32 chunks; a handful means the adds are interleaved
with the loads again).
"""
import argparse
import ctypes
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PHASES = ["start", "chunk sums", "Gram in smem", "nominal", "factor", "solves", "written"]
T_STEPS, N_SAMPLES, SEED = 100, 100000, 0x1255 + 3


def chunk_loads_before_first_add(lib_path):
    """Longest run of 32-bit global loads before an fp32 -> fp64 conversion in the SASS of
    finalize_zero_order_kernel<Quadrotor<double>,128>, or None without cuobjdump."""
    import re
    try:
        txt = subprocess.run(["cuobjdump", "-sass", lib_path], capture_output=True, text=True, check=True).stdout
    except (OSError, subprocess.SubprocessError):
        return None
    for block in re.split(r"\n\s*Function : ", txt)[1:]:
        if not block.startswith("_ZN3irs26finalize_zero_order_kernelINS_9QuadrotorIdEELi128E"):
            continue
        run = best = 0
        for op in re.findall(r"/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P[0-9T]\s+)?([A-Z0-9_.]+)", block):
            if op == "LDG.E":
                run += 1
            elif op == "F2F.F64.F32":
                best, run = max(best, run), 0
        return best
    return None


def build_phase_lib(csrc, out_dir):
    from irs_mpc_b200 import _lib
    path = os.path.join(out_dir, "libirs_mpc_b200_phases.so")
    cmd = (["nvcc"] + _lib.NVCC_FLAGS + ["-DIRS_FINALIZE_PHASES", "-I", _lib.INCLUDE, "-o", path,
                                         os.path.join(csrc, "api.cu")])
    print(" ".join(cmd), flush=True)
    subprocess.run(cmd, check=True)
    return path


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--csrc", default=None, help="source tree of the stamped build (default: this one)")
    ap.add_argument("--phase-lib", default=None, help="a library built with -DIRS_FINALIZE_PHASES")
    ap.add_argument("--out", default=None, help="also write the table here")
    ap.add_argument("--label", default="")
    args = ap.parse_args()

    import torch
    assert torch.cuda.is_available(), "finalize_phases needs a GPU"
    from irs_mpc_b200 import _lib, smoothing
    from irs_mpc_b200 import example_configs as ec
    from irs_mpc_b200.all import GaussianSampling, IrsLqrParameters, IrsLqrZeroOrder, QuadrotorDynamics
    from irs_mpc_b200 import _device

    tmp = tempfile.mkdtemp(prefix="irs_finalize_phases_")
    phase_path = args.phase_lib or build_phase_lib(args.csrc or _lib.CSRC, tmp)
    shipped = _lib.MAIN
    stamped = _lib.Library.at(phase_path)
    read_stamps = ctypes.CDLL(os.path.abspath(phase_path)).irs_finalize_phases
    read_stamps.argtypes = [ctypes.POINTER(ctypes.c_ulonglong)]

    cfg = ec.quadrotor(T=T_STEPS)
    system = QuadrotorDynamics(cfg["h"])
    params = IrsLqrParameters()
    for key in ("Q", "Qd", "R", "x0", "xd_trj", "u_trj_initial", "xbound", "ubound"):
        setattr(params, key, cfg[key])
    sampler = GaussianSampling(cfg["sigma"][:12], cfg["sigma"][12:], N_SAMPLES, power=cfg.get("power", 0.5), seed=SEED)
    solver = IrsLqrZeroOrder(system, params, sampler)
    x_nom = _device.to_device(solver.x_trj[:T_STEPS])
    u_nom = _device.to_device(solver.u_trj)
    ws = smoothing.Workspace(system, smoothing.ZERO_ORDER, T_STEPS, N_SAMPLES)
    smoothing.accumulate(system, smoothing.ZERO_ORDER, x_nom, u_nom, N_SAMPLES, ws, sigma=sampler.sigma(1),
                         seed=SEED, it=1, flags=sampler.flags())
    torch.cuda.synchronize()

    def fit(lib):
        system.lib = lib
        smoothing.finalize(system, smoothing.ZERO_ORDER, x_nom, u_nom, ws, N_SAMPLES)

    def event_us(lib, launches):
        """Kernel time per launch: `launches` fits captured in one CUDA graph (a host loop of ctypes
        launches would time the host), replayed between two events."""
        for _ in range(10):
            fit(lib)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for _ in range(launches):
                fit(lib)
        graph.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        graph.replay()
        e1.record()
        torch.cuda.synchronize()
        return 1e3 * e0.elapsed_time(e1) / launches

    # the stamped build computes what the shipped one does
    fit(shipped)
    ref = [t.clone() for t in (ws.At, ws.Bt, ws.ct, ws.status)]
    fit(stamped)
    torch.cuda.synchronize()
    same = all(torch.equal(a, b) for a, b in zip(ref, (ws.At, ws.Bt, ws.ct, ws.status)))

    K = len(PHASES)
    buf = (ctypes.c_ulonglong * (2 * K))()
    clk, ns = [], []
    for _ in range(args.launches):
        fit(stamped)
        torch.cuda.synchronize()
        assert read_stamps(buf) == 0
        v = np.array(buf[:], dtype=np.int64)
        clk.append(v[:K] - v[0])
        ns.append(v[K:] - v[K])
    clk, ns = np.array(clk), np.array(ns)
    ghz = float(np.median(clk[:, -1] / np.maximum(ns[:, -1], 1)))
    us_shipped = event_us(shipped, args.launches)
    us_stamped = event_us(stamped, args.launches)
    system.lib = shipped

    name = torch.cuda.get_device_name(0)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=20).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        smi = "n/a"
    med = np.median(clk, axis=0)
    lines = ["finalize_zero_order_kernel<Quadrotor<double>,128> phases %s" % args.label,
             "device: %s | power limit, SM clock, max SM clock: %s | clock from the stamps: %.3f GHz" % (name, smi, ghz),
             "shape: P=%d points, N=%d, C=%d chunks, width %d; %d launches; stamped build bit-identical to shipped: %s"
             % (T_STEPS, N_SAMPLES, ws.C, ws.width, args.launches, same),
             "",
             "%-14s %12s %12s %12s %10s" % ("boundary", "cycles", "phase cyc", "phase us", "p90 cyc")]
    prev_main = 0.0
    for k, label in enumerate(PHASES):
        if label == "nominal":      # runs beside the factor, from the Gram barrier on
            ph = clk[:, k] - clk[:, PHASES.index("Gram in smem")]
            lines.append("%-14s %12.0f %12.0f %12.2f %10.0f   (thread 32, from the Gram barrier)"
                         % (label, med[k], np.median(ph), np.median(ph) / ghz / 1e3, np.percentile(clk[:, k], 90)))
            continue
        ph = np.median(clk[:, k] - (clk[:, PHASES.index("Gram in smem")] if label == "factor" else prev_main))
        lines.append("%-14s %12.0f %12.0f %12.2f %10.0f" % (label, med[k], ph, ph / ghz / 1e3, np.percentile(clk[:, k], 90)))
        prev_main = clk[:, k]
    loads = chunk_loads_before_first_add(shipped.path)
    lines += ["",
              "partial loads in flight before the first fp64 add (SASS of the shipped library): %s"
              % ("not checked (no cuobjdump)" if loads is None else loads),
              "block 0, start -> written: %.2f us (median)" % (med[-1] / ghz / 1e3),
              "kernel time, CUDA events over one graph of %d launches: shipped %.2f us, stamped %.2f us"
              % (args.launches, us_shipped, us_stamped)]
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
