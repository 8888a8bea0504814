"""Time the run-time-dimension TVLQR entries (csrc/tvlqr_any.cuh) on the GPU and print one JSON line.

- irs_tvlqr_riccati_any at (4,1), (6,3), (8,4), (16,8), (32,8), (32,32);
- irs_tvlqr_riccati_any against irs_tvlqr_riccati (the tuned kernels, default dispatch) at the built-in pairs, and
  at I = 1 against the generic block kernel tvlqr_riccati_kernel<n,m,256> (both also writing H^-1 and P);
- irs_tvlqr_box_qp_any on make_problem(4, 1, 100, "input") of oracle/box_kkt.py.

T = 100, I in {1, 64, 1024, 4096}.  Each time is the median over `--calls` calls (default 50) of the CUDA-event
time of one call, after `--warmup` untimed calls of the same shape.  Inputs are random "dense"-weight problems
as in tests/test_lqr_kernels.py; their size at I = 4096 (up to 3.4 GB at n = 32) exceeds the L2 cache.

    python tools/tvlqr_any_bench.py [--calls 50] [--warmup 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NEW = [(4, 1), (6, 3), (8, 4), (16, 8), (32, 8), (32, 32)]
BUILTIN = [(2, 1), (5, 2), (6, 2), (12, 4)]
COUNTS = [1, 64, 1024, 4096]
T = 100


def spd(rng, d, lo=0.5):
    M = rng.standard_normal((d, d))
    return M.dot(M.T) / d + lo * np.eye(d)


def device_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        power, clock = (s.strip() for s in out.split(","))
    except Exception as e:      # the timing stands without it, but say so
        power, clock = "unknown (%s)" % e, "unknown"
    return name, power, clock


def time_calls(fn, calls, warmup):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(calls):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms))


def riccati_timer(n, m, I, entry, seed=0, hessians=False):
    from irs_mpc_b200 import _device, _lib
    rng = np.random.default_rng(seed)
    up = _device.to_device
    At = up(np.eye(n) + 0.1 * rng.standard_normal((I, T, n, n)))
    Bt = up(0.3 * rng.standard_normal((I, T, n, m)))
    ct = up(0.1 * rng.standard_normal((I, T, n)))
    xd = up(rng.standard_normal((I, T + 1, n)))
    Q, Qd, R = up(spd(rng, n)), up(10 * spd(rng, n)), up(spd(rng, m))
    K, k = _device.empty((I, T, m, n)), _device.empty((I, T, m))
    import torch
    status = _device.empty((I,), torch.int32)
    head = (n, m, _device.ptr(At), _device.ptr(Bt), _device.ptr(ct), _device.ptr(Q), _device.ptr(Qd), _device.ptr(R),
            _device.ptr(xd), (T + 1) * n, I, T, _device.ptr(K), _device.ptr(k), _device.ptr(status))
    if hessians:      # irs_tvlqr_riccati_any or irs_tvlqr_riccati_ex, writing H^-1 and P as well
        Hinv, P = _device.empty((I, T, m, m)), _device.empty((I, T + 1, n, n))
        args = head + (_device.ptr(Hinv), _device.ptr(P), _device.stream_ptr())
    elif entry == "irs_tvlqr_riccati_any":
        args = head + (None, None, _device.stream_ptr())
    else:
        args = head + (_device.stream_ptr(),)

    def call():
        _lib.call(entry, *args)
    call()
    torch.cuda.synchronize()
    assert int(status.abs().sum().item()) == 0, (entry, n, m, I)
    return call


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("tvlqr_any_bench: needs a GPU")
    import irs_mpc_b200.all  # noqa: F401
    from irs_mpc_b200 import tv_lqr, _device
    from oracle import box_kkt as bk
    name, power, clock = device_info()
    res = {"device": name, "power_limit": power, "max_sm_clock": clock, "T": T, "calls": args.calls,
           "warmup": args.warmup, "unit": "ms per call (median)", "riccati_any": {}, "builtin_pairs": {}}
    for n, m in NEW:
        res["riccati_any"]["%d,%d" % (n, m)] = {
            str(I): round(time_calls(riccati_timer(n, m, I, "irs_tvlqr_riccati_any"), args.calls, args.warmup), 5)
            for I in COUNTS}
    for n, m in BUILTIN:
        row = {}
        for I in COUNTS:
            t_any = time_calls(riccati_timer(n, m, I, "irs_tvlqr_riccati_any"), args.calls, args.warmup)
            t_tuned = time_calls(riccati_timer(n, m, I, "irs_tvlqr_riccati"), args.calls, args.warmup)
            row[str(I)] = {"any": round(t_any, 5), "tuned": round(t_tuned, 5), "ratio": round(t_any / t_tuned, 3)}
        # like for like at I = 1: the generic block kernel tvlqr_riccati_kernel<n, m, 256> (IRS_TVLQR_VARIANT=block;
        # irs_tvlqr_riccati_ex, so that the even pairs reach it too) against the run-time kernel, both writing H^-1, P
        os.environ["IRS_TVLQR_VARIANT"] = "block"
        t_gen = time_calls(riccati_timer(n, m, 1, "irs_tvlqr_riccati_ex", hessians=True), args.calls, args.warmup)
        del os.environ["IRS_TVLQR_VARIANT"]
        t_any = time_calls(riccati_timer(n, m, 1, "irs_tvlqr_riccati_any", hessians=True), args.calls, args.warmup)
        row["1_with_hessians"] = {"any": round(t_any, 5), "generic_block_256": round(t_gen, 5),
                                  "ratio": round(t_any / t_gen, 3)}
        res["builtin_pairs"]["%d,%d" % (n, m)] = row
    # one bounded QP (penalty-augmented Riccati pass + ADMM) as solve_tvlqr runs it
    p = bk.make_problem(4, 1, T, "input", "dense", I=1, seed=4)
    d = {key: _device.to_device(np.ascontiguousarray(p[key])) for key in ("At", "Bt", "ct", "xd", "x0", "Q", "Qd", "R")}
    out = {}

    def box():
        out["r"] = tv_lqr.box_qp_any_device(d["At"], d["Bt"], d["ct"], d["Q"], d["Qd"], d["R"], p["Q"], p["Qd"], p["R"],
                                            d["xd"], (T + 1) * 4, d["x0"], p["xlo"], p["xhi"], p["ulo"], p["uhi"])
    t_box = time_calls(box, max(5, args.calls // 5), 2)
    res["box_qp_any_4_1_input"] = {"ms": round(t_box, 4), "calls": max(5, args.calls // 5),
                                   "admm_iterations": int(out["r"][3][0].item()), "status": int(out["r"][2][0].item())}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
