"""Fingerprint every fp32 quadrotor sampling path: a SHA-256 of the raw partial blocks the zero-order accumulate
writes (both engines, antithetic and independent draws) at the batched-MPC shape (P = 409,600, N = 1000), the bench
shape (N = 1e5, 25 chunks) and ragged N (odd chunks ending in a lone pair member, partial rounds), and of the fp32
dynamics batch.  Two builds compute the same bits exactly when their fingerprints match:

    IRS_MPC_B200_LIB=build_a/libirs_mpc_b200.so python tools/partials_fingerprint.py --out a.json
    IRS_MPC_B200_LIB=build_b/libirs_mpc_b200.so python tools/partials_fingerprint.py --out b.json
    python tools/partials_fingerprint.py --compare a.json b.json
"""
import argparse
import hashlib
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def digest(t):
    from irs_mpc_b200 import _device
    return hashlib.sha256(np.ascontiguousarray(_device.to_numpy(t)).tobytes()).hexdigest()


def fingerprints():
    import torch
    from irs_mpc_b200 import _device, _lib, sampling, smoothing
    from irs_mpc_b200.all import QuadrotorDynamics
    from oracle import example_configs as ec

    cfg = ec.quadrotor()
    s = QuadrotorDynamics(cfg["h"])
    n, m = s.dim_x, s.dim_u
    sig = np.asarray(cfg["sigma"], dtype=np.float64)
    rng = np.random.default_rng(5)
    out = {}

    def nominal(P):
        x = np.asarray(cfg["x0"], dtype=np.float64) + 0.3 * rng.standard_normal((P, n))
        u = np.asarray(cfg["u_trj_initial"][0], dtype=np.float64) + 0.3 * rng.standard_normal((P, m))
        return _device.to_device(x), _device.to_device(u)

    cases = [(409600, 1000, 0), (2, 100000, 0), (3, 4097, 256)] + [(3, N, 0) for N in (1, 33, 257, 8193)]
    for eng in (1, 0):
        _lib.call("irs_set_gram_engine", eng)
        for antithetic in (True, False):
            for P, N, chunk in cases:
                xd, ud = nominal(P)
                sampler = sampling.GaussianSampling(sig[:n], sig[n:], N, power=cfg["power"], seed=99,
                                                    antithetic=antithetic)
                ws = smoothing.Workspace(s, smoothing.ZERO_ORDER, P, N, chunk)
                smoothing.accumulate(s, smoothing.ZERO_ORDER, xd, ud, N, ws, sigma=sampler.sigma(3), seed=99, it=3,
                                     flags=sampler.flags())
                torch.cuda.synchronize()
                out["engine%d antithetic=%d P=%d N=%d S=%d" % (eng, antithetic, P, N, ws.S)] = digest(ws.partials)
    _lib.call("irs_set_gram_engine", -1)
    x = rng.standard_normal((1 << 20, n)).astype(np.float32)
    u = rng.standard_normal((1 << 20, m)).astype(np.float32)
    f = s._run_dynamics(x, u, False, dtype=torch.float32)
    out["dynamics_batch_f32"] = hashlib.sha256(np.ascontiguousarray(f).tobytes()).hexdigest()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--compare", nargs=2)
    args = ap.parse_args()
    if args.compare:
        a, b = (json.load(open(p)) for p in args.compare)
        bad = [k for k in sorted(set(a) | set(b)) if a.get(k) != b.get(k)]
        for k in sorted(a):
            print("%-8s %s" % ("DIFFERS" if k in bad else "same", k))
        sys.exit(1 if bad else 0)
    fp = fingerprints()
    print(json.dumps(fp, indent=1))
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(fp, fh, indent=1)


if __name__ == "__main__":
    main()
