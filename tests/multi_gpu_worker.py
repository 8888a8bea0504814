"""Multi-GPU equivalence checks on real GPUs, one rank per GPU.  Run by tests/test_multi_gpu.py (which
skips on a single-GPU box) or by hand:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29520 tests/multi_gpu_worker.py

 1. timestep sharding (ShardedLinearizer.linearize_t) reproduces the single-GPU linearization bit for bit;
 2. sample sharding (linearize_n, W ranks x N samples) equals ONE GPU drawing the same W*N samples per
    point up to fp32 summation order (1e-5), and is bit-identical on every rank;
 3. the fused peer-memory exchange equals the NCCL all-gather path bit for bit, survives a horizon that
    shrinks and grows again on a live linearizer, and a rank that does not deliver in time raises
    RuntimeError on its peers (never a silent fit on stale blocks);
 4. instance sharding (BatchedIrsLqrZeroOrder with instance_offset) reproduces the unsharded batch bit
    for bit.
Rank 0 prints one line per check.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from irs_mpc_b200 import _device, example_configs as ec, smoothing      # noqa: E402
from irs_mpc_b200.all import BatchedIrsLqrZeroOrder, GaussianSampling, QuadrotorDynamics  # noqa: E402
from irs_mpc_b200.distributed import ShardedLinearizer                   # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
    T, N = 37, 20000                      # T not divisible by the world size on purpose
    cfg = ec.quadrotor(T=T)
    s = QuadrotorDynamics(cfg["h"])
    rng = np.random.default_rng(3)
    x = _device.to_device(0.05 * rng.standard_normal((T, 12)))
    u = _device.to_device(cfg["u_trj_initial"] + 0.05 * rng.standard_normal((T, 4)))
    kw = dict(sigma=cfg["sigma"], seed=99, it=2)
    sh = ShardedLinearizer(s, smoothing.ZERO_ORDER)
    ok = True

    def report(name, passed, detail=""):
        nonlocal ok
        ok = ok and passed
        if rank == 0:
            print("%-34s %s %s" % (name, "PASS" if passed else "FAIL", detail), flush=True)

    # 1. timestep sharding
    A1, B1, c1, st1, _ = smoothing.linearize(s, smoothing.ZERO_ORDER, x, u, N, **kw)
    A1, B1, c1 = A1.clone(), B1.clone(), c1.clone()
    At, Bt, ct, stt = sh.linearize_t(x, u, N, **kw)
    same = torch.equal(At, A1) and torch.equal(Bt, B1) and torch.equal(ct, c1) and int(stt.sum()) == 0
    flags = torch.tensor([1.0 if same else 0.0], device="cuda")
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    report("timestep sharding bit-identical", bool(flags.item() == 1.0), "(T=%d over %d ranks)" % (T, world))
    # the gather fused into the fit kernel (peer memory) against the NCCL all-gather path, repeated steps
    # (output double buffering by epoch parity), and a horizon shorter than the world (ranks without points)
    used_gather = sh._tg is not None
    sh_nccl_t = ShardedLinearizer(s, smoothing.ZERO_ORDER, peer_memory=False)
    ok_t = True
    for rep in range(3):
        Ag, Bg, cg, sg = sh.linearize_t(x, u, N, **kw)
        Ag, Bg, cg = Ag.clone(), Bg.clone(), cg.clone()
        Ac_, Bc_, cc_, sc_ = sh_nccl_t.linearize_t(x, u, N, **kw)
        ok_t = ok_t and torch.equal(Ag, Ac_) and torch.equal(Bg, Bc_) and torch.equal(cg, cc_) and int(sg.sum()) == 0
    Tshort = max(1, world - 1)
    A1s, B1s, c1s, _, _ = smoothing.linearize(s, smoothing.ZERO_ORDER, x[:Tshort].contiguous(), u[:Tshort].contiguous(), N, **kw)
    A1s, c1s = A1s.clone(), c1s.clone()
    Ats, Bts, cts, sts = sh.linearize_t(x[:Tshort].contiguous(), u[:Tshort].contiguous(), N, **kw)
    ok_t = ok_t and torch.equal(Ats, A1s) and torch.equal(cts, c1s) and int(sts.sum()) == 0
    flags = torch.tensor([1.0 if ok_t else 0.0], device="cuda")
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    report("fused gather == NCCL gather", bool(flags.item() == 1.0) and used_gather,
           "(peer memory in use: %s; T=%d and T=%d)" % (used_gather, T, Tshort))

    # 2. sample sharding
    An, Bn, cn, stn = sh.linearize_n(x, u, N, **kw)
    An, Bn, cn = An.clone(), Bn.clone(), cn.clone()
    Aw, Bw, cw, stw, _ = smoothing.linearize(s, smoothing.ZERO_ORDER, x, u, N * world, **kw)

    def rel(a, b):
        return float((a - b).abs().max() / b.abs().max())
    err = max(rel(An, Aw), rel(Bn, Bw))
    gathered = [torch.empty_like(An) for _ in range(world)]
    dist.all_gather(gathered, An)
    identical = all(torch.equal(g, gathered[0]) for g in gathered)
    report("sample sharding vs one GPU", err < 1e-5 and int(stn.sum()) == 0, "(rel err %.2e)" % err)
    report("sample sharding identical on ranks", identical)
    # numpy in / numpy out variant (pinned staging, one copy each way): same bits
    Ah, Bh, ch, sth = sh.linearize_n_numpy(x.cpu().numpy(), u.cpu().numpy(), N, **kw)
    report("linearize_n_numpy == linearize_n", bool((torch.from_numpy(Ah).to(An.device) == An).all())
           and bool((torch.from_numpy(Bh).to(An.device) == Bn).all())
           and bool((torch.from_numpy(ch).to(An.device) == cn).all()) and int(sth.sum()) == 0)
    used_peer = sh._px is not None
    sh_nccl = ShardedLinearizer(s, smoothing.ZERO_ORDER, peer_memory=False)
    Ac, Bc, cc, _ = sh_nccl.linearize_n(x, u, N, **kw)
    same = torch.equal(Ac, An) and torch.equal(Bc, Bn) and torch.equal(cc, cn)
    report("peer-memory exchange == NCCL path", same and used_peer, "(peer memory in use: %s)" % used_peer)
    for k in range(20):                       # epochs / double buffering over repeated steps
        A2, B2, c2, st2 = sh.linearize_n(x, u, N, **kw)
    smoothing.check_status(st2)
    report("peer exchange stable over 20 steps", torch.equal(A2, An) and torch.equal(c2, cn))

    # 2b. a horizon that shrinks and grows again on a LIVE linearizer (shrinking-horizon MPC): the
    #     exchange is reused, the ranks stay in step, and every size still equals the NCCL path
    ok_shape = True
    px_before = sh._px
    for Ts in (11, 5, 23, T):
        As, Bs, cs, sts = sh.linearize_n(x[:Ts].contiguous(), u[:Ts].contiguous(), N, **kw)
        As, Bs, cs = As.clone(), Bs.clone(), cs.clone()
        smoothing.check_status(sts)
        Ar, Br, cr_, _ = sh_nccl.linearize_n(x[:Ts].contiguous(), u[:Ts].contiguous(), N, **kw)
        ok_shape = ok_shape and torch.equal(As, Ar) and torch.equal(Bs, Br) and torch.equal(cs, cr_)
    flags = torch.tensor([1.0 if (ok_shape and sh._px is px_before) else 0.0], device="cuda")
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    report("horizon change on a live exchange", bool(flags.item() == 1.0), "(T = 11, 5, 23, %d; same exchange object)" % T)

    # 2c. a late rank: the others must raise, not fit on stale blocks; the late rank itself still finds
    #     everybody's blocks, and the next step is in step again
    import time
    sh_short = ShardedLinearizer(s, smoothing.ZERO_ORDER, peer_memory=True, peer_timeout_s=0.5)
    sh_short.linearize_n(x, u, N, **kw)       # warm: buffers, rendezvous
    torch.cuda.synchronize()
    dist.barrier()
    raised = False
    if rank == world - 1:
        time.sleep(2.5)
    try:
        Al, Bl, cl, stl = sh_short.linearize_n(x, u, N, **kw)
        smoothing.check_status(stl)
    except RuntimeError as e:
        raised = "peer exchange timed out" in str(e)
    expect = rank != world - 1
    flags = torch.tensor([1.0 if raised == expect else 0.0], device="cuda")
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    report("late rank raises on its peers", bool(flags.item() == 1.0))
    torch.cuda.synchronize()
    dist.barrier()
    Al, Bl, cl, stl = sh_short.linearize_n(x, u, N, **kw)
    smoothing.check_status(stl)
    flags = torch.tensor([1.0 if (torch.equal(Al, An) and torch.equal(cl, cn)) else 0.0], device="cuda")
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    report("exchange recovers after a timeout", bool(flags.item() == 1.0))

    # 4. instance sharding
    I, Tb, Nb = 4 * world, 20, 1000
    cfgb = ec.quadrotor(T=Tb)
    x0 = 0.02 * np.random.default_rng(7).standard_normal((I, 12))
    xd = np.stack([cfgb["xd_trj"] for _ in range(I)])
    smp = GaussianSampling(cfgb["sigma"][:12], cfgb["sigma"][12:], Nb, seed=5)
    full = BatchedIrsLqrZeroOrder(s, cfgb["Q"], cfgb["Qd"], cfgb["R"], x0, xd, cfgb["u_trj_initial"], smp)
    xf, uf, cf = full.local_descent()
    full.check()
    lo, hi = rank * I // world, (rank + 1) * I // world
    part = BatchedIrsLqrZeroOrder(s, cfgb["Q"], cfgb["Qd"], cfgb["R"], x0[lo:hi], xd[lo:hi], cfgb["u_trj_initial"],
                                  smp, instance_offset=lo)
    xp, up, cp = part.local_descent()
    part.check()
    same = torch.equal(xp, xf[lo:hi]) and torch.equal(up, uf[lo:hi]) and torch.equal(cp, cf[lo:hi])
    flags = torch.tensor([1.0 if same else 0.0], device="cuda")
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    report("instance sharding bit-identical", bool(flags.item() == 1.0), "(%d instances over %d ranks)" % (I, world))
    # 5. learned dynamics (tcgen05 network kernel) under both shardings: timestep axis bit-identical to one GPU,
    #    sample axis equal to one GPU drawing all the samples (1e-5) and identical on every rank
    from irs_mpc_b200.all import MlpDynamics
    gm = np.load(os.path.join(ROOT, "tests", "golden", "mlp_pendulum.npz"))
    net = MlpDynamics([(gm["W1"], gm["b1"]), (gm["W2"], gm["b2"]), (gm["W3"], gm["b3"])])
    Tm, Nm = 23, 6000
    xm = _device.to_device(np.cumsum(0.05 * np.ones((Tm, 2)), axis=0))
    um = _device.to_device(0.3 * rng.standard_normal((Tm, 1)))
    kwm = dict(sigma=np.array([1.0, 1.0, 1.0]), seed=17, it=1, flags=8)
    shm = ShardedLinearizer(net, smoothing.ZERO_ORDER)
    A1m, B1m, c1m, _, _ = smoothing.linearize(net, smoothing.ZERO_ORDER, xm, um, Nm, **kwm)
    A1m, B1m, c1m = A1m.clone(), B1m.clone(), c1m.clone()
    Atm, Btm, ctm, sttm = shm.linearize_t(xm, um, Nm, **kwm)
    same_t = torch.equal(Atm, A1m) and torch.equal(Btm, B1m) and torch.equal(ctm, c1m) and int(sttm.sum()) == 0
    Anm, Bnm, cnm, stnm = shm.linearize_n(xm, um, Nm, **kwm)
    Anm, Bnm = Anm.clone(), Bnm.clone()
    Awm, Bwm, _, _, _ = smoothing.linearize(net, smoothing.ZERO_ORDER, xm, um, Nm * world, **kwm)
    errm = max(rel(Anm, Awm), rel(Bnm, Bwm))
    gathered = [torch.empty_like(Anm) for _ in range(world)]
    dist.all_gather(gathered, Anm)
    same_n = all(torch.equal(g, gathered[0]) for g in gathered) and int(stnm.sum()) == 0
    flags = torch.tensor([1.0 if (same_t and same_n and errm < 1e-5) else 0.0], device="cuda")
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    report("learned dynamics sharded", bool(flags.item() == 1.0), "(timestep axis bit-identical: %s, sample axis rel err %.2e)" % (same_t, errm))
    if rank == 0:
        print("ALL PASS" if ok else "FAILURES", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
