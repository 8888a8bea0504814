"""Where the time of a sample-sharded step goes (tuning aid; run under torchrun, one rank per GPU):
kernel alone, local finalize, fused peer finalize (eager / graph), NCCL path."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from irs_mpc_b200 import _device, _graph, example_configs as ec, smoothing      # noqa: E402
from irs_mpc_b200.all import QuadrotorDynamics                                  # noqa: E402
from irs_mpc_b200.distributed import ShardedLinearizer                          # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
    T = 100
    N = int(os.environ.get("MT_N", "100000"))
    cfg = ec.quadrotor(T=T)
    s = QuadrotorDynamics(cfg["h"])
    x = _device.to_device(np.zeros((T, 12)))
    u = _device.to_device(cfg["u_trj_initial"])
    kw = dict(sigma=cfg["sigma"], it=1, flags=8)
    ws = smoothing.Workspace(s, 0, T, N)

    def timed(fn, steps=40, warm=6):
        for k in range(warm):
            fn(k)
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(steps):
            fn(warm + k)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device="cuda")
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def acc(k):
        smoothing.accumulate(s, 0, x, u, N, ws, seed=k, i0=rank * N, **kw)

    def local(k):
        acc(k)
        smoothing.finalize(s, 0, x, u, ws, N)

    res = {"accumulate": timed(acc), "accumulate+local finalize": timed(local)}
    for graphs in (False, True):
        _graph.USE_GRAPHS = graphs
        sh = ShardedLinearizer(s, 0, peer_memory=True)
        res["fused peer finalize, graphs=%s" % graphs] = timed(lambda k: sh.linearize_n(x, u, N, seed=k, **kw))
    _graph.USE_GRAPHS = True
    shn = ShardedLinearizer(s, 0, peer_memory=False)
    res["NCCL all-gather path"] = timed(lambda k: shn.linearize_n(x, u, N, seed=k, **kw))
    _graph.USE_GRAPHS = True
    sht = ShardedLinearizer(s, 0, peer_memory=True)
    res["timestep axis, fused gather"] = timed(lambda k: sht.linearize_t(x, u, N * world, seed=k, **kw))
    shtn = ShardedLinearizer(s, 0, peer_memory=False)
    res["timestep axis, NCCL gather"] = timed(lambda k: shtn.linearize_t(x, u, N * world, seed=k, **kw))
    if rank == 0:
        for k, v in res.items():
            print("%-40s %.4f ms" % (k, v), flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
