"""Worker wire protocol (SURVEY.md section 8(f)-4; reference: zmq_parallel_cmp/array_io.py:6-26,
examples/planar_hand/planar_hand_worker.py:19-80, irs_lqr/irs_lqr_quasistatic.py:118-126, 228-263).
CPU: the framing round-trips and is byte compatible with the reference's array_io.  GPU: a GpuLinearizationWorker
thread answers the solver-side task loop; the blocks equal the direct linearization bit for bit, whatever the
stride."""
import threading

import numpy as np
import pytest

zmq = pytest.importorskip("zmq")


def _pair(ctx, name):
    a, b = ctx.socket(zmq.PUSH), ctx.socket(zmq.PULL)
    a.bind("inproc://" + name)
    b.connect("inproc://" + name)
    return a, b


def test_framing_round_trip():
    from irs_mpc_b200 import worker
    ctx = zmq.Context.instance()
    tx, rx = _pair(ctx, "rt")
    A = np.arange(24, dtype=np.float64).reshape(4, 6) * 0.5
    worker.send_array(tx, A, t=[3, 4, 5, 6], n_samples=100, std=[0.1, 0.2])
    B, t, n_samples, std = worker.recv_array(rx)
    np.testing.assert_array_equal(A, B)
    assert B.dtype == np.float64 and t == [3, 4, 5, 6] and n_samples == 100 and std == [0.1, 0.2]
    C = np.ones((2, 3, 5), dtype=np.float32)[:, ::-1]          # non-contiguous input is sent as its contiguous copy
    worker.send_array(tx, C, t=[0, 1], n_samples=-1, std=[-1])
    D, t, n_samples, std = worker.recv_array(rx)
    np.testing.assert_array_equal(C, D)
    assert D.dtype == np.float32 and (t, n_samples, std) == ([0, 1], -1, [-1])
    tx.close(0)
    rx.close(0)


def test_framing_is_byte_compatible_with_the_reference():
    """The reference's message (zmq_parallel_cmp/array_io.py:6-26) is two frames: pyzmq's send_json of
    dict(dtype=str(A.dtype), shape=A.shape, t=t, n_samples=n_samples, std=std), then the raw C-order array.
    The frames below are those bytes, so the check needs nothing outside this repository."""
    from irs_mpc_b200 import worker
    ctx = zmq.Context.instance()
    tx, rx = _pair(ctx, "compat")
    A = np.random.default_rng(0).standard_normal((5, 7))
    worker.send_array(tx, A, t=[0, 1, 2, 3, 4], n_samples=50, std=[0.3])
    header, payload = rx.recv_multipart()                      # the frames the reference's recv_array parses
    assert header == b'{"dtype": "float64", "shape": [5, 7], "t": [0, 1, 2, 3, 4], "n_samples": 50, "std": [0.3]}'
    assert payload == A.tobytes()
    tx.send_multipart([b'{"dtype": "float64", "shape": [5, 7], "t": [9], "n_samples": -1, "std": [-1]}',
                       (A * 2).tobytes()])                     # and we read what the reference's send_array sends
    B, t, n_samples, std = worker.recv_array(rx)
    np.testing.assert_array_equal(A * 2, B)
    assert (t, n_samples, std) == ([9], -1, [-1])
    tx.close(0)
    rx.close(0)


def test_contiguous_runs():
    from irs_mpc_b200.worker import contiguous_runs
    assert contiguous_runs([]) == []
    assert contiguous_runs([4]) == [(0, 1)]
    assert contiguous_runs([0, 1, 2, 3]) == [(0, 4)]
    assert contiguous_runs([5, 6, 9, 10, 11, 2]) == [(0, 2), (2, 3), (5, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode,stride", [("zero_order_AB", 7), ("zero_order_AB", 3), ("first_order", 5), ("exact", 4)])
def test_gpu_worker_answers_the_solver_loop(mode, stride):
    import torch
    assert torch.cuda.is_available()
    import irs_mpc_b200.all as api
    from irs_mpc_b200 import example_configs as ec, worker
    T, N = 20, 2000
    cfg = ec.quadrotor(T=T)
    system = api.QuadrotorDynamics(cfg["h"])
    rng = np.random.default_rng(1)
    x_trj = 0.1 * rng.standard_normal((T + 1, 12))
    u_trj = cfg["u_trj_initial"] + 0.1 * rng.standard_normal((T, 4))
    std_x, std_u = 0.05, [0.1, 0.2, 0.1, 0.2]
    ctx = zmq.Context.instance()
    sender, receiver = ctx.socket(zmq.PUSH), ctx.socket(zmq.PULL)       # the solver side binds (quasistatic.py:118-126)
    port_tasks = sender.bind_to_random_port("tcp://127.0.0.1")
    port_results = receiver.bind_to_random_port("tcp://127.0.0.1")
    w = worker.GpuLinearizationWorker(system, mode=mode, std_x=std_x, seed=42,
                                      pull_addr="tcp://127.0.0.1:%d" % port_tasks,
                                      push_addr="tcp://127.0.0.1:%d" % port_results)
    n_tasks = -(-T // stride)
    errors = []

    def run():
        try:
            torch.cuda.set_device(0)
            w.serve(max_tasks=n_tasks)
        except Exception as e:      # surfaced below
            errors.append(e)
    th = threading.Thread(target=run)
    th.start()
    try:
        receiver.RCVTIMEO = 60000
        At, Bt = worker.linearize_with_workers(sender, receiver, x_trj, u_trj, N, std_u, stride)
    finally:
        th.join(timeout=60)
        sender.close(0)
        receiver.close(0)
    assert not errors and w.tasks_done == n_tasks
    direct = worker.GpuLinearizationWorker(system, mode=mode, std_x=std_x, seed=42).calc_AB_batch(
        x_trj[:T], u_trj, N, std_u)
    np.testing.assert_array_equal(At, direct[:, :, :12])      # independent of the stride: global point index in Philox
    np.testing.assert_array_equal(Bt, direct[:, :, 12:])
    # and equal to the IrsLqr call surface with the same noise stream
    p = api.IrsLqrParameters()
    p.Q, p.Qd, p.R, p.x0, p.xd_trj, p.u_trj_initial = cfg["Q"], cfg["Qd"], cfg["R"], x_trj[0], cfg["xd_trj"], u_trj
    p.xbound, p.ubound = cfg["xbound"], cfg["ubound"]
    if mode == "exact":
        ref = api.IrsLqrExact(system, p).get_TV_matrices(x_trj, u_trj)
    else:
        smp = api.GaussianSampling(np.full(12, std_x), np.asarray(std_u), N, power=0.5, seed=42)
        cls = api.IrsLqrZeroOrder if mode == "zero_order_AB" else api.IrsLqrFirstOrder
        ref = cls(system, p, smp).get_TV_matrices(x_trj, u_trj)
    np.testing.assert_array_equal(At, ref[0])
    np.testing.assert_array_equal(Bt, ref[1])
