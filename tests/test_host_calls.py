"""The *_host entry points: arguments are checked before anything runs, every call runs on the handle's private stream
(so host calls and device solves on other streams of one handle keep their order), and the staging of a call's
arrays -- packed through pinned memory for small batches, array by array for large ones -- gives the same results."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _net(hidden, seed):
    import torch
    torch.manual_seed(seed)
    dims = [6] + list(hidden) + [1]
    layers = [torch.nn.Linear(dims[i], dims[i + 1], dtype=torch.double) for i in range(len(dims) - 1)]
    return dict(weights=[(l.weight.detach().numpy().copy(), l.bias.detach().numpy().copy()) for l in layers],
                Wn=np.eye(6), mu_f=np.zeros(6), sigma_t=1.0, mu_t=0.0)


def _batch(B, seed):
    from igt_mpc_int_b200 import scenarios as S
    pb = S.mid_episode(B, N=40, seed=seed)
    u = np.random.default_rng(seed).uniform(-0.3, 0.3, size=(B, 40, 2))
    return dict(x0=pb.x0, u_prev=pb.u_prev, curv=pb.curv, obs=pb.obs, nn_ctx=pb.nn_ctx, u=u)


def test_rollout_host_with_A_and_no_Bm_is_rejected():
    from igt_mpc_int_b200.planner import BatchSolver
    s = BatchSolver(N=40)
    B = 4
    z0 = np.zeros((B, 7), np.float32); u = np.zeros((B, 40, 2), np.float32); curv = np.zeros((B, 3), np.float32)
    z = np.empty((B, 41, 7), np.float32); A = np.empty((B, 40, 7, 7), np.float32)
    vp = lambda a: C.c_void_p(a.ctypes.data)
    n0 = s.launches
    rc = s.lib.igt_rollout_host(s._h, B, vp(z0), vp(u), vp(curv), vp(z), vp(A), None, 0)
    assert rc == -1 and b"bad argument" in s.lib.igt_last_error(s._h)
    assert s.launches == n0
    s.close()


def test_host_calls_interleaved_with_device_solves_on_a_side_stream():
    """evaluate, mlp_value and rollout share the handle's value-term scratch and staging with the device solves; run
    between solves queued on another stream they must give what the same calls give one after the other"""
    import torch
    from igt_mpc_int_b200.planner import BatchSolver
    s = BatchSolver(N=40, mlp=_net((160, 64), 3))              # wider than 128: per-thread value term, scratch in HBM
    b = _batch(4096, 11)
    d = {k: torch.from_numpy(np.ascontiguousarray(b[k])).cuda() for k in ("x0", "u_prev", "curv", "obs", "nn_ctx")}
    z0 = b["x0"].astype(np.float32); uf = b["u"].astype(np.float32); cf = b["curv"].astype(np.float32)

    def solve():
        return s.solve_batch_device(d["x0"], d["u_prev"], d["curv"], d["obs"], nn_ctx=d["nn_ctx"])

    def host_calls():
        return (s.evaluate(b["x0"], b["u_prev"], b["curv"], b["obs"], b["u"], nn_ctx=b["nn_ctx"]),
                s.mlp_value(b["x0"][:, 2], b["x0"][:, 5], b["nn_ctx"], tensor_cores=0),
                s.rollout(z0, uf, cf, jac=True))

    ref_solve = solve()
    torch.cuda.synchronize()
    ref_host = host_calls()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        first = solve()
        mid = host_calls()
        second = solve()
    side.synchronize()
    for out in (first, second):
        for k in ref_solve:
            assert np.array_equal(out[k].cpu().numpy(), ref_solve[k].cpu().numpy(), equal_nan=True), k
    ev, mv, ro = mid
    for k in ("cost", "viol", "x"):
        assert np.array_equal(ev[k], ref_host[0][k], equal_nan=True), k
    assert np.array_equal(mv, ref_host[1], equal_nan=True)
    for a, r in zip(ro, ref_host[2]):
        assert np.array_equal(a, r, equal_nan=True)
    s.close()


def test_bank_calls_above_and_below_the_packing_threshold_agree():
    """a batch whose arrays take more than 1 MiB is copied array by array, a small one through one pinned block"""
    from igt_mpc_int_b200.planner import BatchSolver
    s = BatchSolver(N=40, mlp=[_net((64, 32), 1), None, _net((48,), 2)])
    big = _batch(2048, 21)
    B = 16384
    rng = np.random.default_rng(4)
    sN, vN, ctx = rng.uniform(0, 60, B), rng.uniform(0, 12, B), rng.uniform(-1, 1, (B, 4))
    ni = np.where(np.arange(B) % 3 == 1, 2, 0).astype(np.int32)
    n = 64                                                        # well below 1 MiB for both calls
    e_big = s.evaluate(big["x0"], big["u_prev"], big["curv"], big["obs"], big["u"], nn_ctx=big["nn_ctx"], net_idx=ni[:2048])
    e_small = s.evaluate(big["x0"][:n], big["u_prev"][:n], big["curv"][:n], big["obs"][:n], big["u"][:n],
                         nn_ctx=big["nn_ctx"][:n], net_idx=ni[:n])
    for k in ("cost", "viol", "x"):
        assert np.array_equal(e_big[k][:n], e_small[k], equal_nan=True), k
    m_big = s.mlp_value(sN, vN, ctx, tensor_cores=0, net_idx=ni)
    m_small = s.mlp_value(sN[:n], vN[:n], ctx[:n], tensor_cores=0, net_idx=ni[:n])
    assert np.array_equal(m_big[:n], m_small, equal_nan=True)
    s.close()
