"""The latency path (igt_set_option "latency_path", on by default) in gt_mpc: batches of at most one problem per SM
with a value term run solve_small_kernel -- one CTA per problem, its workspace in shared memory -- and give the
throughput kernel's results bit for bit.  Cooperative value term (circle mode, fp64, layers <= 128 wide; one network
or a bank) and per-thread value term (OBCA, fp32, wider networks).  Not offered: the tensor-core value term
(tensor_core_mlp = 1), and horizons whose workspace and value-term buffers exceed a block's shared memory."""
import re

import numpy as np
import pytest

from igt_mpc_int_b200 import _lib, episode
from igt_mpc_int_b200 import scenarios as S
from tests.test_mlp_bank import _wide_net
from tests.test_value_nets import shipped_net

pytestmark = pytest.mark.gpu

KEYS = ("status", "iters", "cost", "viol", "u", "x")
# largest horizons (n_cinf = 74) whose cooperative solve fits the B200's 227 KB of shared memory per block
N_FIT_COOP, N_FIT_COOP_BANK = 45, 44


def _net(k):
    return shipped_net(k)[0]


# mode -> solver arguments and how its problems are posed
MODES = {
    "coop_sc1": dict(mlp=lambda: _net(1)),
    "coop_sc3": dict(mlp=lambda: _net(3)),
    "coop_bank": dict(mlp=lambda: [_net(1), _net(3), _net(6)], bank=True),
    "obca": dict(mlp=lambda: _net(1), d_min=0.0, obca=True),
    "obca_bank": dict(mlp=lambda: [_net(1), _net(3), _net(6)], d_min=0.0, obca=True, bank=True),
    "f32": dict(mlp=lambda: _net(1), precision="f32"),
    "wide": dict(mlp=lambda: _wide_net((160,), 1)),
    "wide_bank": dict(mlp=lambda: [_wide_net((160,), 1), _wide_net((144, 144), 2)], bank=True),
    "f32_bank": dict(mlp=lambda: [_net(1), _net(3), _net(6)], precision="f32", bank=True),
    "coop_N10": dict(mlp=lambda: _net(1), N=10),
}


def _solver(mode, N=None):
    from igt_mpc_int_b200.planner import BatchSolver
    m = MODES[mode]
    kw = {k: m[k] for k in ("d_min", "precision") if k in m}
    return BatchSolver(N=N or m.get("N", 40), mlp=m["mlp"](), **kw)


_PROBLEMS = {}


def _problems(N):
    if N not in _PROBLEMS:
        _PROBLEMS[N] = S.mid_episode(152, N=N, seed=31)
    return _PROBLEMS[N]


def _args(mode, B, N=None):
    m = MODES[mode]
    pb = _problems(N or m.get("N", 40))
    a = dict(x0=pb.x0[:B], u_prev=pb.u_prev[:B], curv=pb.curv[:B], obs_xy=pb.obs[:B], nn_ctx=pb.nn_ctx[:B])
    if m.get("obca"):
        a["obs_psi"] = pb.obs_psi[:B]
    if m.get("bank"):
        a["net_idx"] = ((pb.scenario[:B] - 1) % len(m["mlp"]())).astype(np.int32)   # every network of the bank in one batch
    return {k: np.ascontiguousarray(v) for k, v in a.items()}


def _n_sm():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _assert_same(r, o, what):
    for k in KEYS:
        assert np.array_equal(r[k], o[k], equal_nan=True), (what, k)


@pytest.mark.parametrize("mode", list(MODES))
def test_latency_path_bit_identical_to_throughput_kernel(mode):
    s = _solver(mode)
    for B in (1, 2, 33, _n_sm()):
        a = _args(mode, B)
        s.set_option("latency_path", 0)
        cold0 = s.solve_batch(**a)
        ui = np.nan_to_num(cold0["u"])
        warm0 = s.solve_batch(**a, u_init=ui)
        s.set_option("latency_path", 1)
        cold1 = s.solve_batch(**a)
        warm1 = s.solve_batch(**a, u_init=ui)
        _assert_same(cold1, cold0, (mode, B, "cold"))
        _assert_same(warm1, warm0, (mode, B, "warm"))
        if B >= 33:
            assert np.mean(cold1["status"] == 0) > 0.5, (mode, B)
    s.close()


def _kernels(fn):
    """names of the CUDA kernels fn() launches (torch.profiler, CUDA activities)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.key for e in prof.key_averages()]


def _ran(names):
    small = any(re.search(r"\bsolve_small_kernel\b", n) for n in names)
    throughput = any(re.search(r"\bsolve_kernel\b", n) for n in names)
    return small, throughput


@pytest.mark.parametrize("mode", list(MODES))
def test_latency_path_is_the_kernel_that_runs(mode):
    s = _solver(mode)
    a = _args(mode, 2)
    for flag, want in ((1, (True, False)), (0, (False, True))):
        s.set_option("latency_path", flag)
        assert _ran(_kernels(lambda: s.solve_batch(**a))) == want, (mode, flag)
    s.close()


def test_tensor_core_value_term_stays_on_the_throughput_kernel():
    s = _solver("coop_sc1")
    s.set_option("tensor_core_mlp", 1)
    s.set_option("latency_path", 1)
    assert _ran(_kernels(lambda: s.solve_batch(**_args("coop_sc1", 2)))) == (False, True)
    s.close()


@pytest.mark.parametrize("mode,n_fit", [("coop_sc1", N_FIT_COOP), ("coop_bank", N_FIT_COOP_BANK)])
def test_cooperative_latency_path_horizon_limit(mode, n_fit):
    """up to n_fit the cooperative solve fits shared memory; one step more and it falls back to the throughput kernel,
    with the same results either way"""
    for N, small in ((n_fit, True), (n_fit + 1, False)):
        s = _solver(mode, N=N)
        a = _args(mode, 2, N=N)
        s.set_option("latency_path", 1)
        assert _ran(_kernels(lambda: s.solve_batch(**a))) == (small, not small), (mode, N)
        r1 = s.solve_batch(**a)
        s.set_option("latency_path", 0)
        _assert_same(r1, s.solve_batch(**a), (mode, N))
        s.close()


@pytest.mark.parametrize("obca", [False, True])
def test_bad_bank_index_on_the_device_entry(obca):
    """an index outside the bank or naming an empty slot, on the latency path: status 7 and NaN for that problem, the
    other problems solved as by the throughput kernel"""
    import torch
    from igt_mpc_int_b200.planner import BatchSolver
    s = BatchSolver(N=40, mlp=[_net(1), None, _net(3)], d_min=0.0 if obca else 5.6)   # slots 1 and 3..7 empty
    a = _args("obca_bank" if obca else "coop_bank", 33)
    good = np.where(a["net_idx"] == 1, 2, a["net_idx"]).astype(np.int32)
    d = lambda v: torch.from_numpy(np.ascontiguousarray(v)).cuda()
    for bad in (-1, 8, 1):
        ni = good.copy()
        ni[17] = bad
        out = {}
        for flag in (1, 0):
            s.set_option("latency_path", flag)
            if flag == 1:
                assert _ran(_kernels(lambda: s.solve_batch_device(
                    d(a["x0"]), d(a["u_prev"]), d(a["curv"]), d(a["obs_xy"]), nn_ctx=d(a["nn_ctx"]),
                    obs_psi=d(a["obs_psi"]) if obca else None, net_idx=d(ni)))) == (True, False)
            o = s.solve_batch_device(d(a["x0"]), d(a["u_prev"]), d(a["curv"]), d(a["obs_xy"]), nn_ctx=d(a["nn_ctx"]),
                                     obs_psi=d(a["obs_psi"]) if obca else None, net_idx=d(ni))
            torch.cuda.synchronize()
            out[flag] = {k: v.cpu().numpy() for k, v in o.items()}
        _assert_same(out[1], out[0], ("bad index", bad))
        o = out[1]
        assert o["status"][17] == _lib.STATUS_BAD_NET and o["iters"][17] == 0
        assert np.all(np.isnan(o["x"][17])) and np.all(np.isnan(o["u"][17])) and np.isnan(o["cost"][17])
        assert np.all(o["status"][np.arange(33) != 17] != _lib.STATUS_BAD_NET)
    s.close()


def test_host_driven_closed_loop_identical_on_both_paths():
    """one scenario-1 gt_mpc episode, host-driven, 30 steps: the same trajectory whichever kernel solves the steps"""
    spec = episode.reference_episode_specs(scenarios=(1,))[:1]
    s = _solver("coop_sc1")
    runs = {}
    for flag in (0, 1):
        s.set_option("latency_path", flag)
        runs[flag] = episode.run_closed_loop(s, spec, steps=30, N=40, mode="gt_mpc")
    s.set_option("latency_path", 1)
    assert _ran(_kernels(lambda: episode.run_closed_loop(s, spec, steps=2, N=40, mode="gt_mpc"))) == (True, False)
    s.close()
    assert np.array_equal(runs[1].z_cl, runs[0].z_cl) and np.array_equal(runs[1].u_cl, runs[0].u_cl)
    assert np.array_equal(runs[1].solved, runs[0].solved) and runs[1].solved.any()


@pytest.mark.parametrize("ca_type", ["circle", "obca"])
def test_device_closed_loop_with_bank_identical_on_both_paths(ca_type):
    """two episodes of different scenarios, each with its own network of the bank, on the device loop: 30 steps"""
    from igt_mpc_int_b200.planner import BatchSolver
    specs = episode.reference_episode_specs()
    specs = [specs[0], specs[8 * 2 + 1]]                                   # scenarios 1 and 3
    net_idx = np.array([sp.scenario - 1 for sp in specs])
    assert list(net_idx) == [0, 2]
    d_min = 0.0 if ca_type == "obca" else 5.6
    s = BatchSolver(N=40, mlp=[_net(k) for k in range(1, 9)], d_min=d_min)
    run = lambda steps: episode.run_closed_loop_device(s, specs, steps=steps, N=40, d_min=d_min, mode="gt_mpc",
                                                       ca_type=ca_type, net_idx=net_idx)
    runs = {}
    for flag in (0, 1):
        s.set_option("latency_path", flag)
        runs[flag] = run(30)
    s.set_option("latency_path", 1)
    assert _ran(_kernels(lambda: run(2))) == (True, False)
    s.close()
    assert np.array_equal(runs[1].z_cl, runs[0].z_cl) and np.array_equal(runs[1].u_cl, runs[0].u_cl)
    assert np.array_equal(runs[1].solved, runs[0].solved) and runs[1].solved.any()
