"""Network bank: up to 8 value networks on one handle and a per-problem network index (net_idx), so that gt_mpc
problems of all scenarios -- each planned with its own network V_GT_sc{k}, evaluate.py:123 -- run in one batch.

CPU: the exported symbols, the index routing of the closed-loop driver (with the oracle behind the BatchSolver
interface, one oracle per network) and `evaluate --sc all`.  GPU: the bank's value term, solves and episodes
against single-network handles, bit for bit."""
import os
import re

import numpy as np
import pytest

from igt_mpc_int_b200 import _lib, episode, evaluate
from tests.oracle_backend import OracleBackend
from tests.test_value_nets import raw_to_args, shipped_net

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
NEW_SYMBOLS = ("igt_set_mlp_at", "igt_solve_ex_dev", "igt_solve_ex_host", "igt_eval_ex_host", "igt_mlp_value_ex_host",
               "igt_episode_run_ex_host")


class BankOracleBackend:
    """The CPU oracle behind the BatchSolver interface with a network bank: one OracleBackend per network, problems
    dispatched by net_idx (calls without net_idx use entry 0, as the library's slot 0)."""

    def __init__(self, nets, N=40, **options):
        self.N = N
        self.nets = [None if n is None else OracleBackend(N=N, mlp=n, **options) for n in nets]
        self.net_calls = []

    def _split(self, method, net_idx, B, args, kw):
        if net_idx is None:
            return getattr(self.nets[0], method)(*args, **kw)
        net_idx = np.asarray(net_idx)
        self.net_calls.append(net_idx.copy())
        out = None
        for k in np.unique(net_idx):
            idx = np.where(net_idx == k)[0]
            sub = getattr(self.nets[k], method)(*[a[idx] for a in args], **{n: (None if v is None else v[idx]) for n, v in kw.items()})
            if out is None:
                out = {n: np.zeros((B,) + np.shape(v)[1:], dtype=np.asarray(v).dtype) for n, v in sub.items()}
            for n, v in sub.items():
                out[n][idx] = v
        return out

    def solve_batch(self, x0, u_prev, curv, obs_xy, nn_ctx=None, u_init=None, net_idx=None):
        return self._split("solve_batch", net_idx, len(x0), (x0, u_prev, curv, obs_xy), dict(nn_ctx=nn_ctx, u_init=u_init))

    def evaluate(self, x0, u_prev, curv, obs_xy, u, nn_ctx=None, net_idx=None):
        return self._split("evaluate", net_idx, len(x0), (x0, u_prev, curv, obs_xy, u), dict(nn_ctx=nn_ctx))


def _net(k):
    return shipped_net(k)[0]


# ---------------------------------------------------------------------------------------------------------- CPU
def test_bank_symbols_exported_and_header_constants():
    from igt_mpc_int_b200 import build as libbuild
    libbuild.build()
    lib = _lib.load()
    hdr = open(os.path.join(ROOT, "include", "igt_mpc.h")).read()
    assert re.search(r"#define IGT_MAX_MLP_NETS 8\b", hdr) and re.search(r"#define IGT_STATUS_BAD_NET 7\b", hdr)
    for name in NEW_SYMBOLS:
        assert re.search(r"\b%s\s*\(" % name, hdr), name
        assert hasattr(lib, name), name
        assert name in _lib.EXPORTS
    assert _lib.MAX_MLP_NETS == 8 and _lib.STATUS_BAD_NET == 7 and _lib.STATUS_BAD_NET not in _lib.STATUS_OK
    assert _lib.STATUS_NAMES[7] == "bad_net"


def test_host_loop_routes_each_episode_to_its_network():
    """Episodes of sc1 (2 hidden layers) and sc3 (3 hidden layers) in one loop with net_idx equal each scenario run
    alone with its own network, exactly: the driver hands every solve the indices of its subset."""
    specs = episode.reference_episode_specs(scenarios=(1, 3))
    mixed = [specs[0], specs[8 + 3]]                       # one episode of each scenario
    assert [sp.scenario for sp in mixed] == [1, 3]
    bank = BankOracleBackend([_net(1), None, _net(3)], N=40, max_iter=60)
    r = episode.run_closed_loop(bank, mixed, steps=6, N=40, mode="gt_mpc", net_idx=[0, 2])
    assert all(set(np.unique(c)) <= {0, 2} for c in bank.net_calls) and len(bank.net_calls) >= 6
    for e, k in enumerate((1, 3)):
        alone = episode.run_closed_loop(OracleBackend(N=40, mlp=_net(k), max_iter=60), [mixed[e]], steps=6, N=40, mode="gt_mpc")
        assert np.array_equal(r.z_cl[e], alone.z_cl[0]) and np.array_equal(r.u_cl[e], alone.u_cl[0])
        assert np.array_equal(r.solved[e], alone.solved[0])
    with pytest.raises(ValueError):
        episode.run_closed_loop(bank, mixed, steps=1, N=40, mode="mpc", net_idx=[0, 2])
    with pytest.raises(ValueError):
        episode.run_closed_loop(bank, mixed, steps=1, N=40, mode="gt_mpc", net_idx=[0, 2, 2])


def _write_nets(tmp_path):
    for k in range(1, 9):
        net = _net(k)
        arrs = {"W%d" % i: W for i, (W, _) in enumerate(net["weights"])}
        arrs.update({"b%d" % i: b for i, (_, b) in enumerate(net["weights"])})
        np.savez(tmp_path / ("net_sc%d.npz" % k), **arrs)
    return str(tmp_path / "net_sc{sc}.npz")


def test_evaluate_sc_all_expands_weights_per_scenario(tmp_path):
    path = _write_nets(tmp_path)
    a = evaluate.build_parser().parse_args(["--save_dir", str(tmp_path / "runs"), "--eval_mode", "gt_mpc", "--sc", "all",
                                            "--nn_weights", path, "--steps", "2"])
    assert a.sc == "all"
    assert evaluate.build_parser().parse_args(["--save_dir", "x", "--eval_mode", "mpc", "--sc", "4"]).sc == 4
    with pytest.raises(SystemExit):
        evaluate.build_parser().parse_args(["--save_dir", "x", "--eval_mode", "mpc", "--sc", "9"])
    # {sc} with one scenario: that scenario's network; with all of them: the bank, entry k - 1 = scenario k
    one = evaluate.networks(path, [3])
    assert isinstance(one, dict) and len(one["weights"]) == 4
    assert np.array_equal(one["weights"][0][0], _net(3)["weights"][0][0])
    nets = evaluate.networks(path, list(range(1, 9)))
    assert len(nets) == 8 and [len(n["weights"]) for n in nets] == [3, 3, 4, 3, 3, 4, 4, 3]
    plain = evaluate.networks(str(tmp_path / "net_sc5.npz"), list(range(1, 9)))
    assert isinstance(plain, dict)
    bank = BankOracleBackend(nets, N=40, max_iter=60)
    run_dirs, summary = evaluate.main(a, solver=bank)
    assert len(run_dirs) == 8
    for k, d in enumerate(run_dirs, start=1):
        assert os.path.basename(d).startswith("gt_mpc_sc%d_seed2026_" % k)
        assert [f for _, _, fs in os.walk(d) for f in fs if f == "cl_traj.pkl"], d   # laid out as for --sc k
    assert [s["scenario"] for s in summary] == list(range(1, 9))
    # one loop for all scenarios: every solve call carries the indices of its vehicles, all eight networks in use
    assert len(bank.net_calls) >= 2 and set(np.concatenate(bank.net_calls)) == set(range(8))
    # --sc k with a {sc} path: scenario k's network, no bank (no net_idx)
    single = BankOracleBackend([_net(6)], N=40, max_iter=60)
    b = evaluate.build_parser().parse_args(["--save_dir", str(tmp_path / "runs6"), "--eval_mode", "gt_mpc", "--sc", "6",
                                            "--nn_weights", path, "--steps", "2"])
    run_dir, summary6 = evaluate.main(b, solver=single)
    assert isinstance(run_dir, str) and "gt_mpc_sc6_" in run_dir and not single.net_calls and len(summary6) == 1


# ---------------------------------------------------------------------------------------------------------- GPU
def _bank_solver(**kw):
    from igt_mpc_int_b200.planner import BatchSolver
    return BatchSolver(N=40, mlp=[_net(k) for k in range(1, 9)], **kw)


def _single(k, **kw):
    from igt_mpc_int_b200.planner import BatchSolver
    return BatchSolver(N=40, mlp=_net(k), **kw)


@pytest.mark.gpu
def test_bank_value_term_mixed_networks_bit_identical():
    rows, idx, gold = [], [], []
    for k in range(1, 9):
        _, x, y = shipped_net(k)
        rows.append(x); idx.append(np.full(len(x), k - 1)); gold.append(y)
    x, idx, y = np.concatenate(rows), np.concatenate(idx).astype(np.int32), np.concatenate(gold)
    perm = np.random.default_rng(7).permutation(len(x))
    x, idx, y = x[perm], idx[perm], y[perm]
    sN, vN, ctx = raw_to_args(x)
    s = _bank_solver()
    coop = s.mlp_value(sN, vN, ctx, tensor_cores=2, net_idx=idx)
    per = s.mlp_value(sN, vN, ctx, tensor_cores=0, net_idx=idx)
    assert np.array_equal(coop, per)
    with pytest.raises(_lib.IgtError):
        s.mlp_value(sN, vN, ctx, tensor_cores=1, net_idx=idx)          # the tcgen05 kernel holds one network
    s.close()
    assert np.max(np.abs(coop[:, 0] - y)) < 1e-12 * max(1.0, np.abs(y).max())
    for k in range(8):
        m = idx == k
        one = _single(k + 1)
        assert np.array_equal(coop[m], one.mlp_value(sN[m], vN[m], ctx[m], tensor_cores=2))
        one.close()


@pytest.fixture(scope="module")
def mixed_batch():
    from igt_mpc_int_b200 import scenarios as S
    pb = S.mid_episode(8192, N=40, seed=77)
    perm = np.random.default_rng(5).permutation(8192)
    f = lambda a: np.ascontiguousarray(a[perm])
    return dict(x0=f(pb.x0), u_prev=f(pb.u_prev), curv=f(pb.curv), obs=f(pb.obs), nn_ctx=f(pb.nn_ctx),
                obs_psi=f(pb.obs_psi), net_idx=f(pb.scenario - 1).astype(np.int32))


def _solve(s, b, idx=None, net_idx=None, obca=False):
    sel = slice(None) if idx is None else idx
    return s.solve_batch(b["x0"][sel], b["u_prev"][sel], b["curv"][sel], b["obs"][sel], nn_ctx=b["nn_ctx"][sel],
                         obs_psi=b["obs_psi"][sel] if obca else None, net_idx=net_idx)


def _assert_same(r, o, m=slice(None)):
    for key in ("status", "iters", "cost", "u", "x"):
        assert np.array_equal(r[key][m], o[key], equal_nan=True), key


@pytest.mark.gpu
def test_bank_solves_equal_single_network_handles(mixed_batch, oracle_params):
    b = mixed_batch
    s = _bank_solver()
    r = _solve(s, b, net_idx=b["net_idx"])
    s.close()
    for k in range(8):
        idx = np.where(b["net_idx"] == k)[0]
        one = _single(k + 1)
        one.set_option("tensor_core_mlp", 0)
        _assert_same(r, _solve(one, b, idx), idx)
        one.close()
    assert np.mean(r["status"] == 0) > 0.6
    # north-star tolerances against the oracle with each problem's own network, on 256 problems
    from oracle import c_oracle, nlp
    from tests.util import relerr
    sub = np.arange(256)
    o_status = np.empty(256, dtype=np.int64); o_cost = np.empty(256); o_U = np.empty((256, 40, 2))
    for k in range(8):
        m = sub[b["net_idx"][sub] == k]
        if len(m) == 0:
            continue
        o = c_oracle.COracle(oracle_params[40], nlp.MLPTerm(**_net(k + 1)), max_iter=60).solve(
            b["x0"][m], b["u_prev"][m], b["curv"][m], b["obs"][m], nn_ctx=b["nn_ctx"][m])
        o_status[m], o_cost[m], o_U[m] = o["status"], o["cost"], o["U"]
    assert np.mean(r["status"][sub] == o_status) > 0.98
    ok = (r["status"][sub] == 0) & (o_status == 0)
    assert ok.sum() > 0.6 * 256
    assert np.max(relerr(r["cost"][sub][ok], o_cost[ok])) < 1e-4
    assert np.max(np.abs(r["u"][sub][ok] - o_U[ok])) < 1e-3
    assert np.max(r["viol"][sub][ok]) <= 1e-6


@pytest.mark.gpu
def test_bank_index_zero_reproduces_the_single_network_path(mixed_batch):
    b = mixed_batch
    s = _bank_solver()
    s.set_option("tensor_core_mlp", 0)
    idx = np.arange(2048)
    plain = _solve(s, b, idx)
    banked = _solve(s, b, idx, net_idx=np.zeros(2048, dtype=np.int32))
    s.close()
    _assert_same(banked, plain)


@pytest.mark.gpu
def test_bank_obca_per_thread_path_and_device_entry(mixed_batch):
    import torch
    b = mixed_batch
    idx = np.arange(1024)
    s = _bank_solver(d_min=0.0)
    r = _solve(s, b, idx, net_idx=b["net_idx"][idx], obca=True)
    for k in range(8):
        m = np.where(b["net_idx"][idx] == k)[0]
        one = _single(k + 1, d_min=0.0)
        _assert_same(r, _solve(one, b, idx[m], obca=True), m)
        one.close()
    # the device entry point (in-kernel index check) gives the host path's numbers
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    out = s.solve_batch_device(d(b["x0"][idx]), d(b["u_prev"][idx]), d(b["curv"][idx]), d(b["obs"][idx]),
                               nn_ctx=d(b["nn_ctx"][idx]), obs_psi=d(b["obs_psi"][idx]), net_idx=d(b["net_idx"][idx]))
    torch.cuda.synchronize()
    _assert_same({k: v.cpu().numpy() for k, v in out.items()}, r)
    s.close()


@pytest.mark.gpu
def test_bank_f32_equals_single_network_handles(mixed_batch):
    """the f32 bank kernel (per-thread value term, float descriptor table) against f32 single-network handles"""
    b = mixed_batch
    idx = np.arange(2048)
    s = _bank_solver(precision="f32")
    r = _solve(s, b, idx, net_idx=b["net_idx"][idx])
    s.close()
    for k in range(8):
        m = np.where(b["net_idx"][idx] == k)[0]
        one = _single(k + 1, precision="f32")
        _assert_same(r, _solve(one, b, idx[m]), m)
        one.close()


def _wide_net(hidden, seed):
    """a network with a layer wider than the cooperative evaluation's 128 (torch.nn.Linear's default init)"""
    rng = np.random.default_rng(seed)
    dims = [6] + list(hidden) + [1]
    w = [(rng.uniform(-1, 1, (dims[i + 1], dims[i])) / np.sqrt(dims[i]), rng.uniform(-1, 1, dims[i + 1]) / np.sqrt(dims[i]))
         for i in range(len(dims) - 1)]
    return dict(weights=w, Wn=np.eye(6), mu_f=np.zeros(6), sigma_t=1.0, mu_t=0.0)


@pytest.mark.gpu
def test_bank_wider_than_128_uses_the_per_thread_path(mixed_batch):
    """a bank with a network wider than 128: f64 circle-mode solves take the per-thread bank kernel, bit-identical to
    single-network handles (which take the per-thread kernel as well)"""
    from igt_mpc_int_b200.planner import BatchSolver
    b = mixed_batch
    idx = np.arange(1024)
    nets = [_wide_net((160,), 1), _wide_net((144, 144), 2)]
    ni = (b["net_idx"][idx] % 2).astype(np.int32)
    s = BatchSolver(N=40, mlp=nets)
    r = _solve(s, b, idx, net_idx=ni)
    with pytest.raises(_lib.IgtError):                                   # no cooperative evaluation for this bank
        s.mlp_value(b["x0"][idx, 2], b["x0"][idx, 5], b["nn_ctx"][idx], tensor_cores=2, net_idx=ni)
    s.close()
    for k in range(2):
        m = np.where(ni == k)[0]
        one = BatchSolver(N=40, mlp=nets[k])
        _assert_same(r, _solve(one, b, idx[m]), m)
        one.close()


@pytest.mark.gpu
def test_bank_index_errors(mixed_batch):
    import torch
    b = mixed_batch
    idx = np.arange(512)
    from igt_mpc_int_b200.planner import BatchSolver
    s = BatchSolver(N=40, mlp=[_net(1), None, _net(3)])                 # slot 1 and 3..7 empty
    good = np.where(b["net_idx"][idx] % 2 == 0, 0, 2).astype(np.int32)
    n0 = s.launches
    for bad in (-1, 8, 1, 5):
        ni = good.copy(); ni[17] = bad
        with pytest.raises(_lib.IgtError):
            _solve(s, b, idx, net_idx=ni)
        with pytest.raises(_lib.IgtError):
            s.mlp_value(b["x0"][idx, 2], b["x0"][idx, 5], b["nn_ctx"][idx], tensor_cores=2, net_idx=ni)
    assert s.launches == n0
    with pytest.raises(_lib.IgtError):                                   # net_idx needs nn_ctx
        s.solve_batch(b["x0"][idx], b["u_prev"][idx], b["curv"][idx], b["obs"][idx], net_idx=good)
    ref = _solve(s, b, idx, net_idx=good)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    for bad in (-1, 8, 1):
        ni = good.copy(); ni[17] = bad
        out = s.solve_batch_device(d(b["x0"][idx]), d(b["u_prev"][idx]), d(b["curv"][idx]), d(b["obs"][idx]),
                                   nn_ctx=d(b["nn_ctx"][idx]), net_idx=d(ni))
        torch.cuda.synchronize()
        o = {k: v.cpu().numpy() for k, v in out.items()}
        assert o["status"][17] == _lib.STATUS_BAD_NET and o["iters"][17] == 0
        assert np.all(np.isnan(o["x"][17])) and np.all(np.isnan(o["u"][17])) and np.isnan(o["cost"][17])
        rest = np.arange(512) != 17
        _assert_same(o, {k: v[rest] for k, v in ref.items()}, rest)
    s.close()


@pytest.mark.gpu
def test_bank_episodes_equal_per_scenario_runs():
    """64 reference episodes x 150 steps, gt_mpc, one device loop with the bank (net_idx = scenario - 1), against the
    eight per-scenario device runs (bit for bit) and the host-driven loop with the bank (same criteria as
    test_device_closed_loop_equals_host_driven_loop)."""
    specs = episode.reference_episode_specs()
    net_idx = np.array([sp.scenario - 1 for sp in specs])
    s = _bank_solver()
    rd = episode.run_closed_loop_device(s, specs, steps=150, N=40, mode="gt_mpc", net_idx=net_idx)
    for k in range(8):
        one = _single(k + 1)
        one.set_option("tensor_core_mlp", 0)
        r1 = episode.run_closed_loop_device(one, specs[8 * k:8 * k + 8], steps=150, N=40, mode="gt_mpc")
        one.close()
        sl = slice(8 * k, 8 * k + 8)
        assert np.array_equal(rd.z_cl[sl], r1.z_cl) and np.array_equal(rd.u_cl[sl], r1.u_cl)
        assert np.array_equal(rd.solved[sl], r1.solved)
    rh = episode.run_closed_loop(s, specs, steps=150, N=40, mode="gt_mpc", net_idx=net_idx)
    s.close()
    assert np.array_equal(rd.collision, rh.collision)
    assert np.sum(rd.deadlock != rh.deadlock) <= 1 and np.sum(np.any(rd.goal != rh.goal, axis=1)) <= 1
    assert np.mean(rd.solved == rh.solved) > 0.99
    assert np.max(np.abs(rd.z_cl[:, :, :20] - rh.z_cl[:, :, :20])) < 1e-7


@pytest.mark.gpu
def test_bank_obca_episodes_equal_per_scenario_runs():
    specs = episode.reference_episode_specs()[::4]                        # two episodes per scenario
    net_idx = np.array([sp.scenario - 1 for sp in specs])
    s = _bank_solver(d_min=0.0)
    rd = episode.run_closed_loop_device(s, specs, steps=30, N=40, d_min=0.0, mode="gt_mpc", ca_type="obca", net_idx=net_idx)
    s.close()
    for k in range(8):
        one = _single(k + 1, d_min=0.0)
        r1 = episode.run_closed_loop_device(one, specs[2 * k:2 * k + 2], steps=30, N=40, d_min=0.0, mode="gt_mpc", ca_type="obca")
        one.close()
        sl = slice(2 * k, 2 * k + 2)
        assert np.array_equal(rd.z_cl[sl], r1.z_cl) and np.array_equal(rd.u_cl[sl], r1.u_cl)
        assert np.array_equal(rd.solved[sl], r1.solved)
