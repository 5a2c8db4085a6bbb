"""The product's per-thread solver code (csrc/solver_core.cuh) executed on the CPU by the test
harness tests/hostsim, against the oracle.  This checks kernel LOGIC without a GPU; the -m gpu
tests check the kernels themselves through the C ABI."""
import numpy as np
import pytest

from igt_mpc_int_b200 import scenarios as S, terminal_set as TS
from oracle import c_oracle
from tests.hostsim import harness as H
from tests.util import relerr


@pytest.fixture(scope="module")
def cinf():
    return TS.cinf()


def _tight(p):
    p.max_iter = 300      # tolerances already equal the oracle's
    p.max_trials = 0      # no budget of forward passes, like the oracle's default
    return p


def test_core_fp64_reproduces_oracle_iterates(oracle_params, cinf):
    for N, B in ((40, 48), (10, 16), (20, 16)):
        pb = S.mid_episode(B, N=N)
        p = _tight(H.default_params(1)); p.N = N; p.set_cinf(*cinf)
        r = H.solve(p, pb.x0, pb.u_prev, pb.curv, pb.obs)
        o = c_oracle.COracle(oracle_params[N], max_iter=300).solve(pb.x0, pb.u_prev, pb.curv, pb.obs)
        assert np.array_equal(r["status"], o["status"])
        ok = o["status"] == 0
        assert ok.sum() >= 0.8 * B
        assert np.array_equal(r["iters"][ok], o["iters"][ok])
        assert np.max(relerr(r["cost"][ok], o["cost"][ok])) < 1e-9
        assert np.max(np.abs(r["U"][ok] - o["U"][ok])) < 1e-8
        assert np.max(r["viol"][ok]) <= 1e-6


def test_core_rollout_matches_golden(golden, cinf):
    g = golden["frenet_rk4"]
    p = H.default_params(1); p.set_cinf(*cinf)
    Z, A, Bm = H.rollout(p, 1, g["rz0"], g["ru"], g["rcurv"], jac=True)
    assert np.max(np.abs(Z - g["rz"])) < 1e-10
    # fp32 arithmetic of the same code: 1e-5 relative (scale 1.0) against the fp64 reference model
    Z32 = H.rollout(p, 0, g["rz0"], g["ru"], g["rcurv"])
    e = relerr(Z32, g["rz"])
    assert np.quantile(e, 0.99) < 1e-5
    # Jacobians of the product code == oracle Jacobians
    from oracle import dynamics as D
    for b in range(4):
        _, Ao, Bo = D.frenet_rollout(g["rz0"][b], g["ru"][b], tuple(g["rcurv"][b]), want_jac=True)
        assert np.max(np.abs(A[b] - Ao)) < 1e-12 and np.max(np.abs(Bm[b] - Bo)) < 1e-12


def test_core_default_tolerances_meet_parity_targets(oracle_params, cinf):
    """Product default options (looser than the oracle's) still land within the north-star
    tolerances: 1e-4 relative cost (denominator max(|J|,1)), 1e-3 max |du|, 1e-6 violation."""
    pb = S.mid_episode(48, N=40, seed=77)
    p = H.default_params(1); p.set_cinf(*cinf)
    r = H.solve(p, pb.x0, pb.u_prev, pb.curv, pb.obs)
    o = c_oracle.COracle(oracle_params[40]).solve(pb.x0, pb.u_prev, pb.curv, pb.obs)
    ok = (o["status"] == 0) & (r["status"] == 0)
    assert ok.sum() >= 0.8 * len(pb)
    assert np.max(relerr(r["cost"][ok], o["cost"][ok])) < 1e-4
    assert np.max(np.abs(r["U"][ok] - o["U"][ok])) < 1e-3
    assert np.max(r["viol"][ok]) <= 1e-6


def test_core_x0_infeasible_and_warm_start(oracle_params, cinf):
    pb = S.mid_episode(8, N=40, seed=5)
    p = H.default_params(1); p.set_cinf(*cinf)
    x0 = pb.x0.copy(); x0[0, 5] = 5.5; x0[1, 3] = 0.3          # v0 > v_max, |ey0| > ey_lim
    r = H.solve(p, x0, pb.u_prev, pb.curv, pb.obs)
    assert r["status"][0] == 2 and r["status"][1] == 2 and np.isnan(r["cost"][0])
    cold = H.solve(p, pb.x0, pb.u_prev, pb.curv, pb.obs)
    ok = cold["status"] == 0
    warm = H.solve(p, pb.x0, pb.u_prev, pb.curv, pb.obs, u_init=np.nan_to_num(cold["U"]))
    assert np.all(warm["status"][ok] == 0)
    assert np.max(relerr(warm["cost"][ok], cold["cost"][ok])) < 1e-4


def test_core_iteration_and_trial_budgets_match_oracle(oracle_params, cinf):
    """max_iter 60 (default) and a budget of 150 forward passes against the oracle run with the
    same budgets: the same problems are given up on, with the same status."""
    pb = S.mid_episode(256, N=40, seed=2026)
    p = H.default_params(1); p.set_cinf(*cinf)
    assert p.max_iter == 60 and p.max_trials == 0
    p.max_trials = 150
    r = H.solve(p, pb.x0, pb.u_prev, pb.curv, pb.obs)
    o = c_oracle.COracle(oracle_params[40], max_iter=p.max_iter, max_trials=p.max_trials).solve(pb.x0, pb.u_prev, pb.curv, pb.obs)
    assert np.mean(r["status"] == o["status"]) >= 0.99
    assert (r["status"] != 0).sum() > 0


def test_product_solver_code_obca_mode_matches_oracle(oracle_params):
    """The product's per-thread solver code with the OBCA collision rows (csrc/obca.cuh, Ws<T, 32, true>) run on the CPU
    reproduces the oracle's C port: same statuses, iteration counts and optima (mpc.py:211-221, d_min = 0)."""
    from oracle import nlp, c_oracle
    N = 40
    P = nlp.Params(N=N, d_min=0.0, cinf_A=oracle_params[40].cinf_A, cinf_b=oracle_params[40].cinf_b)
    pb = S.mid_episode(64, N=N, seed=5)
    p = H.default_params(1)
    p.N = N; p.d_min = 0.0
    p.set_cinf(P.cinf_A, P.cinf_b)
    r = H.solve_obca(p, pb.x0, pb.u_prev, pb.curv, pb.obs, pb.obs_psi)
    o = c_oracle.COracle(P, max_iter=p.max_iter).solve(pb.x0, pb.u_prev, pb.curv, pb.obs, obs_psi=pb.obs_psi)
    assert np.array_equal(r["status"], o["status"]) and np.mean(r["iters"] == o["iters"]) > 0.95
    ok = o["status"] == 0
    assert ok.sum() >= 50
    assert np.max(np.abs(r["cost"][ok] - o["cost"][ok]) / np.maximum(1.0, np.abs(o["cost"][ok]))) < 1e-9
    assert np.max(np.abs(r["U"][ok] - o["U"][ok])) < 1e-6 and r["viol"][ok].max() <= 1e-9
    # the rows bind: some solutions sit on the rectangle-distance margin
    from oracle import obca
    dmin = [min(obca.rect_distance(o["Z"][i][k, [0, 1, 6]], np.array([pb.obs[i, k, 0], pb.obs[i, k, 1], pb.obs_psi[i, k]]))[0]
                for k in range(1, N + 1)) for i in np.where(ok)[0]]
    assert min(dmin) < 1e-5 and min(dmin) > -1e-9


def _lane_batch(B, seed):
    """B mid_episode problems with problems that init rejects (v and ey outside their limits, NaN v) and problems
    with a non-finite state that init accepts and the solve then fails on, spread over the batch"""
    pb = S.mid_episode(B, N=40, seed=seed)
    x0 = pb.x0.copy()
    bad = np.random.default_rng(seed).choice(B, 12, replace=False)
    for i, q in enumerate(bad):
        col, val = ((5, 5.5), (5, -0.4), (3, 0.3), (5, np.nan), (0, np.nan), (2, np.inf))[i % 6]
        x0[q, col] = val
    return pb, x0, bad


@pytest.mark.parametrize("case", ["f64", "f32", "obca", "gt_mpc"])
def test_core_lane_reuse_equals_fresh_solver_objects(cinf, case):
    """The kernels keep one Solver object per lane and hand it problem after problem; Solver::init must leave nothing
    of the previous problem that the next solve reads.  Slot q % 32 of the harness solves problems q, q + 32, ... with
    one object (10 problems per slot here), bit-identical to a fresh object per problem -- with rejected problems, failed
    solves and an iteration cap low enough for capped ones (status 1 / 6) in the mix."""
    from tests.test_value_nets import shipped_net
    from oracle import nlp
    B = 320
    pb, x0, bad = _lane_batch(B, seed=31)
    p = H.default_params(0 if case == "f32" else 1)
    p.set_cinf(*cinf)
    p.max_iter = 25
    if case == "obca":
        p.d_min = 0.0
        run = lambda lanes: H.solve_obca(p, x0, pb.u_prev, pb.curv, pb.obs, pb.obs_psi, lanes=lanes)
    else:
        mlp = nlp.MLPTerm(**shipped_net(3)[0]) if case == "gt_mpc" else None
        ctx = pb.nn_ctx if case == "gt_mpc" else None
        run = lambda lanes: H.solve(p, x0, pb.u_prev, pb.curv, pb.obs, nn_ctx=ctx, mlp=mlp, lanes=lanes)
    fresh, reused = run(False), run(True)
    for k in ("status", "iters", "cost", "viol", "U", "Z"):
        assert np.array_equal(reused[k], fresh[k], equal_nan=True), k
    st = fresh["status"]
    assert np.all(st[bad] != 0) and (st[bad] == 2).sum() >= 8
    assert (st == 0).mean() > 0.5 and len(set(st[st != 0]) - {2}) >= 2     # more than one failure status besides 2
