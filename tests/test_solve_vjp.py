"""Gradients through the batched solve (csrc/sens.cuh), on the CPU: the oracle VJP (oracle/sensitivity.py, dense) against
central differences of re-solves by the C port of the oracle, and the product's VJP code run by tests/hostsim against the
oracle VJP on the same (u, y, s).  The GPU side is tests/test_gpu_solve_vjp.py."""
import numpy as np
import pytest

from igt_mpc_int_b200 import scenarios as S, terminal_set as TS
from oracle import c_oracle, dynamics as D, nlp, sensitivity as SE
from tests.hostsim import sens_harness as H

N = 40
# every solve ends at mu = mu_floor (tol_comp just above it) with stationarity <= 1e-10: the re-solves of the finite
# differences then follow the same barrier solution the VJP linearises (s_i y_i = mu_floor held fixed)
TIGHT = dict(max_iter=1000, max_trials=0, mu_floor=1e-4, tol=1e-10, tol_comp=1.5e-4, tol_rp=1e-12)
FD_H = 1e-5


@pytest.fixture(scope="module")
def cinf():
    return TS.cinf()


def _params(cinf, **kw):
    p = H.default_params(1)
    p.set_cinf(*cinf)
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def _oracle_params(cinf):
    return nlp.Params(N=N, cinf_A=cinf[0], cinf_b=cinf[1])     # the solver's row order of the terminal set


def _coll_rows(p):
    """flat indices of the collision rows of nodes 1..N (row_off order, include/igt_mpc.h)"""
    return np.array([8 + 13 * (k - 1) + 4 for k in range(1, N)] + [8 + 13 * (N - 1) + p.n_cinf + 2])


def _stage_s(P, x0, U, curv):
    """arc length of every RK4 stage state of the rollout (oracle/dynamics.frenet_rk4_step)"""
    out, z, h = [], np.array(x0, dtype=np.float64), P.dt / P.n_rk
    full = np.ones(7); full[D.IPSI] = 0.5
    for k in range(N):
        for _ in range(P.n_rk):
            k1 = D.rhs(z, U[k], curv); k2 = D.rhs(z + 0.5 * h * k1, U[k], curv)
            k3 = D.rhs(z + 0.5 * h * k2, U[k], curv); k4 = D.rhs(z + h * full * k3, U[k], curv)
            out += [z[D.IS], z[D.IS] + 0.5 * h * k1[D.IS], z[D.IS] + 0.5 * h * k2[D.IS], z[D.IS] + h * k3[D.IS]]
            z = z + h / 6.0 * (k1 + 2 * k2 + 2 * k3 + k4)
    return np.array(out)


def _problem(pb, b, gt):
    return nlp.Problem(x0=pb.x0[b], u_prev=pb.u_prev[b], curv=tuple(pb.curv[b]), obs=pb.obs[b],
                       nn_ctx=tuple(pb.nn_ctx[b]) if gt else None)


def _fd_case(cinf, pb, mlp, n_keep, rng):
    """(checked, excluded) after comparing the oracle VJP with central differences of C-oracle re-solves"""
    gt = mlp is not None
    P = _oracle_params(cinf)
    p = _params(cinf, **TIGHT)
    ctx = pb.nn_ctx if gt else None
    r = H.solve_duals(p, pb.x0, pb.u_prev, pb.curv, pb.obs, nn_ctx=ctx, mlp=mlp)
    co = c_oracle.COracle(P, mlp=mlp, **TIGHT)
    o = co.solve(pb.x0, pb.u_prev, pb.curv, pb.obs, nn_ctx=ctx, u_init=r["U"])
    cr = _coll_rows(p)
    checked = excluded = 0
    for b in range(len(pb)):
        if checked == n_keep:
            break
        if r["status"][b] != 0 or o["status"][b] != 0 or np.abs(o["U"][b] - r["U"][b]).max() > 1e-7:
            continue
        Y, Sm = r["Y"][b], r["S"][b]
        if not gt and Y[cr].min() > 1e-3:                         # 'mpc' cases: an active collision row
            continue
        bps = np.array(pb.curv[b][:2])
        near_break = np.abs(_stage_s(P, pb.x0[b], r["U"][b], pb.curv[b])[:, None] - bps[None]).min() < 1e2 * FD_H
        if near_break or np.any((Y < 1e-2) & (Sm < 1e-2)):      # curvature break point / degenerate row (y, s below 100 mu_floor)
            excluded += 1
            continue
        gx, gu, gc = rng.standard_normal((N + 1, 7)), rng.standard_normal((N, 2)), rng.standard_normal()
        g0, gup, gob, ok = SE.vjp(P, _problem(pb, b, gt), mlp, r["U"][b], Y, Sm, 0, gx, gu, gc)
        assert ok == 1
        # parameters: every entry of x0 and u_prev, 8 obstacle entries (the most active collision nodes first)
        ks = 1 + np.argsort(np.concatenate([Y[cr[:-1]], Y[cr[-1:]]]))[:4]
        params = [("x0", i) for i in range(7)] + [("u_prev", i) for i in range(2)] + \
                 [("obs", (k, j)) for k in ks for j in range(2)]
        B2 = 2 * len(params)
        x0 = np.repeat(pb.x0[b:b + 1], B2, 0); up = np.repeat(pb.u_prev[b:b + 1], B2, 0)
        ob = np.repeat(pb.obs[b:b + 1], B2, 0)
        for q, (name, i) in enumerate(params):
            for sgn, row in ((1, 2 * q), (-1, 2 * q + 1)):
                if name == "x0":
                    x0[row, i] += sgn * FD_H
                elif name == "u_prev":
                    up[row, i] += sgn * FD_H
                else:
                    ob[row, i[0], i[1]] += sgn * FD_H
        rs = co.solve(x0, up, np.repeat(pb.curv[b:b + 1], B2, 0), ob, nn_ctx=None if not gt else np.repeat(ctx[b:b + 1], B2, 0),
                      u_init=np.repeat(r["U"][b:b + 1], B2, 0))
        if np.any(rs["status"] != 0):                            # a re-solve that did not reach the tight tolerances
            excluded += 1
            continue
        f = np.einsum("bkj,kj->b", rs["Z"], gx) + np.einsum("bkj,kj->b", rs["U"], gu) + gc * rs["cost"]
        g_fd = (f[0::2] - f[1::2]) / (2 * FD_H)
        g = np.array([g0[i] if n == "x0" else gup[i] if n == "u_prev" else gob[i[0], i[1]] for n, i in params])
        assert np.all(np.abs(g - g_fd) <= 1e-4 * max(np.abs(g_fd).max(), 1e-3)), (b, np.abs(g - g_fd).max(), np.argmax(np.abs(g - g_fd)), np.abs(g_fd).max(), Y.min(), Sm[np.argmin(Y)])
        checked += 1
    return checked, excluded


def test_oracle_vjp_matches_finite_differences_of_resolves(cinf):
    """24 problems at N = 40: 'mpc' config-2 draws with an active collision row and gt_mpc with a shipped network;
    random cotangents on x, u and cost; every entry of gx0 and gu_prev and 8 obstacle entries per problem"""
    from tests.test_value_nets import shipped_net
    rng = np.random.default_rng(5)
    n_mpc, ex_mpc = _fd_case(cinf, S.mid_episode(384, N=N, seed=11), None, 16, rng)
    mlp = nlp.MLPTerm(**shipped_net(1)[0])
    n_gt, ex_gt = _fd_case(cinf, S.mid_episode(32, N=N, seed=12), mlp, 8, rng)
    print("checked %d 'mpc' + %d gt_mpc problems; excluded %d + %d (curvature break point within reach of the "
          "difference step, a degenerate row, or a re-solve short of the tight tolerances)" % (n_mpc, n_gt, ex_mpc, ex_gt))
    assert n_mpc == 16 and n_gt == 8


def _rel(a, ref):
    return np.abs(a - ref).max() / max(np.abs(ref).max(), 1e-300)


@pytest.mark.parametrize("mode", ["mpc", "gt_mpc"])
def test_hostsim_vjp_matches_oracle_vjp(cinf, mode):
    """csrc/sens.cuh on the CPU against the dense oracle on the same (u, y, s): gradients to 1e-9 relative and the same
    ok; a status != 0 problem, a non-positive multiplier and a point whose Hessian is made indefinite (a huge collision
    multiplier) give ok = 0 and exact zeros.  The solves end at mu_floor = 1e-4: at the default 1e-8, s / y reaches 1e12
    on active rows and the two factorisations (Riccati vs dense Cholesky) differ by that conditioning, ~1e-7."""
    from tests.test_value_nets import shipped_net
    gt = mode == "gt_mpc"
    mlp = nlp.MLPTerm(**shipped_net(3)[0]) if gt else None
    B = 24
    pb = S.mid_episode(B, N=N, seed=21 if gt else 22)
    ctx = pb.nn_ctx if gt else None
    p = _params(cinf, **TIGHT)
    r = H.solve_duals(p, pb.x0, pb.u_prev, pb.curv, pb.obs, nn_ctx=ctx, mlp=mlp)
    Y, Sm, st = r["Y"].copy(), r["S"].copy(), r["status"].copy()
    good = np.where(st == 0)[0]
    assert len(good) >= 12
    b_bad, b_neg, b_npd = good[-1], good[-2], good[-3]
    st[b_bad] = 1
    Sm[b_neg, 5] = -Sm[b_neg, 5]
    Sm[b_npd, _coll_rows(p)] = 1e6
    rng = np.random.default_rng(3)
    gx, gu, gc = rng.standard_normal((B, N + 1, 7)), rng.standard_normal((B, N, 2)), rng.standard_normal(B)
    hg = H.vjp(p, pb.x0, pb.u_prev, pb.curv, pb.obs, r["U"], Y, Sm, st, gx, gu, gc, nn_ctx=ctx, mlp=mlp)
    P = _oracle_params(cinf)
    n_ok = 0
    for b in range(B):
        og = SE.vjp(P, _problem(pb, b, gt), mlp, r["U"][b], Y[b], Sm[b], st[b], gx[b], gu[b], gc[b])
        assert hg[3][b] == og[3], b
        for i in range(3):
            if og[3]:
                assert _rel(hg[i][b], og[i]) <= 1e-9, (b, i, _rel(hg[i][b], og[i]))
            else:
                assert np.all(hg[i][b] == 0.0)
        n_ok += og[3]
    assert hg[3][b_bad] == 0 and hg[3][b_neg] == 0 and hg[3][b_npd] == 0
    assert n_ok >= len(good) - 3 - 2
    # a NULL cotangent is zero
    z = H.vjp(p, pb.x0, pb.u_prev, pb.curv, pb.obs, r["U"], Y, Sm, st, None, gu, None, nn_ctx=ctx, mlp=mlp)
    o = H.vjp(p, pb.x0, pb.u_prev, pb.curv, pb.obs, r["U"], Y, Sm, st, np.zeros_like(gx), gu, np.zeros(B), nn_ctx=ctx, mlp=mlp)
    for a, c in zip(z, o):
        assert np.array_equal(a, c)
