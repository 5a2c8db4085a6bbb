"""ORACLE (test infrastructure) -- fp64 numpy vector-Jacobian product of a solve through its converged KKT system,
with dense linear algebra.

Only tests/ and tools/ may import this.  It restates what csrc/sens.cuh computes, by a different route:

  The returned (u, y, s) satisfy  grad_u L = 0,  c + y = 0,  s_i y_i = const_i  (L = J + s'c, x = rollout(x0, u)).
  With every row's product s_i y_i held fixed, the implicit function theorem gives
      du/dtheta = -K^-1 M,   K = d2L/du2 + C' Sigma C,   M = d2L/du dtheta + C' Sigma dc/dtheta,   Sigma = diag(s / y),
  theta = (x0, u_prev, obs_xy[1..N]).  Cotangents gx, gu, gcost on the outputs x, u, cost are pulled back to a reduced
  cotangent r on u plus direct terms on theta, and  g_theta = direct - M' K^-1 r.

Here K and M are assembled densely in the space w = (u, x0, u_prev) from the total state Jacobians dx_k/dw; the
second derivatives of the discrete RK4 step are taken by complex step on a complex-safe restatement of
oracle/dynamics.py's forward sensitivities (not by the dual numbers of sens.cuh), and the system is solved by Cholesky.
ok = 0 (zero gradients) when the solve did not converge (status != 0), when a slack or multiplier is not positive,
or when K is not positive definite -- the same condition as a Riccati stage's Quu failing to be positive definite,
since those are the pivots of a block factorisation of K.
"""
import numpy as np

from . import dynamics as D
from . import solver as SV

NZ = 7
ROT = (D.IEY, D.IEPSI, D.IV, D.IPSI)


def _rhs_jac(z, u, curv):
    """oracle/dynamics.rhs with its Jacobians, complex-safe (the pw_const curvature is taken at Re s)."""
    ey, epsi, v, psi = z[D.IEY], z[D.IEPSI], z[D.IV], z[D.IPSI]
    a, df = u[0], u[1]
    K = D.curvature(float(np.real(z[D.IS])), curv)
    rho = D.L_R / (D.L_F + D.L_R)
    t = np.tan(df)
    beta = np.arctan(rho * t)
    dbeta = rho * (1.0 + t * t) / (1.0 + rho * rho * t * t)
    c1, s1 = np.cos(beta + epsi), np.sin(beta + epsi)
    cp, sp = np.cos(psi + beta), np.sin(psi + beta)
    sb, cb = np.sin(beta), np.cos(beta)
    den = 1.0 - K * ey
    sdot = v * c1 / den
    zd = np.zeros(7, dtype=complex)
    zd[D.IS] = sdot
    zd[D.IEY] = v * s1
    zd[D.IEPSI] = v * sb / D.L_R - sdot * K
    zd[D.IV] = a
    zd[D.IX] = v * cp
    zd[D.IY] = v * sp
    zd[D.IPSI] = v * sb / D.L_R
    fz = np.zeros((7, 7), dtype=complex)
    fu = np.zeros((7, 2), dtype=complex)
    ds_dey, ds_depsi, ds_dv, ds_dbeta = v * c1 * K / (den * den), -v * s1 / den, c1 / den, -v * s1 / den
    fz[D.IS, D.IEY], fz[D.IS, D.IEPSI], fz[D.IS, D.IV] = ds_dey, ds_depsi, ds_dv
    fu[D.IS, 1] = ds_dbeta * dbeta
    fz[D.IEY, D.IEPSI], fz[D.IEY, D.IV] = v * c1, s1
    fu[D.IEY, 1] = v * c1 * dbeta
    fz[D.IEPSI, D.IEY] = -K * ds_dey
    fz[D.IEPSI, D.IEPSI] = -K * ds_depsi
    fz[D.IEPSI, D.IV] = sb / D.L_R - K * ds_dv
    fu[D.IEPSI, 1] = (v * cb / D.L_R - K * ds_dbeta) * dbeta
    fu[D.IV, 0] = 1.0
    fz[D.IX, D.IV], fz[D.IX, D.IPSI] = cp, -v * sp
    fu[D.IX, 1] = -v * sp * dbeta
    fz[D.IY, D.IV], fz[D.IY, D.IPSI] = sp, v * cp
    fu[D.IY, 1] = v * cp * dbeta
    fz[D.IPSI, D.IV] = sb / D.L_R
    fu[D.IPSI, 1] = v * cb / D.L_R * dbeta
    return zd, fz, fu


def step_jac(z, u, curv, dt, n_rk):
    """oracle/dynamics.frenet_rk4_step(want_jac=True), complex-safe: (z+, A[7,7], B[7,2])."""
    h = dt / n_rk
    z = np.array(z, dtype=complex)
    u = np.asarray(u, dtype=complex)
    half = np.full(7, 0.5)
    full = np.ones(7)
    full[D.IPSI] = 0.5                      # the k4 psi quirk, kinematic_bicycle_model_frenet.py:111
    S = np.zeros((7, 9), dtype=complex)
    S[:, :7] = np.eye(7)
    E = np.zeros((2, 9))
    E[:, 7:] = np.eye(2)
    for _ in range(n_rk):
        k1, fz, fu = _rhs_jac(z, u, curv)
        d1 = fz @ S + fu @ E
        k2, fz, fu = _rhs_jac(z + h * half * k1, u, curv)
        d2 = fz @ (S + h * half[:, None] * d1) + fu @ E
        k3, fz, fu = _rhs_jac(z + h * half * k2, u, curv)
        d3 = fz @ (S + h * half[:, None] * d2) + fu @ E
        k4, fz, fu = _rhs_jac(z + h * full * k3, u, curv)
        d4 = fz @ (S + h * full[:, None] * d3) + fu @ E
        S = S + h / 6.0 * (d1 + 2 * d2 + 2 * d3 + d4)
        z = z + h / 6.0 * (k1 + 2 * k2 + 2 * k3 + k4)
    return z, S[:, :7], S[:, 7:]


def step_hessian(z, u, curv, lam, dt, n_rk, hc=1e-30):
    """sum_j lam_j d2 F_j / d(z, u)^2 [9, 9] of one step by complex step on its Jacobian."""
    H = np.zeros((9, 9))
    for a in range(9):
        zc = np.array(z, dtype=complex)
        uc = np.array(u, dtype=complex)
        if a < 7:
            zc[a] += 1j * hc
        else:
            uc[a - 7] += 1j * hc
        _, A, B = step_jac(zc, uc, curv, dt, n_rk)
        J = np.concatenate([A, B], axis=1).imag / hc     # d/dw_a of dF/dw [7, 9]
        H[:, a] = lam @ J
    return 0.5 * (H + H.T)


def vjp(P, prob, mlp, U, Y, S, status, gx=None, gu=None, gcost=None):
    """VJP of one problem.  P: nlp.Params; prob: nlp.Problem (circle rows); mlp: nlp.MLPTerm or None ('mpc');
    U[N,2], Y[M], S[M] (rows in the solver's order, oracle/solver.stage_rows / terminal_rows); cotangents gx[N+1,7],
    gu[N,2], gcost (None: zero).  Returns (gx0[7], gu_prev[2], gobs[N+1,2], ok)."""
    N = P.N
    zero = (np.zeros(7), np.zeros(2), np.zeros((N + 1, 2)), 0)
    Y, S = np.asarray(Y, dtype=np.float64), np.asarray(S, dtype=np.float64)
    if status != 0 or not (np.all(Y > 0) and np.all(S > 0) and np.all(np.isfinite(Y)) and np.all(np.isfinite(S))):
        return zero
    gx = np.zeros((N + 1, 7)) if gx is None else np.asarray(gx, dtype=np.float64)
    gu = np.zeros((N, 2)) if gu is None else np.asarray(gu, dtype=np.float64)
    gc = 0.0 if gcost is None else float(gcost)
    U = np.asarray(U, dtype=np.float64)
    Z, A, B = D.frenet_rollout(prob.x0, U, prob.curv, P.dt, P.n_rk, want_jac=True)
    # rows of every node, split by node
    rows, o = [], 0
    for k in range(N + 1):
        if k < N:
            up = prob.u_prev if k == 0 else U[k - 1]
            c, Cx, Cu, hxy = SV.stage_rows(P, prob, k, Z[k], up, U[k])
        else:
            c, Cx, Cu, hxy = SV.terminal_rows(P, prob, Z[N])
        m = len(c)
        rows.append((c, Cx, Cu, hxy, S[o:o + m], Y[o:o + m]))
        o += m
    assert o == len(Y), "row count"
    # w = (u [2N], x0 [7], u_prev [2]); total Jacobians of x_k and of zeta_k = (x_k, up_k), u_k in w
    nw = 2 * N + 9
    iu = lambda k: slice(2 * k, 2 * k + 2)
    X = np.zeros((N + 1, 7, nw))
    X[0][:, 2 * N:2 * N + 7] = np.eye(7)
    for k in range(N):
        X[k + 1] = A[k] @ X[k]
        X[k + 1][:, iu(k)] += B[k]

    def Jloc(k):                            # d(x_k, up_k, u_k)/dw  [11, nw]
        J = np.zeros((11, nw))
        J[:7] = X[k]
        if k == 0:
            J[7:9, 2 * N + 7:] = np.eye(2)
        else:
            J[7:9, iu(k - 1)] = np.eye(2)
        if k < N:
            J[9:11, iu(k)] = np.eye(2)
        return J

    # terminal cost derivatives (nlp.cost): -(s_N - s_0) or -V(s_N, v_N)
    jN = np.zeros(7); HN = np.zeros((7, 7))
    jN[D.IEY], jN[D.IEPSI] = 2 * Z[N, D.IEY], 2 * Z[N, D.IEPSI]
    HN[D.IEY, D.IEY] = HN[D.IEPSI, D.IEPSI] = 2.0
    if mlp is None:
        jN[D.IS] -= 1.0
    else:
        _, g, Hv = mlp.value(Z[N, D.IS], Z[N, D.IV], prob.nn_ctx, order=2)
        jN[D.IS] -= g[0]; jN[D.IV] -= g[1]
        HN[np.ix_([D.IS, D.IV], [D.IS, D.IV])] -= Hv
    # adjoint of the Lagrangian (x part), backward
    lam = [None] * (N + 1)
    c, Cx, Cu, hxy, s, y = rows[N]
    lam[N] = jN + Cx[:, :7].T @ s
    for k in range(N - 1, -1, -1):
        c, Cx, Cu, hxy, s, y = rows[k]
        lx = np.zeros(7); lx[D.IEY], lx[D.IEPSI] = 2 * Z[k, D.IEY], 2 * Z[k, D.IEPSI]
        lam[k] = lx + Cx[:, :7].T @ s + A[k].T @ lam[k + 1]
    # dense Hessian of L + C' Sigma C over w, and the cost gradient over w
    Hw = np.zeros((nw, nw))
    gJ = np.zeros(nw)
    Mo = np.zeros((nw, N + 1, 2))             # d(grad_w L + C' Sigma c)/d o_k
    for k in range(N + 1):
        c, Cx, Cu, hxy, s, y = rows[k]
        sig = s / y
        J = Jloc(k)
        Hl = np.zeros((11, 11))
        if k < N:
            Hl[D.IEY, D.IEY] = Hl[D.IEPSI, D.IEPSI] = 2.0
            Hl[9, 9] = Hl[10, 10] = 2 * P.w_u
            Hdyn = step_hessian(Z[k], U[k], prob.curv, lam[k + 1], P.dt, P.n_rk)
            idx = list(range(7)) + [9, 10]
            Hl[np.ix_(idx, idx)] += Hdyn
            gl = np.zeros(11)
            gl[D.IEY], gl[D.IEPSI] = 2 * Z[k, D.IEY], 2 * Z[k, D.IEPSI]
            gl[9:] = 2 * P.w_u * U[k]
        else:
            Hl[:7, :7] += HN
            gl = np.zeros(11); gl[:7] = jN
        Gr = np.concatenate([Cx, Cu], axis=1)  # [m, 11] row gradients in (x, up, u)
        Hl += Gr.T @ (sig[:, None] * Gr)
        for i, h in enumerate(hxy):
            if not np.isscalar(h):
                Hl[np.ix_([D.IX, D.IY], [D.IX, D.IY])] += s[i] * h
                if k >= 1:                      # the collision row: dc/do = -dc/dp, d2c/dp do = -d2c/dp2
                    Ci = Gr[i] @ J              # total gradient of the row over w
                    n = -Cx[i, [D.IX, D.IY]]    # dc/do
                    Mo[:, k, :] += -(s[i] * (J[[D.IX, D.IY]].T @ h)) + sig[i] * np.outer(Ci, n)
        Hw += J.T @ Hl @ J
        gJ += J.T @ gl
    if mlp is None:
        gJ[2 * N + D.IS] += 1.0                 # -(s_N - s_0): s_0 = x0[s] directly
    K = Hw[:2 * N, :2 * N]
    try:
        Lc = np.linalg.cholesky(0.5 * (K + K.T))
    except np.linalg.LinAlgError:
        return zero
    # reduced cotangent on u and direct terms on (x0, u_prev)
    gw = gc * gJ
    for k in range(N + 1):
        gw += X[k].T @ gx[k]
    gw[:2 * N] += gu.ravel()
    r = gw[:2 * N]
    zsol = np.linalg.solve(Lc.T, np.linalg.solve(Lc, r))
    gz0 = gw[2 * N:] - Hw[2 * N:, :2 * N] @ zsol
    gobs = -np.einsum("w,wkj->kj", zsol, Mo[:2 * N])
    if not (np.all(np.isfinite(gz0)) and np.all(np.isfinite(gobs))):
        return zero
    return gz0[:7].copy(), gz0[7:].copy(), gobs, 1
