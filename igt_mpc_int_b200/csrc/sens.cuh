// sens.cuh -- vector-Jacobian product of one batched solve through its converged KKT system, one problem per thread.
//
// A solve returns (u, y, s): controls, row slacks and row multipliers with
//   grad_u L(u, s; theta) = 0,   c(u; theta) + y = 0,   s_i y_i = const_i,      L = J + s' c,
// in the single-shooting form of the solver (x = rollout(x0, u), zeta_k = [x_k; u_{k-1}], theta = (x0, u_prev, obs_xy)).
// Linearising these equations at the returned point with every row's product s_i y_i held fixed gives
//   (H + C' S Y^-1 C) du = -(L_u,theta + C' S Y^-1 c_theta) dtheta,
// H the EXACT Hessian of the Lagrangian in u (stage cost, value term, the circle rows' 2x2 blocks and the second
// derivatives of the discrete RK4 step weighted by the adjoint), C = dc/du.  The cotangents on x, u and cost are the
// linear terms of a stage-wise LQ problem on this Hessian, so one Riccati backward sweep and one forward sweep give
//   d(gx0, gu_prev) = the value gradient of the augmented initial state zeta_0 = [x0; u_prev],
//   gobs[k]          = -(s H_c dp_k + sigma n (n . dp_k)) of the collision row of node k (dp_k: the forward sweep's
//                      position change, n = (p - o)/|p - o|, H_c = d2c/dp2, sigma = s/y).
// The RK4 second derivatives come from a forward-mode dual number pushed through the solver's own templated step
// (rk4_core<Dual, true>), so the discretisation -- with its k4 psi quirk -- is differentiated, not re-derived; the
// pw_const curvature is locally constant (dK/ds = 0), as in the solver.  f64, circle rows only (DESIGN.md section 10).
// __host__ __device__ like solver_core.cuh: tests/hostsim runs the same code on the CPU.
#pragma once
#include "solver_core.cuh"

namespace igt {

// ------------------------------------------------------------------ forward-mode dual number --
struct Dual {
    double v, d;
    Dual() = default;
    IGT_HD Dual(double x) : v(x), d(0.0) {}
    IGT_HD Dual(double x, double dx) : v(x), d(dx) {}
};
IGT_HD Dual operator+(Dual a, Dual b) { return Dual(a.v + b.v, a.d + b.d); }
IGT_HD Dual operator-(Dual a, Dual b) { return Dual(a.v - b.v, a.d - b.d); }
IGT_HD Dual operator-(Dual a) { return Dual(-a.v, -a.d); }
IGT_HD Dual operator*(Dual a, Dual b) { return Dual(a.v * b.v, a.d * b.v + a.v * b.d); }
IGT_HD Dual operator/(Dual a, Dual b) { const double q = a.v / b.v; return Dual(q, (a.d - q * b.d) / b.v); }
IGT_HD Dual &operator+=(Dual &a, Dual b) { a = a + b; return a; }
IGT_HD Dual &operator-=(Dual &a, Dual b) { a = a - b; return a; }
IGT_HD Dual &operator*=(Dual &a, Dual b) { a = a * b; return a; }
IGT_HD bool operator<(Dual a, Dual b) { return a.v < b.v; }
IGT_HD bool operator>(Dual a, Dual b) { return a.v > b.v; }
IGT_HD bool operator<=(Dual a, Dual b) { return a.v <= b.v; }
IGT_HD bool operator>=(Dual a, Dual b) { return a.v >= b.v; }
IGT_HD bool operator==(Dual a, Dual b) { return a.v == b.v; }
IGT_HD bool operator!=(Dual a, Dual b) { return a.v != b.v; }
IGT_HD Dual sqrt(Dual a) { const double r = ::sqrt(a.v); return Dual(r, a.d / (2.0 * r)); }
IGT_HD Dual tan(Dual a) { const double t = ::tan(a.v); return Dual(t, a.d * (1.0 + t * t)); }
using ::sqrt;   // (the overloads above hide the double ones from the code of this namespace that follows)
using ::tan;
IGT_HD void sincos_t(Dual x, Dual *s, Dual *c)
{
    double sv, cv;
    sincos(x.v, &sv, &cv);
    *s = Dual(sv, cv * x.d);
    *c = Dual(cv, -sv * x.d);
}
// the solver's short Taylor pairs replace sin / cos to < 1e-21; the dual takes the functions themselves
IGT_HD void sincos_small2(Dual d1, Dual d2, Dual &s1, Dual &c1, Dual &s2, Dual &c2)
{
    sincos_t(d1, &s1, &c1);
    sincos_t(d2, &s2, &c2);
}

// ------------------------------------------------------------------ problem io -----------------
struct SensIO {
    const double *x0, *u_prev, *curv, *obs, *ctx;   // the solve's inputs: [B,7] [B,2] [B,3] [B,N+1,2] [B,4] or null
    const int *net_idx = nullptr;                    // [B] bank slots (with ctx) or null: DevParams' network
    const MlpNet<double> *nets = nullptr;
    const double *u, *slack, *mult;                  // the solve's outputs: [B,N,2] [B,M] [B,M]
    const int *status;                               // [B]
    const double *gx, *gu, *gcost;                   // cotangents [B,N+1,7] [B,N,2] [B]; null = zero
    double *gx0, *gu_prev, *gobs;                    // [B,7] [B,2] [B,N+1,2]
    int *ok;                                         // [B]
};

// per-problem scratch: trajectory, feedback gains, feed-forward terms; element e at base[e * stride]
IGT_HD constexpr int sens_ws_size(int N) { return NZ * (N + 1) + 2 * NA * N + 2 * N; }
struct SensWs {
    double *base;
    long stride;
    int N;
    IGT_HD double &Z(int k, int i) const { return base[(long)(k * NZ + i) * stride]; }
    IGT_HD double &K(int k, int r, int j) const { return base[(long)(NZ * (N + 1) + (k * 2 + r) * NA + j) * stride]; }
    IGT_HD double &kf(int k, int r) const { return base[(long)(NZ * (N + 1) + 2 * NA * N + k * 2 + r) * stride]; }
};

// d zeta+ / d (zeta, u) [9][11] from the compact sensitivities Sc of one step (see rk4_core, expand_sens)
IGT_HD void sens_F(const DevParams<double> &P, const double *Sc, double (*F)[NW])
{
    double S[NZ][NSEED];
    expand_sens(P, Sc, S);
    const int wi[NSEED] = { IEY, IEPSI, IV, IPSI, IUA, IUD };
    for (int i = 0; i < NA; i++)
        for (int j = 0; j < NW; j++) F[i][j] = 0.0;
    for (int i = 0; i < NZ; i++)
        for (int m = 0; m < NSEED; m++) F[i][wi[m]] = S[i][m];
    F[IX][IX] = F[IY][IY] = F[IS][IS] = 1.0;                      // x, y feed themselves only; dK/ds = 0
    F[IPA][IUA] = F[IPD][IUD] = 1.0;                               // next stage's previous input
}

// sum_i lam_i d2 F_i / dw2 over w = (zeta, u) [11][11]: one dual pass per seed (ey, epsi, v, psi, a, df) through the
// sensitivity step; the derivative part of the sensitivities is one column of the weighted Hessian
IGT_HD void sens_dyn_hessian(const DevParams<double> &P, const double *z, const double *u, const double *curv,
                             const double *lam, double (*Hd)[NW])
{
    const int wi[NSEED] = { IEY, IEPSI, IV, IPSI, IUA, IUD };
    for (int i = 0; i < NW; i++)
        for (int j = 0; j < NW; j++) Hd[i][j] = 0.0;
    for (int j = 0; j < NSEED; j++) {
        Dual zd[NZ], ud[2], cd[3], zn[NZ], Sc[NSENS];
        for (int i = 0; i < NZ; i++) zd[i] = Dual(z[i], wi[j] == i ? 1.0 : 0.0);
        ud[0] = Dual(u[0], wi[j] == IUA ? 1.0 : 0.0);
        ud[1] = Dual(u[1], wi[j] == IUD ? 1.0 : 0.0);
        for (int i = 0; i < 3; i++) cd[i] = Dual(curv[i]);
        rk4_core<Dual, true>(P, zd, ud, cd, zn, Sc);
        double dSc[NSENS], dS[NZ][NSEED];
        for (int e = 0; e < NSENS; e++) dSc[e] = Sc[e].d;
        expand_sens(P, dSc, dS);
        dS[IPSI][3] = dS[IV][2] = dS[IV][4] = 0.0;                 // the constant entries expand_sens fills in
        for (int m = 0; m < NSEED; m++) {
            double acc = 0.0;
            for (int i = 0; i < NZ; i++) acc += lam[i] * dS[i][m];
            Hd[wi[m]][wi[j]] = acc;
        }
    }
    for (int i = 0; i < NW; i++)                                   // symmetric up to rounding: take the mean
        for (int j = i + 1; j < NW; j++) { const double a = 0.5 * (Hd[i][j] + Hd[j][i]); Hd[i][j] = Hd[j][i] = a; }
}

// Rows of node k at the returned point: adds sum_i (sigma_i g_i g_i' + s_i d2c_i) to Hw[11][11] and sum_i s_i g_i to
// lw[11] (the Lagrangian's row part).  Returns false if a slack or multiplier is not positive and finite.
IGT_HD bool sens_rows(const DevParams<double> &P, int k, const double *z, const double *up, const double *u, double ox,
                      double oy, const double *yv, const double *sv, double (*Hw)[NW], double *lw)
{
    bool good = true;
    visit_rows<true, false>(P, k, z, up, u, ox, oy, 0.0, [&](auto, int r, double, auto I0, double g0, auto I1, double g1,
                                                             auto, double, double hxx, double hxy, double hyy) {
        constexpr int i0 = decltype(I0)::value, i1 = decltype(I1)::value;
        const double y = yv[r], s = sv[r];
        if (!(y > 0.0 && s > 0.0 && y < 1e300 && s < 1e300)) { good = false; return; }
        const double sig = s / y;
        lw[i0] += s * g0;
        Hw[i0][i0] += sig * g0 * g0;
        if constexpr (i1 >= 0) {
            lw[i1] += s * g1;
            Hw[i1][i1] += sig * g1 * g1;
            Hw[i0][i1] += sig * g0 * g1;
            Hw[i1][i0] += sig * g0 * g1;
        }
        Hw[IX][IX] += s * hxx; Hw[IX][IY] += s * hxy; Hw[IY][IX] += s * hxy; Hw[IY][IY] += s * hyy;
    });
    return good;
}

// collision row of node k >= 1 at position p: gobs[k] = -(s H_c dp + sigma n (n . dp))
IGT_HD void sens_gobs(const DevParams<double> &P, double px, double py, double ox, double oy, double y, double s,
                      double dpx, double dpy, double *g)
{
    double dx = px - ox, dy = py - oy;
    double dist = sqrt(dx * dx + dy * dy);
    dist = dist < 1e-9 ? 1e-9 : dist;
    const double id = 1.0 / dist, nx = dx * id, ny = dy * id;
    const double hxx = -(1.0 - nx * nx) * id, hxy = nx * ny * id, hyy = -(1.0 - ny * ny) * id;   // as visit_rows
    const double nd = nx * dpx + ny * dpy, sig = s / y;
    g[0] = -(s * (hxx * dpx + hxy * dpy) + sig * nx * nd);
    g[1] = -(s * (hxy * dpx + hyy * dpy) + sig * ny * nd);
}

// The VJP of problem p.  mlp_scr: [2][6][mlp_width] scratch of the value term (gt_mpc).  Writes zero gradients and
// ok = 0 when status[p] != 0, when a slack or multiplier is not positive, when a stage's Quu is not positive definite
// (no regularisation here) or when a result is not finite.
template <bool BANK>
IGT_HD void vjp_problem(const DevParams<double> &P, const SensIO &io, long p, const SensWs &w, double *mlp_scr, int mlp_width)
{
    const int N = P.N, M = row_total(N, P.n_cinf);
    double *gx0 = io.gx0 + p * NZ, *gup = io.gu_prev + p * 2, *gob = io.gobs + p * (N + 1) * 2;
    for (int i = 0; i < NZ; i++) gx0[i] = 0.0;
    gup[0] = gup[1] = 0.0;
    for (int i = 0; i < 2 * (N + 1); i++) gob[i] = 0.0;
    io.ok[p] = 0;
    if (io.status[p] != 0) return;
    const bool gt = io.ctx != nullptr;
    const MlpNet<double> *net = nullptr;
    if (BANK && gt) {
        const int ni = io.net_idx[p];
        if (!((unsigned)ni < (unsigned)MAX_MLP_NETS && io.nets[ni].n_layers > 0)) return;
        net = io.nets + ni;
    }
    double x0[NZ], uprev[2] = { io.u_prev[2 * p], io.u_prev[2 * p + 1] }, curv[3], ctx[4] = { 0, 0, 0, 0 };
    for (int i = 0; i < NZ; i++) x0[i] = io.x0[p * NZ + i];
    for (int i = 0; i < 3; i++) curv[i] = io.curv[3 * p + i];
    if (gt) for (int i = 0; i < 4; i++) ctx[i] = io.ctx[4 * p + i];
    const double *U = io.u + p * N * 2, *Y = io.slack + p * M, *S = io.mult + p * M, *obs = io.obs + p * (N + 1) * 2;
    const double *gx = io.gx ? io.gx + p * (N + 1) * NZ : nullptr, *gu = io.gu ? io.gu + p * N * 2 : nullptr;
    const double gc = io.gcost ? io.gcost[p] : 0.0;
    // the solve's trajectory (the same step code, so the same bits)
    {
        double z[NZ];
        for (int i = 0; i < NZ; i++) { z[i] = x0[i]; w.Z(0, i) = z[i]; }
        for (int k = 0; k < N; k++) {
            double zn[NZ];
            rk4_step(P, z, U + 2 * k, curv, zn);
            for (int i = 0; i < NZ; i++) { z[i] = zn[i]; w.Z(k + 1, i) = zn[i]; }
        }
    }
    // terminal node: value V[9][9], linear term v[9] (cotangents), Lagrangian adjoint lam[9]
    double V[NA][NA], v[NA], lam[NA];
    {
        double z[NZ], Hw[NW][NW], lw[NW];
        for (int i = 0; i < NZ; i++) z[i] = w.Z(N, i);
        for (int i = 0; i < NW; i++) { lw[i] = 0.0; for (int j = 0; j < NW; j++) Hw[i][j] = 0.0; }
        const double up[2] = { U[2 * (N - 1)], U[2 * (N - 1) + 1] }, u0[2] = { 0.0, 0.0 };
        const int o = row_off(N, P.n_cinf, N);
        if (!sens_rows(P, N, z, up, u0, obs[2 * N], obs[2 * N + 1], Y + o, S + o, Hw, lw)) return;
        TermVal<double> t;
        if (!gt) { t.gs = 1.0; t.gv = t.Hss = t.Hsv = t.Hvv = 0.0; }
        else if (BANK) mlp_eval_body(*net, z[IS], z[IV], ctx, mlp_scr, mlp_scr + 6 * mlp_width, mlp_width, t, true);
        else mlp_eval_body(P, z[IS], z[IV], ctx, mlp_scr, mlp_scr + 6 * mlp_width, mlp_width, t, true);
        double jx[NA];                                             // gradient of the terminal cost in zeta_N
        for (int i = 0; i < NA; i++) jx[i] = 0.0;
        jx[IEY] = 2.0 * z[IEY]; jx[IEPSI] = 2.0 * z[IEPSI]; jx[IS] = -t.gs; jx[IV] = -t.gv;
        Hw[IEY][IEY] += 2.0; Hw[IEPSI][IEPSI] += 2.0;
        Hw[IS][IS] -= t.Hss; Hw[IS][IV] -= t.Hsv; Hw[IV][IS] -= t.Hsv; Hw[IV][IV] -= t.Hvv;
        for (int i = 0; i < NA; i++) {
            lam[i] = jx[i] + lw[i];
            v[i] = gc * jx[i] + (gx && i < NZ ? gx[N * NZ + i] : 0.0);
            for (int j = 0; j < NA; j++) V[i][j] = Hw[i][j];
        }
    }
    for (int k = N - 1; k >= 0; k--) {
        double z[NZ], up[2], u[2] = { U[2 * k], U[2 * k + 1] }, zn[NZ], Sc[NSENS], F[NA][NW], H[NW][NW], g[NW], lw[NW];
        for (int i = 0; i < NZ; i++) z[i] = w.Z(k, i);
        if (k == 0) { up[0] = uprev[0]; up[1] = uprev[1]; } else { up[0] = U[2 * k - 2]; up[1] = U[2 * k - 1]; }
        rk4_step_sens(P, z, u, curv, zn, Sc);
        sens_F(P, Sc, F);
        sens_dyn_hessian(P, z, u, curv, lam, H);                   // H starts as the weighted dynamics term
        for (int i = 0; i < NW; i++) lw[i] = 0.0;
        const int o = row_off(N, P.n_cinf, k);
        if (!sens_rows(P, k, z, up, u, obs[2 * k], obs[2 * k + 1], Y + o, S + o, H, lw)) return;
        // stage cost (mpc.py:359-364)
        double lx[NW];
        for (int i = 0; i < NW; i++) lx[i] = 0.0;
        lx[IEY] = 2.0 * z[IEY]; lx[IEPSI] = 2.0 * z[IEPSI]; lx[IUA] = 2.0 * P.w_u * u[0]; lx[IUD] = 2.0 * P.w_u * u[1];
        H[IEY][IEY] += 2.0; H[IEPSI][IEPSI] += 2.0; H[IUA][IUA] += 2.0 * P.w_u; H[IUD][IUD] += 2.0 * P.w_u;
        // H += F' V F, g = F' v + cotangent terms
        for (int i = 0; i < NW; i++) {
            double acc = 0.0;
            for (int a = 0; a < NA; a++) acc += F[a][i] * v[a];
            g[i] = acc + gc * lx[i];
            for (int j = 0; j < NW; j++) {
                double hh = 0.0;
                for (int a = 0; a < NA; a++) {
                    if (F[a][i] == 0.0) continue;
                    double vf = 0.0;
                    for (int c = 0; c < NA; c++) vf += V[a][c] * F[c][j];
                    hh += F[a][i] * vf;
                }
                H[i][j] += hh;
            }
        }
        if (gx) for (int i = 0; i < NZ; i++) g[i] += gx[k * NZ + i];
        if (gu) { g[IUA] += gu[2 * k]; g[IUD] += gu[2 * k + 1]; }
        if (k == 0 && !gt) g[IS] += gc;                            // 'mpc' cost -(s_N - s_0): s_0 enters directly
        // the next adjoint: lam_k = grad of the stage's Lagrangian part in zeta + F_zeta' lam_{k+1}
        double ln[NA];
        for (int i = 0; i < NA; i++) {
            double acc = lx[i] + lw[i];
            for (int a = 0; a < NA; a++) acc += F[a][i] * lam[a];
            ln[i] = acc;
        }
        for (int i = 0; i < NA; i++) lam[i] = ln[i];
        // Riccati step, no regularisation: Quu must be positive definite
        const double q00 = H[IUA][IUA], q11 = H[IUD][IUD], q01 = 0.5 * (H[IUA][IUD] + H[IUD][IUA]);
        const double det = q00 * q11 - q01 * q01;
        if (!(q00 > 0.0 && det > 0.0)) return;
        const double i00 = q11 / det, i11 = q00 / det, i01 = -q01 / det;
        const double k0 = -(i00 * g[IUA] + i01 * g[IUD]), k1 = -(i01 * g[IUA] + i11 * g[IUD]);
        double K0[NA], K1[NA];
        for (int j = 0; j < NA; j++) {
            const double ha = H[IUA][j], hd = H[IUD][j];
            K0[j] = -(i00 * ha + i01 * hd); K1[j] = -(i01 * ha + i11 * hd);
            w.K(k, 0, j) = K0[j]; w.K(k, 1, j) = K1[j];
        }
        w.kf(k, 0) = k0; w.kf(k, 1) = k1;
        for (int i = 0; i < NA; i++) {
            v[i] = g[i] + H[i][IUA] * k0 + H[i][IUD] * k1;
            for (int j = 0; j < NA; j++) V[i][j] = H[i][j] + H[i][IUA] * K0[j] + H[i][IUD] * K1[j];
        }
        for (int i = 0; i < NA; i++)
            for (int j = i + 1; j < NA; j++) { const double a = 0.5 * (V[i][j] + V[j][i]); V[i][j] = V[j][i] = a; }
    }
    // forward sweep: the state change of the LQ solution, and the collision rows' obstacle gradients
    double gz[NZ + 2];
    for (int i = 0; i < NZ; i++) gz[i] = v[i];
    gz[NZ] = v[IPA]; gz[NZ + 1] = v[IPD];
    double gobs[2 * 65];
    for (int i = 0; i < 2 * (N + 1); i++) gobs[i] = 0.0;
    double dz[NA];
    for (int i = 0; i < NA; i++) dz[i] = 0.0;
    bool finite = true;
    for (int i = 0; i < NZ + 2; i++) finite = finite && fabs(gz[i]) < 1e300;
    for (int k = 0; k < N; k++) {
        double z[NZ], zn[NZ], Sc[NSENS], F[NA][NW], dw[NW];
        for (int i = 0; i < NZ; i++) z[i] = w.Z(k, i);
        rk4_step_sens(P, z, U + 2 * k, curv, zn, Sc);
        sens_F(P, Sc, F);
        for (int i = 0; i < NA; i++) dw[i] = dz[i];
        for (int r = 0; r < 2; r++) {
            double acc = w.kf(k, r);
            for (int j = 0; j < NA; j++) acc += w.K(k, r, j) * dz[j];
            dw[NA + r] = acc;
        }
        for (int i = 0; i < NA; i++) {
            double acc = 0.0;
            for (int j = 0; j < NW; j++) acc += F[i][j] * dw[j];
            dz[i] = acc;
        }
        const int r = row_off(N, P.n_cinf, k + 1) + (k + 1 == N ? 2 : 4);   // the collision row of node k + 1
        sens_gobs(P, zn[IX], zn[IY], obs[2 * (k + 1)], obs[2 * (k + 1) + 1], Y[r], S[r], dz[IX], dz[IY], gobs + 2 * (k + 1));
        finite = finite && fabs(gobs[2 * (k + 1)]) < 1e300 && fabs(gobs[2 * (k + 1) + 1]) < 1e300;
    }
    if (!finite) return;
    for (int i = 0; i < NZ; i++) gx0[i] = gz[i];
    gup[0] = gz[NZ]; gup[1] = gz[NZ + 1];
    for (int i = 0; i < 2 * (N + 1); i++) gob[i] = gobs[i];
    io.ok[p] = 1;
}

}  // namespace igt
