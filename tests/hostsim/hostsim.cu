// tests/hostsim -- TEST HARNESS ONLY.  Runs the product's per-thread solver code
// (igt_mpc_int_b200/csrc/solver_core.cuh) on the CPU, one "thread" after another, so that the
// kernel logic can be checked against the oracle on machines without a GPU.  Never loaded by the
// package; the product path is the CUDA library and fails loudly without a GPU.
#include <vector>
#include <cstdlib>
#include "../../igt_mpc_int_b200/csrc/params_host.hpp"

using namespace igt;

template <typename T, bool OBCA = false>
static int run(const igt_params *p, int B, const double *x0, const double *u_prev, const double *curv,
               const double *obs, const double *obs_psi, const double *ctx, const double *u_init, double *x, double *u, double *cost,
               double *viol, int *status, int *iters, int n_layers, const int *dims, const double *const *W,
               const double *const *b, const double *Wn, const double *mu_f, double sigma_t, double mu_t, bool lanes = false)
{
    DevParams<T> P;
    fill_dev_params(*p, P);
    std::vector<std::vector<T>> keep;
    int width = 6;
    if (n_layers > 0) {
        P.n_layers = n_layers;
        for (int l = 0; l <= n_layers; l++) { P.dims[l] = dims[l]; if (dims[l] > width) width = dims[l]; }
        for (int l = 0; l < n_layers; l++) {
            keep.emplace_back(W[l], W[l] + (size_t)dims[l] * dims[l + 1]);
            P.W[l] = keep.back().data();
            keep.emplace_back(b[l], b[l] + dims[l + 1]);
            P.b[l] = keep.back().data();
        }
        for (int i = 0; i < 36; i++) P.Wn[i] = T(Wn[i]);
        for (int i = 0; i < 6; i++) P.mu_f[i] = T(mu_f[i]);
        P.sigma_t = T(sigma_t); P.mu_t = T(mu_t);
    }
    WsLayout L; L.init(p->N, p->n_cinf, OBCA ? NGE_OBCA : NGE, OBCA ? NHE_OBCA : NHE);
    std::vector<T> ws((size_t)L.total * 32);
    std::vector<T> scratch((size_t)12 * width);
    std::vector<double> guess((size_t)2 * p->N);
    ProbIO io = { x0, u_prev, curv, obs, ctx, u_init, x, u, cost, viol, status, iters };
    io.obs_psi = obs_psi;
    if (!lanes) {
        for (long q = 0; q < B; q++) solve_problem<T, OBCA>(P, io, ws.data(), q % 32, q, guess.data(), scratch.data(), width);
        return 0;
    }
    // persistent lanes, as in the kernels: one solver object per slot, bound once; slot q % 32 solves problems
    // q, q + 32, ... one after the other without the object being rebuilt in between
    std::vector<Solver<T, Ws<T, 32, OBCA>>> sv;
    sv.reserve(32);
    for (int s = 0; s < 32; s++) {
        sv.emplace_back(P);
        sv[s].w.init_layout(P.N, P.n_cinf);
        sv[s].w.bind(ws.data(), s);
        sv[s].mlp_scratch = scratch.data(); sv[s].mlp_width = width;
    }
    for (long q = 0; q < B; q++) solve_bound(sv[q % 32], io, q, guess.data());
    return 0;
}

extern "C" {
int hostsim_default_params(igt_params *p, int precision) { return default_params(p, precision); }

// lanes = 0: a fresh solver object per problem; lanes != 0: one object per slot, reused for every 32nd problem (the
// kernels' persistent lanes).  Both write problem q's results to row q.
int hostsim_solve(const igt_params *p, int B, const double *x0, const double *u_prev, const double *curv,
                  const double *obs, const double *ctx, const double *u_init, double *x, double *u, double *cost,
                  double *viol, int *status, int *iters, int n_layers, const int *dims, const double *const *W,
                  const double *const *b, const double *Wn, const double *mu_f, double sigma_t, double mu_t, int lanes)
{
    if (p->precision == IGT_PREC_F64)
        return run<double>(p, B, x0, u_prev, curv, obs, nullptr, ctx, u_init, x, u, cost, viol, status, iters, n_layers, dims, W, b, Wn, mu_f, sigma_t, mu_t, lanes != 0);
    return run<float>(p, B, x0, u_prev, curv, obs, nullptr, ctx, u_init, x, u, cost, viol, status, iters, n_layers, dims, W, b, Wn, mu_f, sigma_t, mu_t, lanes != 0);
}

// OBCA collision mode (obs_psi[B][N+1] obstacle headings), fp64, 'mpc' cost.  lanes: as in hostsim_solve
int hostsim_solve_obca(const igt_params *p, int B, const double *x0, const double *u_prev, const double *curv,
                       const double *obs, const double *obs_psi, const double *u_init, double *x, double *u, double *cost,
                       double *viol, int *status, int *iters, int lanes)
{
    return run<double, true>(p, B, x0, u_prev, curv, obs, obs_psi, nullptr, u_init, x, u, cost, viol, status, iters, 0,
                             nullptr, nullptr, nullptr, nullptr, nullptr, 0.0, 0.0, lanes != 0);
}

// rectangle signed distance + gradient (csrc/obca.cuh) for n pose pairs: ego[n][3], obs[n][3] -> d[n], g[n][3]
int hostsim_rect_sdist(int n, const double *ego, const double *obs, double *d, double *g)
{
    for (int i = 0; i < n; i++)
        d[i] = obca_rect_sdist(ego[3 * i], ego[3 * i + 1], ego[3 * i + 2], obs[3 * i], obs[3 * i + 1], obs[3 * i + 2], g + 3 * i);
    return 0;
}

// rollout of the product's templated dynamics on the host (fp32 plain / fp64), with sensitivities
int hostsim_rollout(const igt_params *p, int B, int prec, const double *z0, const double *U, const double *curv,
                    double *Z, double *A, double *Bm)
{
    const int N = p->N;
    if (prec == IGT_PREC_F64) {
        DevParams<double> P; fill_dev_params(*p, P);
        for (long q = 0; q < B; q++) {
            double z[NZ], c[3] = { curv[3 * q], curv[3 * q + 1], curv[3 * q + 2] };
            for (int i = 0; i < NZ; i++) { z[i] = z0[q * NZ + i]; Z[q * (N + 1) * NZ + i] = z[i]; }
            for (int k = 0; k < N; k++) {
                double u[2] = { U[(q * N + k) * 2], U[(q * N + k) * 2 + 1] }, zn[NZ], Sc[NSENS], S[NZ][NSEED];
                rk4_step_sens(P, z, u, c, zn, Sc);
                expand_sens(P, Sc, S);
                double zv[NZ];
                rk4_step(P, z, u, c, zv);
                for (int i = 0; i < NZ; i++) { if (zv[i] != zn[i]) return 1; }
                if (A) {
                    double *Ak = A + (q * N + k) * 49, *Bk = Bm + (q * N + k) * 14;
                    for (int i = 0; i < NZ; i++) {
                        for (int j = 0; j < NZ; j++) Ak[i * NZ + j] = (i == j && j < 3) ? 1.0 : 0.0;
                        Ak[i * NZ + IEY] = S[i][0]; Ak[i * NZ + IEPSI] = S[i][1]; Ak[i * NZ + IV] = S[i][2]; Ak[i * NZ + IPSI] = S[i][3];
                        Bk[i * 2] = S[i][4]; Bk[i * 2 + 1] = S[i][5];
                    }
                }
                for (int i = 0; i < NZ; i++) { z[i] = zn[i]; Z[(q * (N + 1) + k + 1) * NZ + i] = zn[i]; }
            }
        }
    } else {
        DevParams<float> P; fill_dev_params(*p, P);
        for (long q = 0; q < B; q++) {
            float z[NZ], c[3] = { (float)curv[3 * q], (float)curv[3 * q + 1], (float)curv[3 * q + 2] };
            for (int i = 0; i < NZ; i++) { z[i] = (float)z0[q * NZ + i]; Z[q * (N + 1) * NZ + i] = z[i]; }
            for (int k = 0; k < N; k++) {
                float u[2] = { (float)U[(q * N + k) * 2], (float)U[(q * N + k) * 2 + 1] }, zn[NZ];
                rk4_step(P, z, u, c, zn);
                for (int i = 0; i < NZ; i++) { z[i] = zn[i]; Z[(q * (N + 1) + k + 1) * NZ + i] = zn[i]; }
            }
        }
    }
    return 0;
}
}
