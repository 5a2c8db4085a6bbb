// tests/hostsim -- TEST HARNESS ONLY.  Runs the product's dual-exporting solve epilogue (Solver::write_duals,
// csrc/solver_core.cuh) and its VJP (csrc/sens.cuh) on the CPU, one "thread" after another, so that the gradient code
// can be checked against the oracle on machines without a GPU.  Never loaded by the package.
#include <vector>
#include "../../igt_mpc_int_b200/csrc/params_host.hpp"
#include "../../igt_mpc_int_b200/csrc/sens.cuh"

using namespace igt;

// the handle's value network in P (slot 0 of a handle); returns the widest layer (6 without a network)
static int set_net(DevParams<double> &P, std::vector<std::vector<double>> &keep, int n_layers, const int *dims,
                   const double *const *W, const double *const *b, const double *Wn, const double *mu_f, double sigma_t,
                   double mu_t)
{
    int width = 6;
    P.n_layers = n_layers;
    if (n_layers <= 0) return width;
    for (int l = 0; l <= n_layers; l++) { P.dims[l] = dims[l]; if (dims[l] > width) width = dims[l]; }
    for (int l = 0; l < n_layers; l++) {
        keep.emplace_back(W[l], W[l] + (size_t)dims[l] * dims[l + 1]);
        P.W[l] = keep.back().data();
        keep.emplace_back(b[l], b[l] + dims[l + 1]);
        P.b[l] = keep.back().data();
    }
    for (int i = 0; i < 36; i++) P.Wn[i] = Wn[i];
    for (int i = 0; i < 6; i++) P.mu_f[i] = mu_f[i];
    P.sigma_t = sigma_t; P.mu_t = mu_t;
    return width;
}

extern "C" {
int senshost_default_params(igt_params *p, int precision) { return default_params(p, precision); }

// fp64 circle-mode solve (fresh solver object per problem) that also writes every row's final slack and multiplier,
// slack[B][M], mult[B][M] (Solver::write_duals, the epilogue of the dual-exporting kernels)
int senshost_solve_duals(const igt_params *p, int B, const double *x0, const double *u_prev, const double *curv,
                         const double *obs, const double *ctx, const double *u_init, double *x, double *u, double *cost,
                         double *viol, int *status, int *iters, double *slack, double *mult, int n_layers, const int *dims,
                         const double *const *W, const double *const *b, const double *Wn, const double *mu_f, double sigma_t,
                         double mu_t)
{
    DevParams<double> P;
    fill_dev_params(*p, P);
    std::vector<std::vector<double>> keep;
    const int width = set_net(P, keep, n_layers, dims, W, b, Wn, mu_f, sigma_t, mu_t);
    WsLayout L; L.init(p->N, p->n_cinf);
    std::vector<double> ws((size_t)L.total * 32), scratch((size_t)12 * width), guess((size_t)2 * p->N);
    ProbIO io = { x0, u_prev, curv, obs, ctx, u_init, x, u, cost, viol, status, iters };
    for (long q = 0; q < B; q++) {
        Solver<double> sv(P);
        sv.w.init_layout(P.N, P.n_cinf);
        sv.w.bind(ws.data(), q % 32);
        sv.mlp_scratch = scratch.data(); sv.mlp_width = width;
        solve_bound(sv, io, q, guess.data());
        sv.write_duals(slack, mult, q);
    }
    return 0;
}

// the VJP of csrc/sens.cuh (vjp_problem) for B problems, one after the other; gx, gu, gcost may be null
int senshost_vjp(const igt_params *p, int B, const double *x0, const double *u_prev, const double *curv, const double *obs,
                 const double *ctx, const double *u, const double *slack, const double *mult, const int *status,
                 const double *gx, const double *gu, const double *gcost, double *gx0, double *gu_prev, double *gobs, int *ok,
                 int n_layers, const int *dims, const double *const *W, const double *const *b, const double *Wn,
                 const double *mu_f, double sigma_t, double mu_t)
{
    DevParams<double> P;
    fill_dev_params(*p, P);
    std::vector<std::vector<double>> keep;
    const int width = set_net(P, keep, n_layers, dims, W, b, Wn, mu_f, sigma_t, mu_t);
    std::vector<double> ws(sens_ws_size(p->N)), scratch((size_t)12 * width);
    SensIO io = { x0, u_prev, curv, obs, ctx, nullptr, nullptr, u, slack, mult, status, gx, gu, gcost, gx0, gu_prev, gobs, ok };
    const SensWs w = { ws.data(), 1, p->N };
    for (long q = 0; q < B; q++) vjp_problem<false>(P, io, q, w, scratch.data(), width);
    return 0;
}
}
