// solver_core.cuh -- per-problem interior-point iLQR for the IGT-MPC NLP, one problem per thread.
//
// Replaces the arithmetic behind reference mpc.py:383-406 (opti.solve() -> CasADi -> IPOPT).
// The NLP is the one assembled in mpc.py:147-160:
//   dynamics   4-substep RK4 Frenet kinematic bicycle, common/kinematic_bicycle_model_frenet.py:69-185
//   rows       mpc.py:177-180 (terminal set), :223-226 (collision), :296-321 (ey, rate, box)
//   cost       mpc.py:356-373
// Method (DESIGN.md "solver"): single shooting on u with the previous input appended to the
// state (zeta = [z; u_prev]) so that the rate rows become stage-local; per iteration
//   sweep 1  forward sensitivities of every stage (6 seeds through the RK stages)
//   sweep 2  adjoint recursion -> KKT residuals -> barrier parameter update
//   sweep 3  Riccati recursion on the perturbed KKT system (slack y, multiplier s per row)
//   sweep 4+ closed-loop nonlinear forward passes with fraction-to-boundary and a
//            (barrier cost, infeasibility) acceptance test.
// All per-problem state lives in a struct-of-arrays workspace in HBM (element e of problem p
// at base[e * stride + p]) so that the 32 problems of a warp read and write 32 consecutive
// words; the small matrices of one stage live in registers.
//
// Everything here is __host__ __device__ so that tests can run the very same code on the CPU
// (tests/hostsim) -- the product only ever launches it from kernels.cu.
#pragma once
#include <cmath>
#include <cstdint>
#include <type_traits>
#include "mlp_tc.cuh"
#include "obca.cuh"

#ifdef __CUDACC__
#define IGT_HD __host__ __device__ __forceinline__
#define IGT_HDN __host__ __device__ __noinline__
#else
#define IGT_HD inline
#define IGT_HDN
#endif

#ifndef IGT_PF_DIST
#define IGT_PF_DIST 1          // stages ahead the latency-bound sweeps (adjoint, step bound) prefetch
#endif
#ifndef IGT_PF_DIST_R
#define IGT_PF_DIST_R 1        // ... and the Riccati sweep (compute-bound: one stage ahead is enough)
#endif

namespace igt {

constexpr int NZ = 7, NA = 9, NW = 11, NSEED = 6;
constexpr int NSENS = 26;   // structural non-zeros of a stage's sensitivities, see rk4_core
enum { IX = 0, IY, IS, IEY, IEPSI, IV, IPSI, IPA, IPD, IUA, IUD };
constexpr int MAX_CINF = 128;
// Node-local summaries of the inequality rows.  The rows of a node touch 8 entries of the gradient in
// w = (zeta, u) and, together with the dynamics second-order term, 22 entries of the symmetric
// w-space Hessian; these are what the sequential sweeps need from a node.
constexpr int NGE = 8, NHE = 22;
// OBCA collision mode (obca.cuh): the row's gradient has a heading entry as well -> one more gradient entry (psi) and
// two more Hessian entries ((x, psi), (y, psi)); they are appended, so the circle mode's tables are a prefix.
constexpr int NGE_OBCA = 9, NHE_OBCA = 24;
// Iterate buffers per workspace slot: the current iterate plus one buffer per step halving of a line
// search, so that all candidates alpha, alpha/2, ... of an iteration can be rolled out at once when
// lanes are idle (speculative line search, see trial_phase_cta).  Candidate j of an iterate living in
// buffer `cur` goes to the j-th buffer other than `cur`, so that the usual case (first candidate
// accepted) keeps toggling between buffers 0 and 1 and the speculative buffers stay cold.
constexpr int MAX_ALPHA = 6, NBUF = MAX_ALPHA + 1;
constexpr int NTC = 8;     // per-candidate scalars: finite flag, cost, terminal value term and its 5 derivatives
IGT_HD constexpr int cand_buf(int cur, int j) { return j < cur ? j : j + 1; }
constexpr int MAX_MLP_LAYERS = 5;
constexpr int MAX_MLP_NETS = 8;   // value networks of one handle's bank (IGT_MAX_MLP_NETS)
constexpr int N_GUESS = 5;

// One value network: the network fields of DevParams, same names (the value-term code is written against either).
// A handle's bank is a table of MAX_MLP_NETS of these in global memory; n_layers == 0 marks an empty slot.
template <typename T>
struct MlpNet {
    int n_layers;
    int dims[MAX_MLP_LAYERS + 1];
    T Wn[36], mu_f[6], sigma_t, mu_t;
    const T *W[MAX_MLP_LAYERS], *b[MAX_MLP_LAYERS];
    const T *Wt[MAX_MLP_LAYERS];
};

template <typename T>
struct DevParams {
    int N, n_rk, n_cinf, max_iter, n_alpha, second_order, n_layers, stall_iter, max_trials;
    int dims[MAX_MLP_LAYERS + 1];
    T dt, h, l_r, lsum, inv_lr, rho;
    T v_min, v_max, a_min, a_max, df_max, ey_lim, da_max, ddf_max, d_min, w_u;
    T tol, tol_rp, tol_comp, mu0, mu_floor, kappa_eps, kappa_mu, theta_mu, y_init_min, tau_min, mu0_warm, y_init_min_warm, alpha_safety, stall_rp;
    T reg_min, reg_up, reg_down, reg_max, reg_jump, eps_phi, gamma_theta, theta_small;
    T acc_tol, acc_rp, acc_comp, x0_tol;
    T cinf_A[MAX_CINF][2], cinf_b[MAX_CINF];
    T Wn[36], mu_f[6], sigma_t, mu_t;
    const T *W[MAX_MLP_LAYERS], *b[MAX_MLP_LAYERS];   // device pointers, row-major [out][in]
    const T *Wt[MAX_MLP_LAYERS];                      // the same weights transposed, [in][out] (mlp_coop.cuh)
};

}  // namespace igt
#include "mlp_coop.cuh"
namespace igt {

// ------------------------------------------------------------------ workspace ----------
// Row bookkeeping: stage 0 carries the 8 input rows; stage k >= 1 carries 5 state rows
// (v hi/lo, ey hi/lo, collision) + 8 input rows (a hi/lo, df hi/lo, rate a +-, rate df +-);
// stage N-1 additionally the n_cinf terminal-set rows; the terminal node 3 rows.
IGT_HD int row_off(int N, int n_cinf, int k)
{
    if (k == 0) return 0;
    int o = 8 + 13 * (k - 1);
    if (k == N) o += n_cinf;
    return o;
}
IGT_HD int row_total(int N, int n_cinf) { return row_off(N, n_cinf, N) + 3; }

struct WsLayout {
    int N, M;
    // the NBUF iterate buffers of an array lie back to back: offset of buffer b = base + b * size (no table lookup with a
    // run-time index, which would put the layout into local memory)
    int oZ0, oU0, oY0, oS0, oTc, oSens, oLam, oKu, oKK, oGw, oRed, oGl, oHl, oTr, oDu, total;
    IGT_HD int oZ(int b) const { return oZ0 + b * (NZ * (N + 1)); }
    IGT_HD int oU(int b) const { return oU0 + b * (2 * N); }
    IGT_HD int oY(int b) const { return oY0 + b * M; }
    IGT_HD int oS(int b) const { return oS0 + b * M; }
    IGT_HD void init(int N_, int n_cinf, int nge = NGE, int nhe = NHE)
    {
        N = N_;
        M = row_total(N, n_cinf);
        int o = 0;
        oZ0 = o; o += NBUF * NZ * (N + 1);
        oU0 = o; o += NBUF * 2 * N;
        oY0 = o; o += NBUF * M;
        oS0 = o; o += NBUF * M;
        oSens = o; o += NSENS * N;
        oLam = o;  o += NZ * (N + 1);
        oKu = o;   o += 2 * N;
        oKK = o;   o += 2 * NA * N;
        oGw = o;   o += nge * (N + 1);     // node-local row summaries, see node_phase1 / node_phase2
        oRed = o;  o += 4 * (N + 1);
        oGl = o;   o += nge * (N + 1);
        oHl = o;   o += nhe * (N + 1);
        oTr = o;   o += NBUF * 3 * (N + 1);  // per-node results of a trial step, see node_phase3
        oDu = o;   o += NBUF * 2 * N;        // control change of a trial step (exact, not new - old)
        oTc = o;   o += NBUF * NTC;          // per-candidate rollout results: finite flag, cost, value term (6)
        total = o;
    }
};

// Workspace addressing: slots are grouped by warp; element e of slot q lives at
//   base[(q / 32) * total * 32 + e * 32 + (q % 32)]
// so the 32 lanes of a warp touch 32 consecutive words for every element, and every element
// offset that is a compile-time constant folds into the load/store immediate.
// STRIDE 1 is the latency path for batches of at most one problem per SM: the workspace of the CTA's one
// problem lives in shared memory, contiguously (bind ignores the slot, nothing is prefetched).
// RSTG (row staging, node phases of the throughput kernel): the slacks and multipliers of a node's (at most 13) stage
// rows are copied into this thread's private column of a shared-memory buffer with per-thread cp.async at the start of
// the item -- no registers in flight, unlike a burst of loads -- and read from there when the rows are visited, instead
// of one dependent L2 / HBM round trip per row (a quarter of the kernel's stall samples in round 1's ncu source view).
constexpr int RSTG_SLOTS = 26;           // 13 rows x (multiplier, slack)
template <typename T, int STRIDE = 32, bool OBCA = false, bool RSTG = false>
struct Ws {
    static constexpr bool obca = OBCA;
    static constexpr bool rstg = RSTG;
    static constexpr int stride = STRIDE;
    T *rs = nullptr;                     // RSTG: this thread's column, slot i at rs[i * blockDim.x]
    int rs_stride = 0;
    IGT_HD void rows_fetch(int b, int o, int n) const
    {
#ifdef __CUDA_ARCH__
        if (RSTG) {
            for (int r = 0; r < n; r++) {
                const unsigned ds = (unsigned)__cvta_generic_to_shared(rs + (2 * r) * rs_stride);
                const unsigned dy = (unsigned)__cvta_generic_to_shared(rs + (2 * r + 1) * rs_stride);
                if (sizeof(T) == 8) {
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(ds), "l"(wb + (L.oS(b) + o + r) * STRIDE) : "memory");
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dy), "l"(wb + (L.oY(b) + o + r) * STRIDE) : "memory");
                } else {
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(ds), "l"(wb + (L.oS(b) + o + r) * STRIDE) : "memory");
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dy), "l"(wb + (L.oY(b) + o + r) * STRIDE) : "memory");
                }
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        }
#endif
    }
    IGT_HD void rows_wait() const
    {
#ifdef __CUDA_ARCH__
        if (RSTG) asm volatile("cp.async.wait_group 0;" ::: "memory");
#endif
    }
    IGT_HD T row_s(int b, int o, int r) const { return RSTG ? rs[(2 * r) * rs_stride] : at(L.oS(b) + o + r); }
    IGT_HD T row_y(int b, int o, int r) const { return RSTG ? rs[(2 * r + 1) * rs_stride] : at(L.oY(b) + o + r); }
    static constexpr int nge = OBCA ? NGE_OBCA : NGE, nhe = OBCA ? NHE_OBCA : NHE;
    T *wb;          // base + (slot / 32) * total * 32 + slot % 32
    WsLayout L;
    IGT_HD void init_layout(int N, int n_cinf) { L.init(N, n_cinf, nge, nhe); }
    IGT_HD void bind(T *base, long slot) { wb = STRIDE == 32 ? base + (slot / 32) * (long)L.total * 32 + (slot % 32) : base; }
    IGT_HD T &at(int e) const { return wb[e * STRIDE]; }
    IGT_HD void pf(int e) const
    {
#ifdef __CUDA_ARCH__
        if (STRIDE == 32) asm volatile("prefetch.global.L1 [%0];" ::"l"(wb + e * 32));
#endif
    }
    // NN consecutive elements from e0: one address computation, then immediate offsets (a prefetch with its own index
    // costs five integer instructions on top of the prefetch itself)
    template <int I, int NN>
    IGT_HD void pf_run_(const T *base) const
    {
#ifdef __CUDA_ARCH__
        if constexpr (I < NN) {
            asm volatile("prefetch.global.L1 [%0+%1];" ::"l"(base), "n"(I * 32 * (int)sizeof(T)));
            pf_run_<I + 1, NN>(base);
        }
#endif
    }
    template <int NN>
    IGT_HD void pf_run(int e0) const { if (STRIDE == 32) pf_run_<0, NN>(wb + e0 * 32); }
    // pointer to element e0; element e0 + i is p[i * STRIDE] -- with a compile-time i the offset folds into the load /
    // store instruction (used in the node phases and in the rollout, functions with registers to spare: every workspace
    // access there used to carry five integer instructions of address arithmetic)
    IGT_HD T *ptr(int e0) const { return wb + (long)e0 * STRIDE; }
    IGT_HD T &Z(int b, int k, int i) const { return at(L.oZ(b) + k * NZ + i); }
    IGT_HD T &U(int b, int k, int i) const { return at(L.oU(b) + k * 2 + i); }
    IGT_HD T &Y(int b, int r) const { return at(L.oY(b) + r); }
    IGT_HD T &S(int b, int r) const { return at(L.oS(b) + r); }
    IGT_HD T &Sens(int k, int e) const { return at(L.oSens + k * NSENS + e); }
    IGT_HD T &Lam(int k, int i) const { return at(L.oLam + k * NZ + i); }
    IGT_HD T &ku(int k, int i) const { return at(L.oKu + k * 2 + i); }
    IGT_HD T &KK(int k, int i, int j) const { return at(L.oKK + (k * 2 + i) * NA + j); }
    IGT_HD T &Gw(int k, int e) const { return at(L.oGw + k * nge + e); }
    IGT_HD T &Red(int k, int e) const { return at(L.oRed + k * 4 + e); }
    IGT_HD T &Gl(int k, int e) const { return at(L.oGl + k * nge + e); }
    IGT_HD T &Hl(int k, int e) const { return at(L.oHl + k * nhe + e); }
    IGT_HD T &Tr(int b, int k, int e) const { return at(L.oTr + (b * (L.N + 1) + k) * 3 + e); }
    IGT_HD T &Du(int b, int k, int i) const { return at(L.oDu + (b * L.N + k) * 2 + i); }
    IGT_HD T &Tc(int b, int e) const { return at(L.oTc + b * NTC + e); }
};

// problem inputs / outputs: batch-major AoS arrays exactly as the C ABI receives them
struct ProbIO {
    const double *x0, *u_prev, *curv, *obs, *ctx, *u_init;   // [B,7] [B,2] [B,3] [B,N+1,2] [B,4] [B,N,2]
    double *x, *u, *cost, *viol;
    int *status, *iters;
    const double *obs_psi = nullptr;                         // [B,N+1] obstacle heading forecast: OBCA collision rows
    const int *warm = nullptr;                               // [B] per-problem warm-start flags (with u_init); null: all warm
};
// inputs of a bank solve (the BANK kernels): a type of its own, so that the other kernels' parameters stay as they are
template <typename T>
struct ProbIONet : ProbIO {
    const int *net_idx = nullptr;                            // [B] value network of each problem in nets
    const MlpNet<T> *nets = nullptr;                         // the handle's bank: [MAX_MLP_NETS] descriptors
    // a bank index that may be dereferenced: 0..MAX_MLP_NETS-1 and a loaded slot
    IGT_HD bool net_ok(int k) const { return (unsigned)k < (unsigned)MAX_MLP_NETS && nets[k].n_layers > 0; }
};
// (only for an io that is a ProbIONet<T>: the BANK code paths)
template <typename T>
IGT_HD const ProbIONet<T> &bank_io(const ProbIO &io) { return static_cast<const ProbIONet<T> &>(io); }

// ------------------------------------------------------------------ dynamics -----------
IGT_HD void sincos_t(float x, float *s, float *c) { sincosf(x, s, c); }
IGT_HD void sincos_t(double x, double *s, double *c) { sincos(x, s, c); }

template <typename T>
struct Slip { T beta, dbeta, sb, cb; };

template <typename T>
IGT_HD Slip<T> slip_of(const DevParams<T> &P, T df)
{   // kinematic_bicycle_model.py:26 (Cartesian Euler model only; the Frenet model uses step_setup)
    Slip<T> r;
    T t = tan(df);
    r.beta = atan(P.rho * t);
    r.dbeta = P.rho * (T(1) + t * t) / (T(1) + P.rho * P.rho * t * t);
    sincos_t(r.beta, &r.sb, &r.cb);
    return r;
}

template <typename T>
IGT_HD T curvature(T s, T b0, T b1, T kv)
{   // casadi pw_const, mpc.py:199: K = kv*(s>=b0) - kv*(s>=b1), zero derivative
    return (s >= b0 ? kv : T(0)) - (s >= b1 ? kv : T(0));
}

// sin(d), cos(d) of the two small within-step drifts d1 = epsi - epsi_0 and d2 = psi - psi_0.
// One MPC step evaluates the right-hand side 16 times at angles that differ from the step's start
// by < 0.15 rad (yaw rate <= 1.4 rad/s), so two full-range sincos per step plus 16 short polynomial
// pairs replace 32 full-range fp64 sincos calls.  Both drifts are evaluated in ONE straight-line
// block (four independent Horner chains: the fp64 pipe issues one DFMA per ~2.2 cycles per warp but
// a dependent DFMA waits ~9), Taylor to d^13 / d^14 with truncation error < 1e-21 for |d| <= 0.25;
// beyond that (never seen in practice) the library is called.
IGT_HD void sincos_small2(double d1, double d2, double &s1, double &c1, double &s2, double &c2)
{
    const double S1 = -1.0 / 6, S2 = 1.0 / 120, S3 = -1.0 / 5040, S4 = 1.0 / 362880, S5 = -1.0 / 39916800,
                 S6 = 1.0 / 6227020800.0;
    const double C1 = -0.5, C2 = 1.0 / 24, C3 = -1.0 / 720, C4 = 1.0 / 40320, C5 = -1.0 / 3628800,
                 C6 = 1.0 / 479001600.0, C7 = -1.0 / 87178291200.0;
    const double x1 = d1 * d1, x2 = d2 * d2;
    double ps1 = S5 + x1 * S6, ps2 = S5 + x2 * S6, pc1 = C6 + x1 * C7, pc2 = C6 + x2 * C7;
    ps1 = S4 + x1 * ps1; ps2 = S4 + x2 * ps2; pc1 = C5 + x1 * pc1; pc2 = C5 + x2 * pc2;
    ps1 = S3 + x1 * ps1; ps2 = S3 + x2 * ps2; pc1 = C4 + x1 * pc1; pc2 = C4 + x2 * pc2;
    ps1 = S2 + x1 * ps1; ps2 = S2 + x2 * ps2; pc1 = C3 + x1 * pc1; pc2 = C3 + x2 * pc2;
    ps1 = S1 + x1 * ps1; ps2 = S1 + x2 * ps2; pc1 = C2 + x1 * pc1; pc2 = C2 + x2 * pc2;
    pc1 = C1 + x1 * pc1; pc2 = C1 + x2 * pc2;
    const double t1 = d1 * x1, t2 = d2 * x2;
    s1 = d1 + t1 * ps1; s2 = d2 + t2 * ps2;
    c1 = 1.0 + x1 * pc1; c2 = 1.0 + x2 * pc2;
    if (fmax(fabs(d1), fabs(d2)) > 0.25) { sincos(d1, &s1, &c1); sincos(d2, &s2, &c2); }
}
IGT_HD void sincos_small2(float d1, float d2, float &s1, float &c1, float &s2, float &c2)
{   // fp32: terms to d^7 / d^8 (truncation < 2e-11 for |d| <= 0.25)
    const float S1 = -1.f / 6, S2 = 1.f / 120, S3 = -1.f / 5040, C1 = -0.5f, C2 = 1.f / 24, C3 = -1.f / 720, C4 = 1.f / 40320;
    const float x1 = d1 * d1, x2 = d2 * d2;
    float ps1 = S2 + x1 * S3, ps2 = S2 + x2 * S3, pc1 = C3 + x1 * C4, pc2 = C3 + x2 * C4;
    ps1 = S1 + x1 * ps1; ps2 = S1 + x2 * ps2; pc1 = C2 + x1 * pc1; pc2 = C2 + x2 * pc2;
    pc1 = C1 + x1 * pc1; pc2 = C1 + x2 * pc2;
    s1 = d1 + d1 * x1 * ps1; s2 = d2 + d2 * x2 * ps2;
    c1 = 1.f + x1 * pc1; c2 = 1.f + x2 * pc2;
    if (fmaxf(fabsf(d1), fabsf(d2)) > 0.25f) { sincosf(d1, &s1, &c1); sincosf(d2, &s2, &c2); }
}

// Constants of one MPC step of the Frenet model (kinematic_bicycle_model_frenet.py:72): the slip angle
// beta = atan(rho tan(df)) enters only through sin / cos, which follow from tan(df) algebraically, and
// through beta + epsi, psi + beta, whose sin / cos at the step's start come from the angle-addition rule.
template <typename T>
struct StepK {
    T h, a, yawc, pdc, dbeta, sb, cb, tdf;   // yawc = sin(beta)/l_r, pdc = cos(beta)/l_r * dbeta/ddf
    T e0, p0, s1b, c1b, spb, cpb;            // sin / cos of (beta + epsi_0) and (psi_0 + beta)
    T b0, b1, kv;
};

template <typename T>
IGT_HD StepK<T> step_setup(const DevParams<T> &P, const T *z0, const T *u, const T *curv)
{
    StepK<T> c;
    c.h = P.h; c.a = u[0];
    const T t = tan(u[1]), r = P.rho * t;
    const T iq = T(1) / (T(1) + r * r);
    c.tdf = t;
    c.cb = sqrt(iq); c.sb = r * c.cb;
    c.dbeta = P.rho * (T(1) + t * t) * iq;
    c.yawc = c.sb * P.inv_lr;
    c.pdc = c.cb * P.inv_lr * c.dbeta;
    c.e0 = z0[IEPSI]; c.p0 = z0[IPSI];
    T se, ce, sp, cp;
    sincos_t(c.e0, &se, &ce);
    sincos_t(c.p0, &sp, &cp);
    c.s1b = se * c.cb + ce * c.sb; c.c1b = ce * c.cb - se * c.sb;
    c.spb = sp * c.cb + cp * c.sb; c.cpb = cp * c.cb - sp * c.sb;
    c.b0 = curv[0]; c.b1 = curv[1]; c.kv = curv[2];
    return c;
}

// time derivative of (s, ey, epsi, x, y, psi) (v' = a) and, if JAC, its 13 state + 6 steering partials
template <typename T>
struct Deriv { T s, ey, ep, x, y, ps; };
template <typename T>
struct RhsJac { T s_ey, s_ep, s_v, s_d, ey_ep, ey_v, ey_d, e_ey, e_ep, e_v, e_d, x_v, x_ps, x_d, y_v, y_ps, y_d, p_v, p_d; };

// KF: the curvature of this evaluation is given (Kf) instead of looked up from s -- the fp32 rollout kernel decides the
// pw_const branch in double from its compensated arc length, see rollout_kernel
template <typename T, bool JAC, bool KF = false>
IGT_HD void stage_deriv(const StepK<T> &c, T s, T ey, T ep, T v, T ps, Deriv<T> &d, RhsJac<T> &J, T Kf = T(0))
{   // kinematic_bicycle_model_frenet.py:71-91
    T s1, c1, sp, cp;
    {
        T sd1, cd1, sd2, cd2;
        sincos_small2(ep - c.e0, ps - c.p0, sd1, cd1, sd2, cd2);
        s1 = c.s1b * cd1 + c.c1b * sd1; c1 = c.c1b * cd1 - c.s1b * sd1;
        sp = c.spb * cd2 + c.cpb * sd2; cp = c.cpb * cd2 - c.spb * sd2;
    }
    T K = T(0), iden = T(1);
    if (c.kv != T(0)) {                                        // straight routes: no curvature test, no division
        K = KF ? Kf : curvature(s, c.b0, c.b1, c.kv);
        if (K != T(0)) iden = T(1) / (T(1) - K * ey);
    }
    const T sdot = v * c1 * iden;
    const T yaw = v * c.yawc;
    d.s = sdot;
    d.ey = v * s1;
    d.ep = yaw - sdot * K;
    d.x = v * cp;
    d.y = v * sp;
    d.ps = yaw;
    if (JAC) {
        const T db = c.dbeta;
        J.s_ey = sdot * K * iden;
        J.s_ep = -v * s1 * iden;
        J.s_v = c1 * iden;
        J.s_d = J.s_ep * db;
        J.ey_ep = v * c1; J.ey_v = s1; J.ey_d = J.ey_ep * db;
        J.e_ey = -K * J.s_ey; J.e_ep = -K * J.s_ep;
        J.e_v = c.yawc - K * J.s_v;
        J.e_d = v * c.pdc - K * J.s_d;
        J.x_v = cp; J.x_ps = -d.y; J.x_d = J.x_ps * db;
        J.y_v = sp; J.y_ps = d.x; J.y_d = J.y_ps * db;
        J.p_v = c.yawc; J.p_d = v * c.pdc;
    }
}

// Sensitivities of one MPC step, structural non-zeros only (26 of the 7 x 6 entries of
// d z+ / d (ey, epsi, v, psi, a, df); d z+/d(x, y, s) = unit vectors since dK/ds == 0):
//   rows x, y        w.r.t. (v, psi, a, df)        -- x, y follow v and psi only
//   rows s, ey, epsi w.r.t. (ey, epsi, v, a, df)   -- psi feeds nothing but x, y
//   row  psi         w.r.t. (v, a, df); d psi+/d psi = 1;  row v: d v+/d v = 1, d v+/d a = dt.
enum { SX = 0, SY = 4, SS = 8, SEY = 13, SEP = 18, SPS = 23 };

// One MPC step: n_rk RK4 sub-steps.  k4 evaluates xdot, ydot at psi + h/2*k3[psi]
// (kinematic_bicycle_model_frenet.py:111) -- reproduced on purpose.  SENS adds the forward
// sensitivities; the state arithmetic is the same expression for expression, so both variants
// return bit-identical states (the solver relies on it: a trial point rolled out with or without
// sensitivities is the same point).
template <typename T, bool SENS>
IGT_HD void rk4_core(const DevParams<T> &P, const T *z0, const T *u_in, const T *curv_in, T *zn, T *Sc)
{
    const StepK<T> c = step_setup(P, z0, u_in, curv_in);
    const T h = c.h, hh = h * T(0.5), h6 = h / T(6), a = c.a;
    const int n_rk = P.n_rk;
    T x = z0[IX], y = z0[IY], s = z0[IS], ey = z0[IEY], ep = z0[IEPSI], v = z0[IV], ps = z0[IPSI];
    // sensitivities of the rows that feed back (ey, epsi, psi): value at the sub-step's start;
    // of the rows that do not (x, y, s): running sum of the weighted stage tangents over all sub-steps
    T Sey[5], Sep[5], Sps[3], Ax[4], Ay[4], As[5];
    if (SENS) {
#pragma unroll
        for (int j = 0; j < 5; j++) { Sey[j] = T(0); Sep[j] = T(0); As[j] = T(0); }
#pragma unroll
        for (int j = 0; j < 4; j++) { Ax[j] = T(0); Ay[j] = T(0); }
        Sps[0] = Sps[1] = Sps[2] = T(0);
        Sey[0] = T(1); Sep[1] = T(1);
    }
#pragma unroll 1
    for (int it = 0; it < n_rk; it++) {
        T ss = s, sey = ey, sep = ep, sv = v, sps = ps;           // stage state
        T ks = T(0), key = T(0), kep = T(0), kx = T(0), ky = T(0), kps = T(0);
        T Tey[5], Tep[5], Tps[3], Dey[5], Dep[5], Dps[3];        // stage tangents, weighted sums of this sub-step
        const T tva0 = T(it) * h;                                 // d v / d a at the sub-step's start
        if (SENS) {
#pragma unroll
            for (int j = 0; j < 5; j++) { Tey[j] = Sey[j]; Tep[j] = Sep[j]; Dey[j] = T(0); Dep[j] = T(0); }
#pragma unroll
            for (int j = 0; j < 3; j++) { Tps[j] = Sps[j]; Dps[j] = T(0); }
        }
#pragma unroll
        for (int st = 0; st < 4; st++) {
            const T wgt = (st == 0 || st == 3) ? T(1) : T(2);
            const T cf = (st == 2) ? h : hh;                      // step to the next stage's state; psi always moves by
                                                                  // h/2, after k3 as well (the k4 quirk)
            Deriv<T> d;
            RhsJac<T> J;
            stage_deriv<T, SENS>(c, ss, sey, sep, sv, sps, d, J);
            ks += wgt * d.s; key += wgt * d.ey; kep += wgt * d.ep; kx += wgt * d.x; ky += wgt * d.y; kps += wgt * d.ps;
            if (SENS) {
                const T tva = st == 0 ? tva0 : (st == 3 ? tva0 + h : tva0 + hh);   // d v_stage / d a
                T ds[5], dey[5], dep[5];
#pragma unroll
                for (int j = 0; j < 5; j++) {
                    ds[j] = J.s_ey * Tey[j] + J.s_ep * Tep[j];
                    dey[j] = J.ey_ep * Tep[j];
                    dep[j] = J.e_ey * Tey[j] + J.e_ep * Tep[j];
                }
                ds[2] += J.s_v; dey[2] += J.ey_v; dep[2] += J.e_v;
                ds[3] += J.s_v * tva; dey[3] += J.ey_v * tva; dep[3] += J.e_v * tva;
                ds[4] += J.s_d; dey[4] += J.ey_d; dep[4] += J.e_d;
                const T dx[4] = { J.x_v + J.x_ps * Tps[0], J.x_ps, J.x_v * tva + J.x_ps * Tps[1], J.x_ps * Tps[2] + J.x_d };
                const T dy[4] = { J.y_v + J.y_ps * Tps[0], J.y_ps, J.y_v * tva + J.y_ps * Tps[1], J.y_ps * Tps[2] + J.y_d };
                const T dps[3] = { J.p_v, J.p_v * tva, J.p_d };
#pragma unroll
                for (int j = 0; j < 5; j++) {
                    As[j] += wgt * ds[j]; Dey[j] += wgt * dey[j]; Dep[j] += wgt * dep[j];
                    if (st < 3) { Tey[j] = Sey[j] + cf * dey[j]; Tep[j] = Sep[j] + cf * dep[j]; }
                }
#pragma unroll
                for (int j = 0; j < 4; j++) { Ax[j] += wgt * dx[j]; Ay[j] += wgt * dy[j]; }
#pragma unroll
                for (int j = 0; j < 3; j++) {
                    Dps[j] += wgt * dps[j];
                    if (st < 3) Tps[j] = Sps[j] + hh * dps[j];
                }
            }
            if (st < 3) {
                ss = s + cf * d.s; sey = ey + cf * d.ey; sep = ep + cf * d.ep; sv = v + cf * a;
                sps = ps + hh * d.ps;
            }
        }
        x += h6 * kx; y += h6 * ky; s += h6 * ks; ey += h6 * key; ep += h6 * kep; ps += h6 * kps;
        v += h6 * (a + T(2) * a + T(2) * a + a);
        if (SENS) {
#pragma unroll
            for (int j = 0; j < 5; j++) { Sey[j] += h6 * Dey[j]; Sep[j] += h6 * Dep[j]; }
#pragma unroll
            for (int j = 0; j < 3; j++) Sps[j] += h6 * Dps[j];
        }
    }
    zn[IX] = x; zn[IY] = y; zn[IS] = s; zn[IEY] = ey; zn[IEPSI] = ep; zn[IV] = v; zn[IPSI] = ps;
    if (SENS) {
#pragma unroll
        for (int j = 0; j < 4; j++) { Sc[SX + j] = h6 * Ax[j]; Sc[SY + j] = h6 * Ay[j]; }
#pragma unroll
        for (int j = 0; j < 5; j++) { Sc[SS + j] = h6 * As[j]; Sc[SEY + j] = Sey[j]; Sc[SEP + j] = Sep[j]; }
#pragma unroll
        for (int j = 0; j < 3; j++) Sc[SPS + j] = Sps[j];
    }
}

template <typename T>
IGT_HDN void rk4_step(const DevParams<T> &P, const T *z0, const T *u_in, const T *curv_in, T *zn)
{
    rk4_core<T, false>(P, z0, u_in, curv_in, zn, nullptr);
}

// one MPC step with its compact sensitivities Sc[NSENS]
template <typename T>
IGT_HDN void rk4_step_sens(const DevParams<T> &P, const T *z0, const T *u_in, const T *curv_in, T *zn, T *Sc)
{
    rk4_core<T, true>(P, z0, u_in, curv_in, zn, Sc);
}

// dense d z+ / d (ey, epsi, v, psi, a, df) [7][6] from the compact form (ABI output, tests)
template <typename T>
IGT_HD void expand_sens(const DevParams<T> &P, const T *Sc, T (*S)[NSEED])
{
#pragma unroll
    for (int i = 0; i < NZ; i++)
#pragma unroll
        for (int j = 0; j < NSEED; j++) S[i][j] = T(0);
    const int c4[4] = { 2, 3, 4, 5 }, c5[5] = { 0, 1, 2, 4, 5 }, c3[3] = { 2, 4, 5 };
    for (int j = 0; j < 4; j++) { S[IX][c4[j]] = Sc[SX + j]; S[IY][c4[j]] = Sc[SY + j]; }
    for (int j = 0; j < 5; j++) { S[IS][c5[j]] = Sc[SS + j]; S[IEY][c5[j]] = Sc[SEY + j]; S[IEPSI][c5[j]] = Sc[SEP + j]; }
    for (int j = 0; j < 3; j++) S[IPSI][c3[j]] = Sc[SPS + j];
    S[IPSI][3] = T(1); S[IV][2] = T(1); S[IV][4] = P.dt;
}

// Cartesian Euler model, z = (x, y, psi, v): kinematic_bicycle_model.py:27-31
template <typename T>
IGT_HD void euler_step(const DevParams<T> &P, const T *z, const T *u, T *zn, T *A, T *B)
{
    T x = z[0], y = z[1], psi = z[2], v = z[3], dt = P.dt;
    Slip<T> sl = slip_of(P, u[1]);
    T lsum = P.lsum, t = tan(u[1]);
    T cp = cos(psi + sl.beta), sp = sin(psi + sl.beta);
    zn[0] = x + dt * v * cp;
    zn[1] = y + dt * v * sp;
    zn[2] = psi + dt * (v * sl.cb / lsum * t);
    zn[3] = v + dt * u[0];
    if (A) {
        for (int i = 0; i < 16; i++) A[i] = T(0);
        for (int i = 0; i < 8; i++) B[i] = T(0);
        A[0] = A[5] = A[10] = A[15] = T(1);
        A[2] = -dt * v * sp; A[3] = dt * cp;
        A[6] = dt * v * cp;  A[7] = dt * sp;
        A[11] = dt * sl.cb / lsum * t;
        B[1] = -dt * v * sp * sl.dbeta;
        B[3] = dt * v * cp * sl.dbeta;
        B[5] = dt * v / lsum * (-sl.sb * sl.dbeta * t + sl.cb * (T(1) + t * t));
        B[6] = dt;
    }
}

// ------------------------------------------------------------------ value term ---------
template <typename T>
struct TermVal { T V, gs, gv, Hss, Hsv, Hvv; };

// gt_mpc terminal value (mpc.py:326-354, :367-369; model.py:14-67) on CUDA cores, one
// problem per thread: value + first and second forward tangents in (s_N, v_N).
// Scratch: two [6][width] slabs of the caller's workspace.  NP: DevParams<T> (the handle's network, mlp_eval_thread) or
// MlpNet<T> (a bank entry, mlp_eval_thread_net).
template <typename T, typename NP>
IGT_HD void mlp_eval_body(const NP &P, T sN, T vN, const T *ctx, T *ha, T *hb, int width, TermVal<T> &out, bool want_deriv)
{
    T xN[6] = { ctx[0], ctx[1], ctx[2], sN - ctx[0], vN - ctx[1], ctx[3] - ctx[2] };
    const int R = want_deriv ? 6 : 1;
    for (int i = 0; i < 6; i++) {
        T acc = T(0);
        for (int j = 0; j < 6; j++) acc += P.Wn[i * 6 + j] * (xN[j] - P.mu_f[j]);
        ha[0 * width + i] = acc;
        if (want_deriv) {
            ha[1 * width + i] = P.Wn[i * 6 + 3];
            ha[2 * width + i] = P.Wn[i * 6 + 4];
            ha[3 * width + i] = ha[4 * width + i] = ha[5 * width + i] = T(0);
        }
    }
    for (int l = 0; l < P.n_layers; l++) {
        int nin = P.dims[l], nout = P.dims[l + 1];
        const T *W = P.W[l], *b = P.b[l];
        for (int o = 0; o < nout; o++) {
            T acc[6] = { b[o], T(0), T(0), T(0), T(0), T(0) };
            for (int i = 0; i < nin; i++) {
                T w = W[(long)o * nin + i];
                for (int r = 0; r < R; r++) acc[r] += w * ha[r * width + i];
            }
            if (l < P.n_layers - 1) {
                T y = tanh(acc[0]), d1 = T(1) - y * y, d2 = T(-2) * y * d1;
                hb[0 * width + o] = y;
                if (want_deriv) {
                    T ts = acc[1], tv = acc[2];
                    hb[1 * width + o] = d1 * ts;
                    hb[2 * width + o] = d1 * tv;
                    hb[3 * width + o] = d1 * acc[3] + d2 * ts * ts;
                    hb[4 * width + o] = d1 * acc[4] + d2 * ts * tv;
                    hb[5 * width + o] = d1 * acc[5] + d2 * tv * tv;
                }
            } else {
                for (int r = 0; r < R; r++) hb[r * width + o] = acc[r];
            }
        }
        T *t = ha; ha = hb; hb = t;
    }
    out.V = ha[0] * P.sigma_t + P.mu_t;
    if (want_deriv) {
        out.gs = ha[1 * width] * P.sigma_t; out.gv = ha[2 * width] * P.sigma_t;
        out.Hss = ha[3 * width] * P.sigma_t; out.Hsv = ha[4 * width] * P.sigma_t; out.Hvv = ha[5 * width] * P.sigma_t;
    } else {
        out.gs = out.gv = out.Hss = out.Hsv = out.Hvv = T(0);
    }
}
template <typename T>
IGT_HDN void mlp_eval_thread(const DevParams<T> &P, T sN, T vN, const T *ctx, T *ha, T *hb, int width,
                             TermVal<T> &out, bool want_deriv)
{
    mlp_eval_body(P, sN, vN, ctx, ha, hb, width, out, want_deriv);
}
template <typename T>
IGT_HDN void mlp_eval_thread_net(const MlpNet<T> &P, T sN, T vN, const T *ctx, T *ha, T *hb, int width,
                                 TermVal<T> &out, bool want_deriv)
{
    mlp_eval_body(P, sN, vN, ctx, ha, hb, width, out, want_deriv);
}

// sum of log(y_i) with one log per LOGCHUNK factors (slacks lie in [1e-11, 1e3], so a product of
// 16 stays far inside the fp64 range; fp32 uses 3)
template <typename T> struct LogChunk { static constexpr int n = 16; };
template <> struct LogChunk<float> { static constexpr int n = 3; };
template <typename T>
struct LogSum {
    T sum, prod; int cnt;
    IGT_HD LogSum() : sum(T(0)), prod(T(1)), cnt(0) {}
    IGT_HD void add(T y) { prod *= y; if (++cnt == LogChunk<T>::n) { sum += log(prod); prod = T(1); cnt = 0; } }
    IGT_HD T total() const { return cnt ? sum + log(prod) : sum; }
};

// ------------------------------------------------------------------ rows ---------------
// visit every inequality row of stage k (k == N: terminal node) in workspace order.
// f(IC<slot>, r, c, IC<i0>, g0, IC<i1>, g1, IC<i2>, g2, hxx, hxy, hyy): value, up to three gradient entries in
// w = (zeta, u) (i1 / i2 < 0: unused; the third is the heading entry of the OBCA row), 2x2 Hessian block on (x, y)
// (circle collision row only).
// The indices travel as types so that every use indexes registers statically.  `slot` is the row's
// fixed register slot (0,1 speed; 2,3 ey; 4 collision; 5..12 input and rate rows), the same for every
// stage.  The terminal-set rows of stage N-1 (slot -1) are visited only if CINF; the node phases run
// them in their own loops (cinf_rows), node_phase3 both of its passes over them in one.
template <int I> struct IC { static constexpr int value = I; };
constexpr int NSLOT = 13;
IGT_HD int slot_base(int N, int k) { return k == 0 ? 5 : (k == N ? 2 : 0); }      // workspace row = slot - base
IGT_HD bool slot_used(int N, int k, int slot) { return k == 0 ? slot >= 5 : (k == N ? (slot >= 2 && slot <= 4) : true); }

template <bool CINF = true, bool OBCA = false, typename T, typename F>
IGT_HD void visit_rows(const DevParams<T> &P, int k, const T *z, const T *up, const T *u, T ox, T oy, T opsi, F &&f)
{
    const T Z0 = T(0);
    using NO = IC<-1>;
    int r = 0;
    if (k >= 1) {
        if (k < P.N) {
            f(IC<0>{}, r++, z[IV] - P.v_max, IC<IV>{}, T(1), NO{}, Z0, NO{}, Z0, Z0, Z0, Z0);      // mpc.py:317
            f(IC<1>{}, r++, P.v_min - z[IV], IC<IV>{}, T(-1), NO{}, Z0, NO{}, Z0, Z0, Z0, Z0);     // mpc.py:316
        }
        f(IC<2>{}, r++, z[IEY] - P.ey_lim, IC<IEY>{}, T(1), NO{}, Z0, NO{}, Z0, Z0, Z0, Z0);      // mpc.py:298
        f(IC<3>{}, r++, -P.ey_lim - z[IEY], IC<IEY>{}, T(-1), NO{}, Z0, NO{}, Z0, Z0, Z0, Z0);    // mpc.py:299
        if constexpr (!OBCA) {   // mpc.py:226 in the equivalent distance form d_min - |p - o| <= 0
            T dx = z[IX] - ox, dy = z[IY] - oy;
            T dist = sqrt(dx * dx + dy * dy);
            dist = dist < T(1e-9) ? T(1e-9) : dist;
            T id = T(1) / dist, nx = dx * id, ny = dy * id;
            f(IC<4>{}, r++, P.d_min - dist, IC<IX>{}, -nx, IC<IY>{}, -ny, NO{}, Z0, -(T(1) - nx * nx) * id, nx * ny * id, -(T(1) - ny * ny) * id);
        } else {                 // mpc.py:211-221 with the duals maximised out (obca.cuh): margin - signed rectangle distance
            T gd[3];
            const T sd = obca_rect_sdist(z[IX], z[IY], z[IPSI], ox, oy, opsi, gd);
            f(IC<4>{}, r++, P.d_min + T(OBCA_MARGIN) - sd, IC<IX>{}, -gd[0], IC<IY>{}, -gd[1], IC<IPSI>{}, -gd[2], Z0, Z0, Z0);
        }
    }
    if (k == P.N) return;
    f(IC<5>{}, r++, u[0] - P.a_max, IC<IUA>{}, T(1), NO{}, Z0, NO{}, Z0, Z0, Z0, Z0);             // mpc.py:319
    f(IC<6>{}, r++, P.a_min - u[0], IC<IUA>{}, T(-1), NO{}, Z0, NO{}, Z0, Z0, Z0, Z0);            // mpc.py:318
    f(IC<7>{}, r++, u[1] - P.df_max, IC<IUD>{}, T(1), NO{}, Z0, NO{}, Z0, Z0, Z0, Z0);            // mpc.py:321
    f(IC<8>{}, r++, -P.df_max - u[1], IC<IUD>{}, T(-1), NO{}, Z0, NO{}, Z0, Z0, Z0, Z0);          // mpc.py:320
    T da = u[0] - up[0], dd = u[1] - up[1];
    f(IC<9>{}, r++, da - P.da_max, IC<IPA>{}, T(-1), IC<IUA>{}, T(1), NO{}, Z0, Z0, Z0, Z0);          // mpc.py:303-311
    f(IC<10>{}, r++, -da - P.da_max, IC<IPA>{}, T(1), IC<IUA>{}, T(-1), NO{}, Z0, Z0, Z0, Z0);
    f(IC<11>{}, r++, dd - P.ddf_max, IC<IPD>{}, T(-1), IC<IUD>{}, T(1), NO{}, Z0, Z0, Z0, Z0);
    f(IC<12>{}, r++, -dd - P.ddf_max, IC<IPD>{}, T(1), IC<IUD>{}, T(-1), NO{}, Z0, Z0, Z0, Z0);
    if (CINF && k == P.N - 1)
#pragma unroll 1
        for (int m = 0; m < P.n_cinf; m++)                                          // mpc.py:177-180
            f(IC<-1>{}, r++, P.cinf_A[m][0] * z[IV] + P.cinf_A[m][1] * u[0] - P.cinf_b[m], IC<IV>{}, P.cinf_A[m][0], IC<IUA>{},
              P.cinf_A[m][1], NO{}, Z0, Z0, Z0, Z0);
}

// prefetch the slacks (and multipliers) of all rows of node k of iterate buffer b into L1, issued before
// the node's other work so that the per-row loads further down hit; o = row_off(N, n_cinf, k)
template <bool WANT_S, typename T, typename W>
IGT_HD void prefetch_rows(const DevParams<T> &P, const W &w, int k, int b, int o)
{
    const int ns = k == 0 ? 8 : (k == P.N ? 3 : 13);
    if (W::rstg) {                                               // (the terminal-set rows of node N-1 are loaded in place)
        w.rows_fetch(b, o, ns);
        if (k == P.N - 1)
            for (int r = ns; r < ns + P.n_cinf; r++) { w.pf(w.L.oY(b) + o + r); if (WANT_S) w.pf(w.L.oS(b) + o + r); }
        return;
    }
    const int n = ns + (k == P.N - 1 ? P.n_cinf : 0);
    for (int r = 0; r < n; r++) {
        w.pf(w.L.oY(b) + o + r);
        if (WANT_S) w.pf(w.L.oS(b) + o + r);
    }
}

// the terminal-set rows of stage N-1 (mpc.py:177-180; workspace rows o + 13 ...) of iterate buffer b:
// f(r, A0, A1, b, s, y) per row.  IGT_CINF_BATCH: multipliers and slacks are loaded eight rows at a time before
// the rows' arithmetic (one exposed memory latency per group instead of one per row).
#ifndef IGT_CINF_BATCH
#define IGT_CINF_BATCH 0
#endif
template <typename T, typename W, typename F>
IGT_HD void cinf_rows(const DevParams<T> &P, const W &w, int b, int o, F &&f)
{
#if !IGT_CINF_BATCH
#pragma unroll 1
    for (int m = 0; m < P.n_cinf; m++)
        f(o + NSLOT + m, P.cinf_A[m][0], P.cinf_A[m][1], P.cinf_b[m], w.S(b, o + NSLOT + m), w.Y(b, o + NSLOT + m));
#else
#pragma unroll 1
    for (int m0 = 0; m0 < P.n_cinf; m0 += 8) {
        T s8[8], y8[8];
#pragma unroll
        for (int j = 0; j < 8; j++)
            if (m0 + j < P.n_cinf) { s8[j] = w.S(b, o + NSLOT + m0 + j); y8[j] = w.Y(b, o + NSLOT + m0 + j); }
#pragma unroll
        for (int j = 0; j < 8; j++)
            if (m0 + j < P.n_cinf)
                f(o + NSLOT + m0 + j, P.cinf_A[m0 + j][0], P.cinf_A[m0 + j][1], P.cinf_b[m0 + j], s8[j], y8[j]);
    }
#endif
}

// symmetric 11x11 / 9x9 storage (upper triangle, row-major)
IGT_HD constexpr int sym11(int i, int j) { return i <= j ? i * NW - i * (i - 1) / 2 + (j - i) : j * NW - j * (j - 1) / 2 + (i - j); }
IGT_HD constexpr int sym9(int i, int j) { return i <= j ? i * NA - i * (i - 1) / 2 + (j - i) : j * NA - j * (j - 1) / 2 + (i - j); }

// structural non-zeros of F = d zeta+ / d w  (rows: zeta+ [9], cols: w [11])
IGT_HD constexpr bool fmask(int a, int j)
{
    return (a == IX && (j == IX || j == IV || j == IPSI || j == IUA || j == IUD)) ||
           (a == IY && (j == IY || j == IV || j == IPSI || j == IUA || j == IUD)) ||
           (a == IS && (j == IS || j == IEY || j == IEPSI || j == IV || j == IUA || j == IUD)) ||
           (a == IEY && (j == IEY || j == IEPSI || j == IV || j == IUA || j == IUD)) ||
           (a == IEPSI && (j == IEY || j == IEPSI || j == IV || j == IUA || j == IUD)) ||
           (a == IV && (j == IV || j == IUA)) ||
           (a == IPSI && (j == IV || j == IPSI || j == IUA || j == IUD)) ||
           (a == IPA && j == IUA) || (a == IPD && j == IUD);
}

// F[9][11] = d zeta+ / d w of stage k from its stored compact sensitivities (see NSENS)
template <typename T, typename W>
IGT_HD void load_F(const DevParams<T> &P, const W &w, int k, T (*F)[NW])
{
#pragma unroll
    for (int a = 0; a < NA; a++)
#pragma unroll
        for (int j = 0; j < NW; j++) F[a][j] = T(0);
    F[IX][IX] = T(1); F[IY][IY] = T(1); F[IS][IS] = T(1); F[IV][IV] = T(1); F[IPSI][IPSI] = T(1);
    F[IPA][IUA] = T(1); F[IPD][IUD] = T(1);
    F[IV][IUA] = P.dt;
    F[IX][IV] = w.Sens(k, SX + 0); F[IX][IPSI] = w.Sens(k, SX + 1); F[IX][IUA] = w.Sens(k, SX + 2); F[IX][IUD] = w.Sens(k, SX + 3);
    F[IY][IV] = w.Sens(k, SY + 0); F[IY][IPSI] = w.Sens(k, SY + 1); F[IY][IUA] = w.Sens(k, SY + 2); F[IY][IUD] = w.Sens(k, SY + 3);
    F[IS][IEY] = w.Sens(k, SS + 0); F[IS][IEPSI] = w.Sens(k, SS + 1); F[IS][IV] = w.Sens(k, SS + 2);
    F[IS][IUA] = w.Sens(k, SS + 3); F[IS][IUD] = w.Sens(k, SS + 4);
    F[IEY][IEY] = w.Sens(k, SEY + 0); F[IEY][IEPSI] = w.Sens(k, SEY + 1); F[IEY][IV] = w.Sens(k, SEY + 2);
    F[IEY][IUA] = w.Sens(k, SEY + 3); F[IEY][IUD] = w.Sens(k, SEY + 4);
    F[IEPSI][IEY] = w.Sens(k, SEP + 0); F[IEPSI][IEPSI] = w.Sens(k, SEP + 1); F[IEPSI][IV] = w.Sens(k, SEP + 2);
    F[IEPSI][IUA] = w.Sens(k, SEP + 3); F[IEPSI][IUD] = w.Sens(k, SEP + 4);
    F[IPSI][IV] = w.Sens(k, SPS + 0); F[IPSI][IUA] = w.Sens(k, SPS + 1); F[IPSI][IUD] = w.Sens(k, SPS + 2);
}

// dt * Hess(lambda . f) on (ey, epsi, v, psi, df), added into the symmetric w-space Hessian
template <typename T>
IGT_HD void add_dyn_hessian(const DevParams<T> &P, const T *z, const T *u, const T *curv, const T *lam, T *H)
{
    const StepK<T> c = step_setup(P, z, u, curv);               // sin / cos of beta, beta + epsi, psi + beta
    T ey = z[IEY], v = z[IV];
    T K = curvature(z[IS], curv[0], curv[1], curv[2]);
    T t = c.tdf, rho = P.rho;
    T q = T(1) + rho * rho * t * t;
    T b1 = c.dbeta;
    T b2 = rho * T(2) * t * (T(1) - rho * rho) / (q * q) * (T(1) + t * t);
    T cth = c.c1b, sth = c.s1b, cph = c.cpb, sph = c.spb, cb = c.cb, sb = c.sb;
    T iD = T(1) / (T(1) - K * ey);
    T m = lam[IS] - K * lam[IEPSI], n = (lam[IEPSI] + lam[IPSI]) * P.inv_lr;
    T ley = lam[IEY], lx = lam[IX], ly = lam[IY];
    T G_ey = m * cth * K * iD * iD;
    T G_epsi = -m * sth * iD + ley * cth;
    T G_psi = -lx * sph + ly * cph;
    T G_b = G_epsi + n * cb + G_psi;
    T G_eyey = m * cth * T(2) * K * K * iD * iD * iD;
    T G_eyepsi = -m * sth * K * iD * iD;
    T G_epsiepsi = -m * cth * iD - ley * sth;
    T G_psipsi = -lx * cph - ly * sph;
    T G_bb = G_epsiepsi - n * sb + G_psipsi;
    T dt = P.dt;
    H[sym11(IEY, IEY)] += dt * v * G_eyey;
    H[sym11(IEY, IEPSI)] += dt * v * G_eyepsi;
    H[sym11(IEPSI, IEPSI)] += dt * v * G_epsiepsi;
    H[sym11(IPSI, IPSI)] += dt * v * G_psipsi;
    H[sym11(IEY, IV)] += dt * G_ey;
    H[sym11(IEPSI, IV)] += dt * G_epsi;
    H[sym11(IV, IPSI)] += dt * G_psi;
    H[sym11(IEY, IUD)] += dt * v * G_eyepsi * b1;
    H[sym11(IEPSI, IUD)] += dt * v * G_epsiepsi * b1;
    H[sym11(IPSI, IUD)] += dt * v * G_psipsi * b1;
    H[sym11(IV, IUD)] += dt * G_b * b1;
    H[sym11(IUD, IUD)] += dt * v * (G_bb * b1 * b1 + G_b * b2);
}

// gradient entries / Hessian entries kept per node (compile-time tables as functions so that every
// use indexes registers statically after unrolling)
IGT_HD constexpr int ge_idx(int e)
{
    return e == 0 ? IV : e == 1 ? IEY : e == 2 ? IX : e == 3 ? IY : e == 4 ? IUA : e == 5 ? IUD : e == 6 ? IPA : e == 7 ? IPD : IPSI;
}
IGT_HD constexpr int he_i(int e)
{
    return e == 0 ? IV : e == 1 ? IEY : e == 2 ? IX : e == 3 ? IX : e == 4 ? IY : e == 5 ? IUA : e == 6 ? IUD
         : e == 7 ? IPA : e == 8 ? IPA : e == 9 ? IPD : e == 10 ? IPD : e == 11 ? IV
         : e == 12 ? IEY : e == 13 ? IEPSI : e == 14 ? IPSI : e == 15 ? IEY : e == 16 ? IEPSI : e == 17 ? IV
         : e == 18 ? IEY : e == 19 ? IEPSI : e == 20 ? IPSI : e == 21 ? IV : e == 22 ? IX : IY;
}
IGT_HD constexpr int he_j(int e)
{
    return e == 0 ? IV : e == 1 ? IEY : e == 2 ? IX : e == 3 ? IY : e == 4 ? IY : e == 5 ? IUA : e == 6 ? IUD
         : e == 7 ? IPA : e == 8 ? IUA : e == 9 ? IPD : e == 10 ? IUD : e == 11 ? IUA
         : e == 12 ? IEPSI : e == 13 ? IEPSI : e == 14 ? IPSI : e == 15 ? IV : e == 16 ? IV : e == 17 ? IPSI
         : e == 18 ? IUD : e == 19 ? IUD : e == 20 ? IUD : e == 21 ? IUD : IPSI;
}

// what a node phase needs to know about the problem it works for
template <typename T>
struct NodeCtx {
    T curv[3], uprev[2], mu, alpha;
    const double *obs, *x0p, *obs_psi;    // obs_psi: this problem's [N+1] obstacle headings (OBCA mode) or null
    int cur, second_order, ls;
};

template <typename T, typename W>
IGT_HD void node_load(const DevParams<T> &P, const W &w, const NodeCtx<T> &c, int k, T *z, T *up, T *u)
{
    const int b = c.cur;
    constexpr int S = W::stride;
    const T *pz = w.ptr(w.L.oZ(b) + k * NZ), *pu = w.ptr(w.L.oU(b) + k * 2);
#pragma unroll
    for (int i = 0; i < NZ; i++) z[i] = pz[i * S];
    if (k == 0) { up[0] = c.uprev[0]; up[1] = c.uprev[1]; }
    else { up[0] = pu[-2 * S]; up[1] = pu[-1 * S]; }
    if (k < P.N) { u[0] = pu[0]; u[1] = pu[S]; } else { u[0] = u[1] = T(0); }
}

// Node phase 1 (independent of the barrier parameter and of the adjoint): sensitivities of stage k
// and the row summaries the adjoint sweep needs -- sum of g * s per gradient entry, and the node's
// share of the residual norms (primal residual, largest multiplier, min / max of s * y).
template <typename T, typename W>
IGT_HD void node_phase1(const DevParams<T> &P, const W &w, const NodeCtx<T> &c, int k)
{
    const int N = P.N, b = c.cur;
    const int o = row_off(N, P.n_cinf, k);
    prefetch_rows<true>(P, w, k, b, o);                          // they arrive while the sensitivities are computed
    T z[NZ], up[2], u[2];
    node_load(P, w, c, k, z, up, u);
    if (k < N) {
        T zn[NZ], Sc[NSENS];
        rk4_step_sens(P, z, u, c.curv, zn, Sc);
        { T *ps = w.ptr(w.L.oSens + k * NSENS);
#pragma unroll
          for (int e = 0; e < NSENS; e++) ps[e * W::stride] = Sc[e]; }
    }
    T gw[NW];
#pragma unroll
    for (int i = 0; i < NW; i++) gw[i] = T(0);
    T rp = T(0), s_max = T(0), sy_min = T(1e30), sy_max = T(0);
    w.rows_wait();
    visit_rows<false, W::obca>(P, k, z, up, u, T(c.obs[2 * k]), T(c.obs[2 * k + 1]), W::obca ? T(c.obs_psi[k]) : T(0),
                               [&](auto, int r, T cv, auto I0, T g0, auto I1, T g1, auto I2, T g2, T, T, T) {
        constexpr int i0 = decltype(I0)::value, i1 = decltype(I1)::value, i2 = decltype(I2)::value;
        const T s = w.row_s(b, o, r), y = w.row_y(b, o, r);
        gw[i0] += g0 * s;
        if constexpr (i1 >= 0) gw[i1] += g1 * s;
        if constexpr (i2 >= 0) gw[i2] += g2 * s;
        rp = fmax(rp, fabs(cv + y));
        s_max = fmax(s_max, s);
        T sy = s * y;
        sy_min = fmin(sy_min, sy); sy_max = fmax(sy_max, sy);
    });
    if (k == N - 1)
        cinf_rows(P, w, b, o, [&](int, T A0, T A1, T bb, T s, T y) {
            const T cv = A0 * z[IV] + A1 * u[0] - bb;
            gw[IV] += A0 * s; gw[IUA] += A1 * s;
            rp = fmax(rp, fabs(cv + y));
            s_max = fmax(s_max, s);
            T sy = s * y;
            sy_min = fmin(sy_min, sy); sy_max = fmax(sy_max, sy);
        });
#pragma unroll
    for (int e = 0; e < W::nge; e++) w.ptr(w.L.oGw + k * W::nge)[e * W::stride] = gw[ge_idx(e)];
    { T *pr = w.ptr(w.L.oRed + k * 4); pr[0] = rp; pr[W::stride] = s_max; pr[2 * W::stride] = sy_min; pr[3 * W::stride] = sy_max; }
}

// Node phase 2 (after the barrier update and the adjoint sweep): the rows' share of the perturbed
// KKT system of node k -- gradient sum of g * (s + (s c + mu) / y), Hessian sum of (s / y) g g' plus
// s * Hess(c) for the collision row -- and the dynamics second-order term dt * Hess(lambda_{k+1} . f).
template <typename T, typename W>
IGT_HD void node_phase2(const DevParams<T> &P, const W &w, const NodeCtx<T> &c, int k)
{
    const int N = P.N, b = c.cur;
    const T mu = c.mu;
    const int o = row_off(N, P.n_cinf, k);
    prefetch_rows<true>(P, w, k, b, o);
    T z[NZ], up[2], u[2];
    node_load(P, w, c, k, z, up, u);
    T g[NW], H[66];
#pragma unroll
    for (int i = 0; i < NW; i++) g[i] = T(0);
#pragma unroll
    for (int i = 0; i < 66; i++) H[i] = T(0);
    if (k < N && c.second_order) {
        T ln[NZ];
#pragma unroll
        for (int i = 0; i < NZ; i++) ln[i] = w.ptr(w.L.oLam + (k + 1) * NZ)[i * W::stride];
        add_dyn_hessian(P, z, u, c.curv, ln, H);
    }
    w.rows_wait();
    visit_rows<false, W::obca>(P, k, z, up, u, T(c.obs[2 * k]), T(c.obs[2 * k + 1]), W::obca ? T(c.obs_psi[k]) : T(0),
                               [&](auto, int r, T cv, auto I0, T g0, auto I1, T g1, auto I2, T g2, T hxx, T hxy, T hyy) {
        constexpr int i0 = decltype(I0)::value, i1 = decltype(I1)::value, i2 = decltype(I2)::value;
        const T s = w.row_s(b, o, r), y = w.row_y(b, o, r);
        T iy = T(1) / y, rhat = s * cv + mu, sig = s * iy, gr = s + rhat * iy;
        g[i0] += g0 * gr;
        H[sym11(i0, i0)] += sig * g0 * g0;
        if constexpr (i1 >= 0) {
            g[i1] += g1 * gr;
            H[sym11(i1, i1)] += sig * g1 * g1;
            H[sym11(i0, i1)] += sig * g0 * g1;
        }
        if constexpr (i2 >= 0) {                                  // OBCA row: heading entry, Gauss-Newton (no row Hessian)
            g[i2] += g2 * gr;
            H[sym11(i2, i2)] += sig * g2 * g2;
            H[sym11(i0, i2)] += sig * g0 * g2;
            H[sym11(i1, i2)] += sig * g1 * g2;
        }
        if constexpr (i0 == IX && i2 < 0) {
            H[sym11(IX, IX)] += s * hxx; H[sym11(IX, IY)] += s * hxy; H[sym11(IY, IY)] += s * hyy;
        }
    });
    if (k == N - 1)
        cinf_rows(P, w, b, o, [&](int, T A0, T A1, T bb, T s, T y) {
            const T cv = A0 * z[IV] + A1 * u[0] - bb;
            T iy = T(1) / y, rhat = s * cv + mu, sig = s * iy, gr = s + rhat * iy;
            g[IV] += A0 * gr;
            H[sym11(IV, IV)] += sig * A0 * A0;
            g[IUA] += A1 * gr;
            H[sym11(IUA, IUA)] += sig * A1 * A1;
            H[sym11(IV, IUA)] += sig * A0 * A1;
        });
#pragma unroll
    for (int e = 0; e < W::nge; e++) w.ptr(w.L.oGl + k * W::nge)[e * W::stride] = g[ge_idx(e)];
#pragma unroll
    for (int e = 0; e < W::nhe; e++) w.ptr(w.L.oHl + k * W::nhe)[e * W::stride] = H[sym11(he_i(e), he_j(e))];
}

// Closed-loop nonlinear rollout of candidate j of the line search (step alpha / 2^j) from the
// current iterate into buffer cand_buf(cur, j): controls and states only; the rows of the trial
// point are evaluated by node_phase3.  Tc(buffer, .) = (1 if the rollout stayed finite, cost).
template <typename T, typename W>
IGT_HD void rollout_item(const DevParams<T> &P, const W &w, const NodeCtx<T> &c, int j)
{
    const int N = P.N, b = c.cur, nb = cand_buf(c.cur, j);
    T alpha = c.alpha;
    for (int i = 0; i < j; i++) alpha *= T(0.5);
    T zn[NZ], upn[2] = { c.uprev[0], c.uprev[1] };
    T J = T(0), su = T(0);
    bool fail = false;
#pragma unroll
    for (int i = 0; i < NZ; i++) { zn[i] = T(c.x0p[i]); w.Z(nb, 0, i) = zn[i]; }
    for (int k = 0; k < N; k++) {
        T dw[NA];
        if (k + 1 < N) {
            w.template pf_run<NZ>(w.L.oZ(b) + (k + 1) * NZ);
            w.template pf_run<2>(w.L.oU(b) + (k + 1) * 2);
            w.template pf_run<2>(w.L.oKu + (k + 1) * 2);
            w.template pf_run<2 * NA>(w.L.oKK + (k + 1) * 2 * NA);
        }
        constexpr int S = W::stride;
        const T *pz = w.ptr(w.L.oZ(b) + k * NZ), *pu = w.ptr(w.L.oU(b) + k * 2), *pk = w.ptr(w.L.oKu + k * 2),
                *pK = w.ptr(w.L.oKK + k * 2 * NA);
        T *qu = w.ptr(w.L.oU(nb) + k * 2), *qd = w.ptr(w.L.oDu + (nb * N + k) * 2), *qz = w.ptr(w.L.oZ(nb) + (k + 1) * NZ);
#pragma unroll
        for (int i = 0; i < NZ; i++) dw[i] = zn[i] - pz[i * S];
        if (k == 0) { dw[IPA] = T(0); dw[IPD] = T(0); }
        else { dw[IPA] = upn[0] - pu[-2 * S]; dw[IPD] = upn[1] - pu[-1 * S]; }
        T d0 = alpha * pk[0], d1 = alpha * pk[S];
#pragma unroll
        for (int i = 0; i < NA; i++) { d0 += pK[i * S] * dw[i]; d1 += pK[(NA + i) * S] * dw[i]; }
        T un[2] = { pu[0] + d0, pu[S] + d1 };
        J += zn[IEPSI] * zn[IEPSI] + zn[IEY] * zn[IEY];
        su += un[0] * un[0] + un[1] * un[1];
        qu[0] = un[0]; qu[S] = un[1];
        qd[0] = d0; qd[S] = d1;
        T zz[NZ];
        rk4_step(P, zn, un, c.curv, zz);
        bool fin = true;
#pragma unroll
        for (int i = 0; i < NZ; i++) { zn[i] = zz[i]; qz[i * S] = zz[i]; fin = fin && (zz[i] == zz[i]) && fabs(zz[i]) < T(1e15); }
        if (!fin) { fail = true; break; }
        upn[0] = un[0]; upn[1] = un[1];
    }
    J += zn[IEPSI] * zn[IEPSI] + zn[IEY] * zn[IEY];
    w.Tc(nb, 0) = fail ? T(0) : T(1);
    w.Tc(nb, 1) = J + P.w_u * su;
}

// Node phase 3 (after the rollout of candidate j): slack / multiplier update of the rows of node k
// along the step actually taken (d w_k = new - old iterate), the fraction-to-boundary test, and the
// node's share of the infeasibility and of the barrier sum at the new point.
// Tr(buffer, k, .) = (sum |c + y|, sum log y, 1 if the boundary rule failed).
template <typename T, typename W>
IGT_HD void node_phase3(const DevParams<T> &P, const W &w, const NodeCtx<T> &c, int k, int j)
{
    const int N = P.N, b = c.cur, nb = cand_buf(c.cur, j);
    if (w.Tc(nb, 0) == T(0)) return;                            // the rollout left the finite range
    const int o = row_off(N, P.n_cinf, k);
    prefetch_rows<true>(P, w, k, b, o);
    T alpha = c.alpha;
    for (int i = 0; i < j; i++) alpha *= T(0.5);
    const T mu = c.mu, tau = fmax(P.tau_min, T(1) - mu);
    T z[NZ], up[2], u[2], zn[NZ], upn[2], un[2], dw[NW];
    node_load(P, w, c, k, z, up, u);
    constexpr int S = W::stride;
    const T *qz = w.ptr(w.L.oZ(nb) + k * NZ), *qu = w.ptr(w.L.oU(nb) + k * 2), *qd = w.ptr(w.L.oDu + (nb * N + k) * 2);
#pragma unroll
    for (int i = 0; i < NZ; i++) { zn[i] = qz[i * S]; dw[i] = zn[i] - z[i]; }
    if (k == 0) { upn[0] = c.uprev[0]; upn[1] = c.uprev[1]; }
    else { upn[0] = qu[-2 * S]; upn[1] = qu[-1 * S]; }
    if (k < N) { un[0] = qu[0]; un[1] = qu[S]; } else { un[0] = un[1] = T(0); }
    dw[IPA] = upn[0] - up[0]; dw[IPD] = upn[1] - up[1];
    if (k < N) { dw[IUA] = qd[0]; dw[IUD] = qd[S]; } else { dw[IUA] = dw[IUD] = T(0); }
    T *py = w.ptr(w.L.oY(nb) + o), *ps = w.ptr(w.L.oS(nb) + o);      // rows of the trial point: row r at py[r * S]
    const T ox = T(c.obs[2 * k]), oy = T(c.obs[2 * k + 1]), opsi = W::obca ? T(c.obs_psi[k]) : T(0);
    bool fail = false;
    T ynv[NSLOT];
    w.rows_wait();
    visit_rows<false, W::obca>(P, k, z, up, u, ox, oy, opsi, [&](auto SL, int r, T cv, auto I0, T g0, auto I1, T g1, auto I2, T g2, T, T, T) {
        constexpr int sl = decltype(SL)::value, i0 = decltype(I0)::value, i1 = decltype(I1)::value, i2 = decltype(I2)::value;
        const T s = w.row_s(b, o, r), y = w.row_y(b, o, r);
        T dc = g0 * dw[i0];
        if constexpr (i1 >= 0) dc += g1 * dw[i1];
        if constexpr (i2 >= 0) dc += g2 * dw[i2];
        T yn = y - alpha * (cv + y) - dc;
        T sn = s + (alpha * (s * cv + mu) + s * dc) / y;
        if (yn < (T(1) - tau) * y) fail = true;                 // fraction to the boundary
        sn = fmax(sn, (T(1) - tau) * s);                        // multiplier safeguard
        ynv[sl] = yn;
        py[r * S] = yn; ps[r * S] = sn;
    });
    // infeasibility and barrier sum at the trial point: the stage rows first, then (stage N-1) the
    // terminal-set rows, whose update along the step and value at the new point share one loop
    T th = T(0);
    LogSum<T> lg;
    if (!fail)
        visit_rows<false, W::obca>(P, k, zn, upn, un, ox, oy, opsi, [&](auto SL, int, T cv, auto, T, auto, T, auto, T, T, T, T) {
            constexpr int sl = decltype(SL)::value;
            th += fabs(cv + ynv[sl]);
            lg.add(ynv[sl]);
        });
    if (k == N - 1)
        cinf_rows(P, w, b, o, [&](int r, T A0, T A1, T bb, T s, T y) {
            const T cv = A0 * z[IV] + A1 * u[0] - bb;
            T dc = A0 * dw[IV];
            dc += A1 * dw[IUA];
            T yn = y - alpha * (cv + y) - dc;
            T sn = s + (alpha * (s * cv + mu) + s * dc) / y;
            if (yn < (T(1) - tau) * y) fail = true;
            sn = fmax(sn, (T(1) - tau) * s);
            w.Y(nb, r) = yn; w.S(nb, r) = sn;
            if (!fail) { th += fabs(A0 * zn[IV] + A1 * un[0] - bb + yn); lg.add(yn); }
        });
    { T *pt = w.ptr(w.L.oTr + (nb * (N + 1) + k) * 3); pt[0] = th; pt[S] = fail ? T(0) : lg.total(); pt[2 * S] = fail ? T(1) : T(0); }
}

// ------------------------------------------------------------------ the solver ---------
// BANK: gt_mpc problems take their value network from the bank, nets[net_idx[p]] of ProbIONet.  The pointer lives in a base
// that is empty without BANK, so the other solvers keep their layout (and their local-memory footprint).
template <typename T, bool BANK> struct SolverNet { const MlpNet<T> *net; };   // this problem's network
template <typename T> struct SolverNet<T, false> {};
template <typename T, typename W = Ws<T>, bool BANK = false>
struct Solver : SolverNet<T, BANK> {
    static constexpr bool obca = W::obca;
    static constexpr bool bank = BANK;
    const DevParams<T> &P;
    W w;
    T x0[NZ], uprev[2], curv[3], ctx[4];
    const double *obs;        // this problem's [N+1][2] forecast (AoS, read-only)
    const double *obs_psi = nullptr;   // this problem's [N+1] obstacle headings (OBCA mode)
    const double *x0p;        // this problem's x0[7] in the caller's array
    bool gt;                  // gt_mpc terminal cost
    T *mlp_scratch;           // [2][6][width] when gt (per-thread slab), else null
    int mlp_width;
    // iteration state
    int cur;                  // buffer holding the current iterate
    int status, iters, ls, need_back, trials;   // need_back: 2 = full backward, 1 = Riccati only, 0 = none
    bool done;
    T mu, reg, alpha, Jcur, lgcur, thetacur, phi;
    T reg_hint;               // set by a failed Riccati sweep: the shift that makes the failing stage's Quu positive definite
    T stat, rp, s_max, sy_min, sy_max;
    TermVal<T> tcur, tcand;
    T Jcand, lgcand, thetacand;   // trial quantities (without the terminal value term)
    T phi_noise = T(0);           // absolute noise floor of the merit (fp32 tensor-core value term)
    bool trial_ok;

    IGT_HD Solver(const DevParams<T> &P_) : P(P_) {}

    IGT_HD T ox(int k) const { return T(obs[2 * k]); }
    IGT_HD T oy(int k) const { return T(obs[2 * k + 1]); }
    IGT_HD T opsi(int k) const { return W::obca ? T(obs_psi[k]) : T(0); }
    // value of the collision row of node k at (x, y, psi) in the units the reference writes it in:
    // circle mpc.py:226 d_min^2 - |p - o|^2; OBCA mpc.py:216 d_min + 1e-6 - (dual value = rectangle distance)
    IGT_HD T collision_row_ref(int k, T x, T y, T psi) const
    {
        if (W::obca) { T gd[3]; return P.d_min + T(OBCA_MARGIN) - obca_rect_sdist(x, y, psi, ox(k), oy(k), opsi(k), gd); }
        const T dx = x - ox(k), dy = y - oy(k);
        return P.d_min * P.d_min - dx * dx - dy * dy;
    }

    // terminal value -(cost contribution): 'mpc' V = s_N - s_0 ; 'gt_mpc' V = MLP
    IGT_HD void terminal_value(T sN, T vN, TermVal<T> &t, bool want_deriv)
    {
        if (!gt) {
            t.V = sN - x0[IS]; t.gs = T(1); t.gv = T(0); t.Hss = t.Hsv = t.Hvv = T(0);
        } else if constexpr (BANK) {
            mlp_eval_thread_net(*this->net, sN, vN, ctx, mlp_scratch, mlp_scratch + 6 * mlp_width, mlp_width, t, want_deriv);
        } else {
            mlp_eval_thread(P, sN, vN, ctx, mlp_scratch, mlp_scratch + 6 * mlp_width, mlp_width, t, want_deriv);
        }
    }

    // stage k of the step-bound sweep: iterate, slacks (not the multipliers), sensitivities, gains
    IGT_HD void prefetch_bound(int b, int k) const
    {
        if (k > P.N) return;
        w.template pf_run<NZ>(w.L.oZ(b) + k * NZ);
        const int o = row_off(P.N, P.n_cinf, k);
        w.template pf_run<NSLOT>(w.L.oY(b) + o);                 // (first and last node: a few words of the next node as well)
        if (k == P.N) return;
        w.template pf_run<2>(w.L.oU(b) + k * 2);
        w.template pf_run<2>(w.L.oKu + k * 2);
        w.template pf_run<NSENS>(w.L.oSens + k * NSENS);
        w.template pf_run<2 * NA>(w.L.oKK + k * 2 * NA);
    }

    // next stage of the backward sweeps: sensitivities, node summaries, the few iterate entries used
    IGT_HD void prefetch_back(int b, int k, bool riccati) const
    {
        if (k < 0) return;
        w.template pf_run<NSENS>(w.L.oSens + k * NSENS);
        w.template pf_run<2>(w.L.oZ(b) + k * NZ + IEY);
        w.template pf_run<2>(w.L.oU(b) + k * 2);
        if (riccati) {
            w.template pf_run<W::nge>(w.L.oGl + k * W::nge);
            w.template pf_run<W::nhe>(w.L.oHl + k * W::nhe);
        } else {
            w.template pf_run<W::nge>(w.L.oGw + k * W::nge);
            w.template pf_run<4>(w.L.oRed + k * 4);
        }
    }

    IGT_HD void load_z(int b, int k, T *z) const
    {
#pragma unroll
        for (int i = 0; i < NZ; i++) z[i] = w.Z(b, k, i);
    }
    IGT_HD void load_up(int b, int k, T *up) const
    {
        if (k == 0) { up[0] = uprev[0]; up[1] = uprev[1]; }
        else { up[0] = w.U(b, k - 1, 0); up[1] = w.U(b, k - 1, 1); }
    }

    // tracking controller rollout towards cruise speed vt; returns the merit
    // J('mpc' cost) + 100 * sum of row violations (collision in metres).  If u_out is given the
    // controls are stored there ([N][2] doubles).
    IGT_HD T guess_rollout(T vt, double *u_out)
    {
        const int N = P.N;
        T z[NZ], up[2] = { uprev[0], uprev[1] };
        T J = T(0), su = T(0), viol = T(0);
#pragma unroll
        for (int i = 0; i < NZ; i++) z[i] = x0[i];
        J += z[IEPSI] * z[IEPSI] + z[IEY] * z[IEY];
        // the feed-forward steering angle takes two values along a route (pw_const curvature): the one of the arc is
        // computed once per rollout instead of three transcendental calls per step
        const T dff_arc = atan(T(2) * tan(asin(curv[2] * P.l_r)));
        for (int k = 0; k < N; k++) {
            T K = curvature(z[IS], curv[0], curv[1], curv[2]);
            T a = T(0.5) * (vt - z[IV]);
            a = fmin(fmax(a, up[0] - P.da_max), up[0] + P.da_max);
            a = fmin(fmax(a, P.a_min), P.a_max);
            T dff = K == T(0) ? T(0) : (K == curv[2] ? dff_arc : atan(T(2) * tan(asin(K * P.l_r))));
            T d = dff - T(0.3) * z[IEY] - T(0.8) * z[IEPSI];
            d = fmin(fmax(d, up[1] - P.ddf_max), up[1] + P.ddf_max);
            d = fmin(fmax(d, -P.df_max), P.df_max);
            T u[2] = { a, d };
            if (u_out) { u_out[2 * k] = double(a); u_out[2 * k + 1] = double(d); }
            su += a * a + d * d;
            if (k == N - 1)
                for (int m = 0; m < P.n_cinf; m++)
                    viol += fmax(T(0), P.cinf_A[m][0] * z[IV] + P.cinf_A[m][1] * a - P.cinf_b[m]);
            T zn[NZ];
            rk4_step(P, z, u, curv, zn);
#pragma unroll
            for (int i = 0; i < NZ; i++) z[i] = zn[i];
            up[0] = a; up[1] = d;
            J += z[IEPSI] * z[IEPSI] + z[IEY] * z[IEY];
            if (k + 1 < N) viol += fmax(T(0), z[IV] - P.v_max) + fmax(T(0), P.v_min - z[IV]);
            viol += fmax(T(0), fabs(z[IEY]) - P.ey_lim);
            if (W::obca) viol += fmax(T(0), collision_row_ref(k + 1, z[IX], z[IY], z[IPSI]));
            else { T dx = z[IX] - ox(k + 1), dy = z[IY] - oy(k + 1); viol += fmax(T(0), P.d_min - sqrt(dx * dx + dy * dy)); }
        }
        J += P.w_u * su - (z[IS] - x0[IS]);
        return J + T(100) * viol;
    }

    IGT_HD void load_inputs(const ProbIO &io, long p, bool has_ctx)
    {
        x0p = io.x0 + p * NZ;
        for (int i = 0; i < NZ; i++) x0[i] = T(x0p[i]);
        uprev[0] = T(io.u_prev[p * 2]); uprev[1] = T(io.u_prev[p * 2 + 1]);
        for (int i = 0; i < 3; i++) curv[i] = T(io.curv[p * 3 + i]);
        obs = io.obs + p * (P.N + 1) * 2;
        if (W::obca) obs_psi = io.obs_psi + p * (P.N + 1);
        gt = has_ctx;
        if (gt) for (int i = 0; i < 4; i++) ctx[i] = T(io.ctx[p * 4 + i]);
    }

    // cold-start rule: best of N_GUESS tracking rollouts (DESIGN.md "initial guess") -> u_out[N][2]
    IGT_HD void compute_guess(const ProbIO &io, long p, double *u_out)
    {
        load_inputs(io, p, false);
        const T speeds[N_GUESS] = { T(5.0), T(3.5), T(2.0), T(1.0), T(0.0) };
        T best = guess_rollout(speeds[0], nullptr);
        int bestg = 0;
        for (int g = 1; g < N_GUESS; g++) {
            T m = guess_rollout(speeds[g], nullptr);
            if (m < best) { best = m; bestg = g; }
        }
        guess_rollout(speeds[bestg], u_out);
    }

    // load inputs, pre-check x0, build the initial iterate from the controls u_src[N][2]
    // (warm start or cold-start guess).  Returns false if the problem is finished already.
    IGT_HD bool init(const ProbIO &io, long p, bool has_ctx, const double *u_src, bool warm)
    {
        const int N = P.N;
        load_inputs(io, p, has_ctx);
        cur = 0; status = 1; iters = 0; ls = 0; need_back = 2; done = false; trials = 0;
        if constexpr (BANK) {   // an index outside the bank or naming an empty slot: no solve, never dereferenced
            if (gt) {
                const ProbIONet<T> &bio = bank_io<T>(io);
                const int k = bio.net_idx[p];
                if (!bio.net_ok(k)) { status = 7; done = true; return false; }
                this->net = bio.nets + k;
            }
        }
        mu = warm ? P.mu0_warm : P.mu0; reg = T(0); alpha = T(1); reg_hint = T(0);
        const T y_min = warm ? P.y_init_min_warm : P.y_init_min;
        {   // rows on x0 alone: mpc.py:316-317 and :298-299 at k = 0
            const T tol = P.x0_tol;
            if (!(x0[IV] >= P.v_min - tol && x0[IV] <= P.v_max + tol && fabs(x0[IEY]) <= P.ey_lim + tol)) {
                status = 2; done = true;
                return false;
            }
        }
        {
            T z[NZ];
            for (int i = 0; i < NZ; i++) { z[i] = x0[i]; w.Z(0, 0, i) = z[i]; }
            for (int k = 0; k < N; k++) {
                T u[2] = { T(u_src[2 * k]), T(u_src[2 * k + 1]) }, zn[NZ];
                w.U(0, k, 0) = u[0]; w.U(0, k, 1) = u[1];
                rk4_step(P, z, u, curv, zn);
                for (int i = 0; i < NZ; i++) { z[i] = zn[i]; w.Z(0, k + 1, i) = zn[i]; }
            }
        }
        // slacks / multipliers, J, sum log y, theta of the initial iterate
        T J = T(0), su = T(0), th = T(0);
        LogSum<T> lg;
        for (int k = 0; k <= N; k++) {
            T z[NZ], up[2], u[2] = { T(0), T(0) };
            load_z(0, k, z); load_up(0, k, up);
            if (k < N) { u[0] = w.U(0, k, 0); u[1] = w.U(0, k, 1); su += u[0] * u[0] + u[1] * u[1]; }
            J += z[IEPSI] * z[IEPSI] + z[IEY] * z[IEY];
            int o = row_off(N, P.n_cinf, k);
            visit_rows<true, W::obca>(P, k, z, up, u, ox(k), oy(k), opsi(k), [&](auto, int r, T c, auto, T, auto, T, auto, T, T, T, T) {
                T y = fmax(-c, y_min);
                w.Y(0, o + r) = y;
                w.S(0, o + r) = mu / y;
                lg.add(y);
                th += fabs(c + y);
            });
        }
        Jcur = J + P.w_u * su; lgcur = lg.total(); thetacur = th;
        return true;
    }

    // value of the terminal state of buffer b
    IGT_HD void terminal_of(int b, TermVal<T> &t, bool want_deriv)
    {
        terminal_value(w.Z(b, P.N, IS), w.Z(b, P.N, IV), t, want_deriv);
    }

    IGT_HD NodeCtx<T> node_ctx() const
    {
        NodeCtx<T> c;
        c.curv[0] = curv[0]; c.curv[1] = curv[1]; c.curv[2] = curv[2];
        c.uprev[0] = uprev[0]; c.uprev[1] = uprev[1];
        c.mu = mu; c.alpha = alpha; c.obs = obs; c.obs_psi = obs_psi; c.x0p = x0p; c.cur = cur; c.second_order = P.second_order; c.ls = ls;
        return c;
    }

    // sweep 2: adjoint recursion and KKT residuals from the node summaries of node_phase1
    IGT_HD void adjoint_sweep()
    {
        const int N = P.N, b = cur;
        T lam[NA];
        stat = T(0); rp = T(0); s_max = T(0); sy_min = T(1e30); sy_max = T(0);
        for (int k = N; k >= 0; k--) {
            T gw[NW];
            prefetch_back(b, k - IGT_PF_DIST, false);
#pragma unroll
            for (int i = 0; i < NW; i++) gw[i] = T(0);
#pragma unroll
            for (int e = 0; e < W::nge; e++) gw[ge_idx(e)] = w.Gw(k, e);
            rp = fmax(rp, w.Red(k, 0)); s_max = fmax(s_max, w.Red(k, 1));
            sy_min = fmin(sy_min, w.Red(k, 2)); sy_max = fmax(sy_max, w.Red(k, 3));
            const T ey = w.Z(b, k, IEY), epsi = w.Z(b, k, IEPSI);
            if (k == N) {
#pragma unroll
                for (int i = 0; i < NA; i++) lam[i] = gw[i];
                lam[IS] -= tcur.gs; lam[IV] -= tcur.gv;
            } else {
                T F[NA][NW];
                load_F(P, w, k, F);
                T ln[NA];
#pragma unroll
                for (int i = 0; i < NA; i++) ln[i] = lam[i];
#pragma unroll
                for (int j = 0; j < 2; j++) {
                    T gu = T(2) * P.w_u * w.U(b, k, j) + gw[NA + j];
#pragma unroll
                    for (int a = 0; a < NA; a++) if (fmask(a, NA + j)) gu += F[a][NA + j] * ln[a];
                    stat = fmax(stat, fabs(gu));
                }
#pragma unroll
                for (int i = 0; i < NA; i++) {
                    T acc = gw[i];
#pragma unroll
                    for (int a = 0; a < NA; a++) if (fmask(a, i)) acc += F[a][i] * ln[a];
                    lam[i] = acc;
                }
            }
            lam[IEY] += T(2) * ey; lam[IEPSI] += T(2) * epsi;
#pragma unroll
            for (int i = 0; i < NZ; i++) w.Lam(k, i) = lam[i];
        }
    }

    // The current iterate satisfies the reference's own IPOPT tolerances (mpc.py:133-135: tol = dual_inf_tol =
    // constr_viol_tol = 1e-3, IPOPT's default compl_inf_tol 1e-4; the primal bound tightened to the north star's 1e-6):
    // when the solve ends in a failure (iteration cap, regularisation limit, budget of forward passes) at such a point,
    // it is returned with status 6 instead.  Never pre-empts the tight convergence test.  Residuals are those of
    // the last adjoint sweep.
    IGT_HD bool acceptable() const
    {
        return P.acc_tol > T(0) && stat <= P.acc_tol * fmax(T(1), s_max) && rp <= P.acc_rp && sy_max <= P.acc_comp;
    }

    // convergence test, exits, barrier update.  Residuals are those of the last adjoint sweep; a
    // regularisation change alone does not alter them, so repeating the test is harmless.
    IGT_HD void test_and_update()
    {
        if (stat <= P.tol * fmax(T(1), s_max) && rp <= P.tol_rp && sy_max <= P.tol_comp) {
            status = 0; done = true;
            return;
        }
        if (iters >= P.max_iter) { status = acceptable() ? 6 : 1; done = true; return; }
        if (iters >= P.stall_iter && rp > P.stall_rp) { status = 5; done = true; return; }   // stalled, infeasible
        while (mu > P.mu_floor &&
               fmax(fmax(stat, rp), fmax(fabs(sy_max - mu), fabs(sy_min - mu))) <= P.kappa_eps * mu)
            mu = fmax(P.mu_floor, fmin(P.kappa_mu * mu, pow(mu, P.theta_mu)));
        phi = Jcur - tcur.V - mu * lgcur;
    }

    // sweep 3: Riccati recursion on the perturbed KKT system; node-local terms come from
    // node_phase2.  Returns false if some Quu + reg I is not positive definite.
    IGT_HD bool riccati_sweep()
    {
        const int N = P.N, b = cur;
        T Vx[NA], Vxx[45];
        {
            T g[NW], H[66];
#pragma unroll
            for (int i = 0; i < NW; i++) g[i] = T(0);
#pragma unroll
            for (int i = 0; i < 66; i++) H[i] = T(0);
#pragma unroll
            for (int e = 0; e < W::nge; e++) g[ge_idx(e)] = w.Gl(N, e);
#pragma unroll
            for (int e = 0; e < 5; e++) H[sym11(he_i(e), he_j(e))] = w.Hl(N, e);     // terminal rows: ey, collision
            if (W::obca) {                                                            // ... and the OBCA row's heading entries
                H[sym11(IPSI, IPSI)] = w.Hl(N, 14); H[sym11(IX, IPSI)] = w.Hl(N, 22); H[sym11(IY, IPSI)] = w.Hl(N, 23);
            }
#pragma unroll
            for (int i = 0; i < NA; i++) {
                Vx[i] = g[i];
#pragma unroll
                for (int j = i; j < NA; j++) Vxx[sym9(i, j)] = H[sym11(i, j)];
            }
            Vx[IEY] += T(2) * w.Z(b, N, IEY); Vx[IEPSI] += T(2) * w.Z(b, N, IEPSI);
            Vx[IS] -= tcur.gs; Vx[IV] -= tcur.gv;
            Vxx[sym9(IEY, IEY)] += T(2); Vxx[sym9(IEPSI, IEPSI)] += T(2);
            Vxx[sym9(IS, IS)] -= tcur.Hss; Vxx[sym9(IS, IV)] -= tcur.Hsv; Vxx[sym9(IV, IV)] -= tcur.Hvv;
        }
        for (int k = N - 1; k >= 0; k--) {
            T F[NA][NW];
            prefetch_back(b, k - IGT_PF_DIST_R, true);
            load_F(P, w, k, F);
            T g[NW], H[66];
            // g = F' Vx,  H = F' Vxx F   (structural zeros skipped at compile time)
            T VF[NA][NW];
#pragma unroll
            for (int a = 0; a < NA; a++)
#pragma unroll
                for (int j = 0; j < NW; j++) {
                    T acc = T(0);
#pragma unroll
                    for (int c = 0; c < NA; c++) if (fmask(c, j)) acc += Vxx[sym9(a, c)] * F[c][j];
                    VF[a][j] = acc;
                }
#pragma unroll
            for (int i = 0; i < NW; i++) {
                T acc = T(0);
#pragma unroll
                for (int a = 0; a < NA; a++) if (fmask(a, i)) acc += F[a][i] * Vx[a];
                g[i] = acc;
#pragma unroll
                for (int j = i; j < NW; j++) {
                    T hh = T(0);
#pragma unroll
                    for (int a = 0; a < NA; a++) if (fmask(a, i)) hh += F[a][i] * VF[a][j];
                    H[sym11(i, j)] = hh;
                }
            }
            // stage cost (mpc.py:359-364) and the node-local terms
            g[IEY] += T(2) * w.Z(b, k, IEY); g[IEPSI] += T(2) * w.Z(b, k, IEPSI);
            g[IUA] += T(2) * P.w_u * w.U(b, k, 0); g[IUD] += T(2) * P.w_u * w.U(b, k, 1);
            H[sym11(IEY, IEY)] += T(2); H[sym11(IEPSI, IEPSI)] += T(2);
            H[sym11(IUA, IUA)] += T(2) * P.w_u; H[sym11(IUD, IUD)] += T(2) * P.w_u;
#pragma unroll
            for (int e = 0; e < W::nge; e++) g[ge_idx(e)] += w.Gl(k, e);
#pragma unroll
            for (int e = 0; e < W::nhe; e++) H[sym11(he_i(e), he_j(e))] += w.Hl(k, e);
            T q00 = H[sym11(IUA, IUA)] + reg, q11 = H[sym11(IUD, IUD)] + reg, q01 = H[sym11(IUA, IUD)];
            T det = q00 * q11 - q01 * q01;
            if (!(q00 > T(0) && det > T(1e-12) * q00 * q11)) {
                const T a_ = H[sym11(IUA, IUA)], b_ = H[sym11(IUD, IUD)];
                const T lmin = T(0.5) * (a_ + b_) - sqrt(T(0.25) * (a_ - b_) * (a_ - b_) + q01 * q01);
                reg_hint = lmin < T(0) ? -lmin * P.reg_jump : T(0);
                return false;
            }
            T idet = T(1) / det;
            T i00 = q11 * idet, i11 = q00 * idet, i01 = -q01 * idet;
            T k0 = -(i00 * g[IUA] + i01 * g[IUD]), k1 = -(i01 * g[IUA] + i11 * g[IUD]);
            T K0[NA], K1[NA];
#pragma unroll
            for (int j = 0; j < NA; j++) {
                T ha = H[sym11(j, IUA)], hd = H[sym11(j, IUD)];
                K0[j] = -(i00 * ha + i01 * hd);
                K1[j] = -(i01 * ha + i11 * hd);
                w.KK(k, 0, j) = K0[j]; w.KK(k, 1, j) = K1[j];
            }
            w.ku(k, 0) = k0; w.ku(k, 1) = k1;
            // (Quu + reg I) [k K] = -[g_u H_ux], so the value function of the stage reduces to the Schur
            // complement form; the reg terms keep it exact when Quu had to be regularised
            const T rk0 = reg * k0, rk1 = reg * k1;
#pragma unroll
            for (int i = 0; i < NA; i++)
                Vx[i] = g[i] + H[sym11(i, IUA)] * k0 + H[sym11(i, IUD)] * k1 - K0[i] * rk0 - K1[i] * rk1;
#pragma unroll
            for (int i = 0; i < NA; i++)
#pragma unroll
                for (int j = i; j < NA; j++)
                    Vxx[sym9(i, j)] = H[sym11(i, j)] + H[sym11(i, IUA)] * K0[j] + H[sym11(i, IUD)] * K1[j]
                                      - reg * (K0[i] * K0[j] + K1[i] * K1[j]);
        }
        return true;
    }

    // largest step keeping every slack inside the fraction-to-boundary rule on the LINEARISED
    // closed-loop model (d zeta+ = F [d zeta; d u], d u = ku + Ku d zeta)
    IGT_HD void step_bound()
    {
        const int N = P.N, b = cur;
        const T tau = fmax(P.tau_min, T(1) - mu);
        // the binding row is kept as a (numerator, denominator) pair updated with selects and divided once at the end:
        // a branch with an inlined fp64 division behind every row (taken by some lane of a warp almost always) cost a
        // third of this sweep's instructions
        T an = T(1), ad = T(1), dz[NA];
#pragma unroll
        for (int i = 0; i < NA; i++) dz[i] = T(0);
        for (int k = 0; k <= N; k++) {
            T z[NZ], up[2], u[2] = { T(0), T(0) }, dw[NW];
            prefetch_bound(b, k + IGT_PF_DIST);
            // every load of the stage is issued up front (one exposed memory latency per stage, not one per row:
            // the rows below branch, so the compiler cannot hoist their loads itself)
            const int o = row_off(N, P.n_cinf, k), sb0 = slot_base(N, k);
            T yv[NSLOT];
#pragma unroll
            for (int sl = 0; sl < NSLOT; sl++) if (slot_used(N, k, sl)) yv[sl] = w.Y(b, o + sl - sb0);
            load_z(b, k, z); load_up(b, k, up);
#pragma unroll
            for (int i = 0; i < NA; i++) dw[i] = dz[i];
            dw[IUA] = T(0); dw[IUD] = T(0);
            if (k < N) {
                u[0] = w.U(b, k, 0); u[1] = w.U(b, k, 1);
                T d0 = w.ku(k, 0), d1 = w.ku(k, 1);
#pragma unroll
                for (int j = 0; j < NA; j++) { d0 += w.KK(k, 0, j) * dz[j]; d1 += w.KK(k, 1, j) * dz[j]; }
                dw[IUA] = d0; dw[IUD] = d1;
                // the next stage's state change right away: the 26 sensitivities are dead before the rows are visited
                // (their registers were what this sweep spilled: 530 -> 338 bytes of spills in the kernel's main function)
                T F[NA][NW];
                load_F(P, w, k, F);
#pragma unroll
                for (int i = 0; i < NA; i++) {
                    T acc = T(0);
#pragma unroll
                    for (int j = 0; j < NW; j++) if (fmask(i, j)) acc += F[i][j] * dw[j];
                    dz[i] = acc;
                }
            }
            visit_rows<false, W::obca>(P, k, z, up, u, ox(k), oy(k), opsi(k), [&](auto SL, int, T c, auto I0, T g0, auto I1, T g1, auto I2, T g2, T, T, T) {
                constexpr int sl = decltype(SL)::value, i0 = decltype(I0)::value, i1 = decltype(I1)::value, i2 = decltype(I2)::value;
                const T y = yv[sl];
                T dc = g0 * dw[i0];
                if constexpr (i1 >= 0) dc += g1 * dw[i1];
                if constexpr (i2 >= 0) dc += g2 * dw[i2];
                T dy = -(c + y) - dc;
                const T ty = tau * y;
                const bool tighter = dy < T(0) && -dy * an > ty * ad;
                an = tighter ? ty : an; ad = tighter ? -dy : ad;
            });
            if (k == N - 1) {
#pragma unroll 1
                for (int m0 = 0; m0 < P.n_cinf; m0 += 8) {
                    T y8[8];
#pragma unroll
                    for (int j = 0; j < 8; j++) if (m0 + j < P.n_cinf) y8[j] = w.Y(b, o + NSLOT + m0 + j);
#pragma unroll
                    for (int j = 0; j < 8; j++)
                        if (m0 + j < P.n_cinf) {
                            const T A0 = P.cinf_A[m0 + j][0], A1 = P.cinf_A[m0 + j][1], y = y8[j];
                            const T c = A0 * z[IV] + A1 * u[0] - P.cinf_b[m0 + j];
                            T dc = A0 * dw[IV];
                            dc += A1 * dw[IUA];
                            T dy = -(c + y) - dc;
                            const T ty = tau * y;
                            const bool tighter = dy < T(0) && -dy * an > ty * ad;
                            an = tighter ? ty : an; ad = tighter ? -dy : ad;
                        }
                }
            }
        }
        alpha = (an / ad) * P.alpha_safety;
    }

    // The backward pass is split so that the kernels can run the node-local work of all stages of
    // all problems of a CTA in parallel (node_phase1 / node_phase2) between the sequential sweeps:
    //   [node_phase1 of every node]  backward_pre()  [node_phase2 of every node]  backward_post()
    // backward_pre: adjoint sweep (if the iterate changed), convergence test, barrier update.
    // Returns true if node_phase2 has to run before backward_post (fresh iterate, still going).
    IGT_HD bool backward_pre()
    {
        const bool fresh = need_back == 2;
        if (fresh) { adjoint_sweep(); need_back = 1; }
        test_and_update();
        return fresh && !done;
    }

    // backward_post: Riccati sweep (regularisation raised until it succeeds) and the step bound
    IGT_HD void backward_post()
    {
        for (;;) {
            if (riccati_sweep()) break;
            reg = fmax(fmax(reg * P.reg_up, P.reg_min), reg_hint);
            if (reg > P.reg_max) { status = acceptable() ? 6 : 3; done = true; return; }
        }
        need_back = 0;
        ls = 0;
        step_bound();
    }

    // whole backward pass by one thread (tests/hostsim; the kernels interleave the CTA-wide phases)
    IGT_HD void backward()
    {
        if (need_back == 2) {
            const NodeCtx<T> c = node_ctx();
            for (int k = 0; k <= P.N; k++) node_phase1(P, w, c, k);
        }
        if (backward_pre()) {
            const NodeCtx<T> c = node_ctx();
            for (int k = 0; k <= P.N; k++) node_phase2(P, w, c, k);
        }
        if (!done) backward_post();
    }

    // gather the results of candidate j (rollout_item + node_phase3): trial_ok, cost, infeasibility, barrier sum
    IGT_HD void collect_trial(int j)
    {
        const int nb = cand_buf(cur, j);
        trial_ok = w.Tc(nb, 0) != T(0);
        if (!trial_ok) return;
        T th = T(0), lg = T(0), bad = T(0);
#if !defined(IGT_COLLECT_BATCH)
        for (int k = 0; k <= P.N; k++) { th += w.Tr(nb, k, 0); lg += w.Tr(nb, k, 1); bad += w.Tr(nb, k, 2); }
#else
        for (int k0 = 0; k0 <= P.N; k0 += 8) {                   // eight nodes' loads in flight at a time, summed in node order
            T t8[8][3];
#pragma unroll
            for (int i = 0; i < 8; i++)
                if (k0 + i <= P.N) { t8[i][0] = w.Tr(nb, k0 + i, 0); t8[i][1] = w.Tr(nb, k0 + i, 1); t8[i][2] = w.Tr(nb, k0 + i, 2); }
#pragma unroll
            for (int i = 0; i < 8; i++)
                if (k0 + i <= P.N) { th += t8[i][0]; lg += t8[i][1]; bad += t8[i][2]; }
        }
#endif
        Jcand = w.Tc(nb, 1); thetacand = th; lgcand = lg;
        if (bad > T(0)) trial_ok = false;
    }

    // acceptance test of the collected candidate (needs tcand, its terminal value)
    IGT_HD bool trial_passes() const
    {
        if (!trial_ok) return false;
        T phin = Jcand - tcand.V - mu * lgcand;
        return (phin == phin) && fabs(phin) < T(1e30) &&
               (phin < phi - P.eps_phi * fabs(phi) || thetacand < thetacur * (T(1) - P.gamma_theta) ||
                (thetacand <= P.theta_small && phin <= phi + fmax(P.eps_phi * fmax(T(1), fabs(phi)), phi_noise)));
    }

    // close a batch of `tried` candidates alpha, alpha/2, ...: `jacc` >= 0 is the first that passed (the
    // one sequential halving would have stopped at; collect_trial(jacc) is the last one collected)
    IGT_HD void finish_trials(int jacc, int tried)
    {
        if (jacc >= 0) {
            cur = cand_buf(cur, jacc);
            Jcur = Jcand; lgcur = lgcand; thetacur = thetacand; tcur = tcand;
            reg = reg > P.reg_min ? reg / P.reg_down : T(0);
            need_back = 2;
            iters++;
        } else {
            for (int i = 0; i < tried; i++) alpha *= T(0.5);
            ls += tried;
            if (ls >= P.n_alpha) {
                reg = fmax(reg * P.reg_up, P.reg_min);
                iters++;
                if (reg > P.reg_max) { status = acceptable() ? 6 : 4; done = true; }
                need_back = 1;
            }
        }
        // budget of forward passes, checked between iterations like the iteration cap
        if (!done && (jacc >= 0 || need_back == 1) && trials >= P.max_trials) { status = (jacc < 0 && acceptable()) ? 6 : 1; done = true; }
    }

    // judge candidates 0 .. nj-1 in the order sequential halving would try them
    // (stored: the terminal value terms of the candidates were evaluated CTA-wide on the tensor cores and
    // left in Tc(buffer, 2..7), see tc_candidates)
    // judge candidates j0 .. j1-1 (none of the earlier ones passed); returns the first that passes or -1
    IGT_HD int judge_trials(int j0, int j1, bool stored, int &tried)
    {
        int jacc = -1;
        for (int j = j0; j < j1 && jacc < 0; j++) {
            trials++; tried++;
            collect_trial(j);
            if (trial_ok) {
                const int nb = cand_buf(cur, j);
                if (stored) {
                    tcand.V = w.Tc(nb, 2); tcand.gs = w.Tc(nb, 3); tcand.gv = w.Tc(nb, 4);
                    tcand.Hss = w.Tc(nb, 5); tcand.Hsv = w.Tc(nb, 6); tcand.Hvv = w.Tc(nb, 7);
                } else {
                    terminal_of(nb, tcand, true);
                }
            }
            if (trial_passes()) jacc = j;
        }
        return jacc;
    }
    IGT_HD void accept_trials(int nj, bool stored = false)
    {
        int tried = 0;
        const int jacc = judge_trials(0, nj, stored, tried);
        finish_trials(jacc, tried);
    }

    // one candidate evaluated start to finish by one thread (tests/hostsim; the kernels run the
    // rollouts and node_phase3 of all candidates CTA-wide, see trial_phase_cta)
    IGT_HD void trial_serial()
    {
        const NodeCtx<T> c = node_ctx();
        rollout_item(P, w, c, 0);
        for (int k = 0; k <= P.N; k++) node_phase3(P, w, c, k, 0);
        accept_trials(1);
    }

    // write the outputs of this problem (x, u, cost, max row violation in reference units)
    IGT_HD void write_out(const ProbIO &io, long p)
    {
        const int N = P.N, b = cur;
        if (status == 2 || (BANK && status == 7)) {
            for (int i = 0; i < (N + 1) * NZ; i++) io.x[p * (N + 1) * NZ + i] = NAN;
            for (int i = 0; i < N * 2; i++) io.u[p * N * 2 + i] = NAN;
            io.cost[p] = NAN; io.viol[p] = INFINITY; io.status[p] = BANK ? status : 2; io.iters[p] = 0;
            return;
        }
        T m = T(0);
        for (int k = 0; k <= N; k++) {
            T z[NZ], up[2];
            load_z(b, k, z); load_up(b, k, up);
            for (int i = 0; i < NZ; i++) io.x[(p * (N + 1) + k) * NZ + i] = double(z[i]);
            m = fmax(m, fabs(z[IEY]) - P.ey_lim);
            if (k >= 1) m = fmax(m, collision_row_ref(k, z[IX], z[IY], z[IPSI]));
            if (k < N) {
                T u[2] = { w.U(b, k, 0), w.U(b, k, 1) };
                io.u[(p * N + k) * 2] = double(u[0]); io.u[(p * N + k) * 2 + 1] = double(u[1]);
                m = fmax(m, fmax(P.v_min - z[IV], z[IV] - P.v_max));
                m = fmax(m, fmax(P.a_min - u[0], u[0] - P.a_max));
                m = fmax(m, fabs(u[1]) - P.df_max);
                m = fmax(m, fabs(u[0] - up[0]) - P.da_max);
                m = fmax(m, fabs(u[1] - up[1]) - P.ddf_max);
                if (k == N - 1)
                    for (int q = 0; q < P.n_cinf; q++)
                        m = fmax(m, P.cinf_A[q][0] * z[IV] + P.cinf_A[q][1] * u[0] - P.cinf_b[q]);
            }
        }
        io.cost[p] = double(Jcur - tcur.V);
        io.viol[p] = double(m);
        io.status[p] = status;
        io.iters[p] = iters;
    }
};

// Whole solve of problem p in workspace slot `slot`, one thread, start to finish.
// (tests/hostsim calls this on the CPU; the kernels use the persistent-lane driver below.)
template <typename T, bool OBCA = false>
IGT_HD void solve_problem(const DevParams<T> &P, const ProbIO &io, T *ws_base, long slot, long p,
                          double *guess_buf, T *mlp_scratch, int mlp_width)
{
    Solver<T, Ws<T, 32, OBCA>> sv(P);
    sv.w.init_layout(P.N, P.n_cinf);
    sv.w.bind(ws_base, slot);
    sv.mlp_scratch = mlp_scratch; sv.mlp_width = mlp_width;
    const double *u_src = io.u_init ? io.u_init + p * P.N * 2 : guess_buf;
    if (!io.u_init) sv.compute_guess(io, p, guess_buf);
    if (sv.init(io, p, io.ctx != nullptr, u_src, io.u_init != nullptr)) {
        sv.terminal_of(sv.cur, sv.tcur, true);
        while (!sv.done) {
            if (sv.need_back) sv.backward();
            if (sv.done) break;
            sv.trial_serial();
        }
    }
    sv.write_out(io, p);
}

#ifdef __CUDACC__
// Scheduler state shared by all lanes of a solve launch (device memory, zeroed by the host before it).
struct Sched {
    unsigned long long *counter;   // next fresh problem
};

// Persistent-lane driver: every thread owns one workspace slot and keeps pulling problems from
// a global counter until none are left.  All 32 lanes of a warp walk the phases of an iteration
// (backward sweeps, forward trial, acceptance) together, each lane on its own problem and at
// its own iteration count, so a slow or failing problem delays only its own lane.
// (An earlier version handed the stragglers of the tail over to idle warps of other CTAs through a
// resume queue.  Since the node phases and the line-search candidates of a thin CTA are dealt out over
// all of its threads anyway, packing stragglers no longer shortens a round -- its length is the serial
// latency of one problem's sweeps -- and the queue polling cost 2 %: removed.)
template <typename T>
__device__ __forceinline__ void term_from_tc(const float *o, TermVal<T> &t)
{
    t.V = T(o[0]); t.gs = T(o[1]); t.gv = T(o[2]); t.Hss = T(o[3]); t.Hsv = T(o[4]); t.Hvv = T(o[5]);
}

// TC = true: the gt_mpc value term of all 256 problems of the CTA is evaluated together on the
// tensor cores (mlp_tc.cuh) at the two CTA-uniform points of the loop where it is needed.
// CTA-wide node phases.  The node-local work of an iteration (node_phase1: sensitivities and row
// summaries; node_phase2: perturbed-KKT terms of the rows and the dynamics second-order term)
// depends only on that node's (z_k, u_k, y, s) and on a few per-problem scalars, so the (problem,
// node) pairs of every problem of the CTA that needs the phase are independent work items; they
// are dealt out over all threads of the CTA.  Every lane is busy whatever the mix of per-problem
// states, a lone straggler gets its N + 1 nodes done by N + 1 threads at once, and the loop body is
// small enough to stay in the instruction cache.
#ifndef IGT_MAX_SOLVE_BLOCK
#define IGT_MAX_SOLVE_BLOCK 256
#endif
constexpr int MAX_SOLVE_BLOCK = IGT_MAX_SOLVE_BLOCK;
template <typename T>
struct NodeList {                    // shared-memory work list of one CTA-wide phase
    int cslot;                       // constant-memory slot of this launch's parameters (ConstP<T>::get)
    void *rstg;                      // row-staging buffer in dynamic shared memory (Ws RSTG), or null
    int wcnt[MAX_SOLVE_BLOCK / 32];
    int slot[MAX_SOLVE_BLOCK];
    int more[MAX_SOLVE_BLOCK];       // CTA-wide value term, second pass: this problem's first candidate was rejected
    NodeCtx<T> ctx[MAX_SOLVE_BLOCK];
};

// compact the problems of the CTA that need a phase into the shared work list (slot order is kept,
// so that neighbouring lanes mostly work on neighbouring slots); returns their number
template <typename T, typename S>
__device__ __forceinline__ int cta_list_build(bool need, long bound, const S &sv, NodeList<T> &nl, int *my_idx = nullptr)
{
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    const unsigned m = __ballot_sync(FULL, need);
    if (lane == 0) nl.wcnt[warp] = __popc(m);
    __syncthreads();
    int base = 0, n = 0;
    for (int i = 0; i < nw; i++) { int c = nl.wcnt[i]; if (i < warp) base += c; n += c; }
    if (need) {
        const int idx = base + __popc(m & ((1u << lane) - 1u));
        nl.slot[idx] = (int)bound;
        nl.ctx[idx] = sv.node_ctx();
        if (my_idx) *my_idx = idx;
    }
    __syncthreads();
    return n;
}

// The item loops of the CTA-wide phases live in functions of their own (not inlined): each gets its own
// register allocation, so that the spills of one phase do not leak into the others or into the
// per-problem sweeps of the main loop.  The parameters come from constant memory through ConstP<T>,
// which the translation unit defines.  BANK does not change what they compute: it only gives the bank kernels
// instantiations of their own, so that each instantiation keeps a single calling kernel (NVVM then binds the work list
// argument to that kernel's __shared__ NodeList instead of passing a generic pointer) and the other kernels compile as
// they would without the bank.
template <typename T> struct ConstP;

template <typename T, int PHASE, int STRIDE, bool OBCA, bool RSTG, bool BANK>
__device__ __noinline__ void phase_items(T *ws_base, const NodeList<T> *nl, int n, int n_spec)
{
    const DevParams<T> &P = ConstP<T>::get(nl->cslot);
    Ws<T, STRIDE, OBCA, RSTG && PHASE != 3> w; w.init_layout(P.N, P.n_cinf);
    if (RSTG && PHASE != 3) { w.rs = reinterpret_cast<T *>(nl->rstg) + threadIdx.x; w.rs_stride = blockDim.x; }
    if (PHASE == 1 || PHASE == 2) {
        const int total = n * (P.N + 1);
        for (int it = threadIdx.x; it < total; it += blockDim.x) {
            const int j = it % n, k = it / n;
            w.bind(ws_base, nl->slot[j]);
            if (PHASE == 1) node_phase1(P, w, nl->ctx[j], k);
            else node_phase2(P, w, nl->ctx[j], k);
        }
    } else if (PHASE == 3) {                                      // rollouts of the line-search candidates
        for (int it = threadIdx.x; it < n * n_spec; it += blockDim.x) {
            const int q = it % n, j = it / n;
            if (j < P.n_alpha - nl->ctx[q].ls) { w.bind(ws_base, nl->slot[q]); rollout_item(P, w, nl->ctx[q], j); }
        }
    } else {                                                      // rows of the trial points
        const int total = n * n_spec * (P.N + 1);
        for (int it = threadIdx.x; it < total; it += blockDim.x) {
            const int q = it % n, r = it / n, j = r % n_spec, k = r / n_spec;
            if (j < P.n_alpha - nl->ctx[q].ls) { w.bind(ws_base, nl->slot[q]); node_phase3(P, w, nl->ctx[q], k, j); }
        }
    }
}

template <typename T, int PHASE, int STRIDE, bool RSTG, typename S>
__device__ __forceinline__ void node_phase_cta(const DevParams<T> &P, T *ws_base, const WsLayout &L, bool need,
                                               long bound, const S &sv, NodeList<T> &nl)
{
    const int n = cta_list_build(need, bound, sv, nl);
    if (n > 0) phase_items<T, PHASE, STRIDE, S::obca, RSTG, S::bank>(ws_base, &nl, n, 1);
    __syncthreads();
}

#ifdef IGT_PHASE_CLOCKS
__device__ long long g_mid_t;            // debug: end of the rollouts of CTA 0's last trial phase
#define IGT_MID_TICK() do { if (blockIdx.x == 0 && threadIdx.x == 0) g_mid_t = clock64(); } while (0)
#else
#define IGT_MID_TICK() do { } while (0)
#endif

// CTA-wide trial phase with a speculative line search.  The candidates alpha, alpha/2, ... of one
// line search are judged against the same reference point, so they are independent: when fewer
// problems than threads are in their trial phase (the tail of a batch, small batches), the spare
// threads roll out the next halvings at the same time, each into its own iterate buffer, and the
// owner then takes the first candidate that passes -- the same iterate sequential halving reaches,
// in one pass instead of up to n_alpha.  Returns the number of candidates per problem.
#ifndef IGT_SPEC_BUDGET
#define IGT_SPEC_BUDGET IGT_MAX_SOLVE_BLOCK
#endif
template <typename T, int STRIDE, bool RSTG, typename S>
__device__ __forceinline__ int trial_phase_cta(const DevParams<T> &P, T *ws_base, const WsLayout &L, bool need,
                                               long bound, const S &sv, NodeList<T> &nl, bool speculate, int &n_out,
                                               int *my_idx = nullptr)
{
    const int n = cta_list_build(need, bound, sv, nl, my_idx);
    n_out = n;
    if (n == 0) { IGT_MID_TICK(); return 1; }                     // CTA-uniform
    // IGT_SPEC_BUDGET: most candidates (problems x halvings) evaluated at once; the default fills the CTA's threads
    int n_spec = 1;
    if (speculate) { n_spec = IGT_SPEC_BUDGET / n; n_spec = n_spec < 1 ? 1 : (n_spec > P.n_alpha ? P.n_alpha : n_spec); }
    phase_items<T, 3, STRIDE, S::obca, false, S::bank>(ws_base, &nl, n, n_spec);
    __syncthreads();
    IGT_MID_TICK();
    phase_items<T, 4, STRIDE, S::obca, RSTG, S::bank>(ws_base, &nl, n, n_spec);
    __syncthreads();
    return n_spec;
}

// gt_mpc with the tensor-core value term: the terminal values (and derivatives) of all n * n_spec
// line-search candidates of the CTA in one CTA-wide evaluation -- thread t takes candidate t / n of the
// t % n-th listed problem -- left in Tc(candidate buffer, 2..7) for the owner's accept_trials.
// COOP: the same with the exact cooperative evaluation (mlp_coop.cuh) instead of the tensor cores; COOP + BANK: each
// candidate with its problem's network, the index read here from io (not held by the solver loop).
template <typename T, bool COOP, bool BANK, typename WS>
__device__ __forceinline__ void tc_candidates(const DevParams<T> &P, const ProbIO &io, T *ws_base, const WS &wproto,
                                              const NodeList<T> &nl, int n, int n_spec, MlpTcCtx *tc, uint8_t *coop_smem,
                                              int jlo = 0, bool filter = false)
{
    if (n == 0) return;                                            // CTA-uniform
    const int t = threadIdx.x, q = t % n, j = jlo + t / n;
    bool valid = j < n_spec && j < P.n_alpha - nl.ctx[q].ls && (!filter || nl.more[q]);
    WS w = wproto;
    int nb = 0;
    using V = typename std::conditional<COOP, T, float>::type;
    V cx[4] = { V(0), V(0), V(0), V(0) }, o[6], sN = V(0), vN = V(0);
    int net = 0;
    if (valid) {
        w.bind(ws_base, nl.slot[q]);
        nb = cand_buf(nl.ctx[q].cur, j);
        valid = w.Tc(nb, 0) != T(0);                               // the rollout stayed finite
    }
    if (valid) {
        const long p = (nl.ctx[q].x0p - io.x0) / NZ;
#pragma unroll
        for (int i = 0; i < 4; i++) cx[i] = V(io.ctx[p * 4 + i]);
        sN = V(w.Z(nb, P.N, IS)); vN = V(w.Z(nb, P.N, IV));
        if (BANK) net = bank_io<T>(io).net_idx[p];
    }
    if (__syncthreads_or(valid)) {
        if constexpr (COOP && BANK) mlp_coop_eval_bank(bank_io<T>(io).nets, coop_smem, valid, net, sN, vN, cx, o);
        else if constexpr (COOP) mlp_coop_eval(P, coop_smem, valid, sN, vN, cx, o);
        else mlp_tc_eval(*tc, valid, sN, vN, cx, o);
        if (valid) {
#pragma unroll
            for (int i = 0; i < 6; i++) w.Tc(nb, 2 + i) = T(o[i]);
        }
    }
    __syncthreads();
}

// Optional per-phase cycle counters of the first thread of CTA 0 (build with -DIGT_PHASE_CLOCKS;
// tools/phase_clocks.py reads them through igt_debug_phase_clocks).
#ifdef IGT_PHASE_CLOCKS
__device__ long long g_phase_clk[16];
__device__ long long g_round_clk[512];   // per loop pass of CTA 0: cycles, and the number of its active problems
__device__ int g_round_n[512];
__device__ int g_round_ph[512][12];      // per loop pass: kcycles per phase
__device__ long long g_cta_clk[512];     // per CTA: cycles from its start to its exit, and its loop passes
__device__ int g_cta_rounds[512];
__device__ int g_round_mx[512][4];       // per loop pass, max over CTA 0's threads: adjoint, Riccati (all retries), step bound kcycles; Riccati sweeps
#define IGT_TICK(i) do { if (clk_on) { long long t_ = clock64(); clk[i] += t_ - clk_t; if (round_i < 512) g_round_ph[round_i][i] += (int)((t_ - clk_t) >> 10); clk_t = t_; } } while (0)
#else
#define IGT_TICK(i) do { } while (0)
#endif

// BANK: gt_mpc with the handle's network bank, each problem with network io.net_idx[p] (per-thread or, with COOP,
// cooperative value term; not with TC)
template <typename T, bool TC, int STRIDE = 32, bool OBCA = false, bool COOP = false, bool RSTG = false, bool BANK = false>
__device__ __forceinline__ void solve_persistent(const DevParams<T> &P, const ProbIO &io, T *ws_base,
                                                 long slot, long B, const Sched &sc,
                                                 const double *guess, T *mlp_scratch, int mlp_width, MlpTcCtx *tc,
                                                 int quota, int cslot, uint8_t *coop_smem = nullptr, void *rstg_smem = nullptr)
{
    __shared__ NodeList<T> nl;
    if (threadIdx.x == 0) { nl.cslot = cslot; nl.rstg = rstg_smem; }   // (the first CTA barrier of the loop publishes them)
    static_assert(!(TC && BANK), "the tensor-core value term holds one network");
    Solver<T, Ws<T, STRIDE, OBCA>, BANK> sv(P);
    sv.w.init_layout(P.N, P.n_cinf);
    sv.w.bind(ws_base, slot);
    sv.mlp_scratch = mlp_scratch; sv.mlp_width = mlp_width;
    const unsigned FULL = 0xffffffffu;
    // only the first `quota` threads of a CTA fetch fresh problems, so that a batch smaller than the
    // machine is spread over all SMs; the other threads still work in the CTA-wide phases
    bool active = false, exhausted = (int)threadIdx.x >= quota;
    long p = -1;
    const long bound = slot;
    if (TC) sv.phi_noise = T(3e-7);
    constexpr bool CTA_MLP = TC || COOP;                          // value term evaluated CTA-wide at the two uniform points below
#ifdef IGT_PHASE_CLOCKS
    const bool clk_on = blockIdx.x == 0 && threadIdx.x == 0;
    long long clk[16] = { 0 }, clk_t = clock64(), round_t = clk_t;
    const long long cta_t0 = clk_t;
    int round_i = 0, cta_rounds = 0;
    if (clk_on) for (int i = 0; i < 12; i++) g_round_ph[0][i] = 0;
#endif
    // All warps of the CTA (one CTA per SM) walk the phases together -- scheduling, backward
    // sweeps, forward trial -- separated by CTA barriers, so that the SM's instruction cache
    // holds one phase's loop body at a time instead of eight warps' worth of different code.
    for (;;) {
        // ---- phase 0: scheduling (fetch fresh problems, park / adopt stragglers) ----
        bool fresh = false;
        if (!active && !exhausted) {
            p = (long)atomicAdd(sc.counter, 1ULL);
            if (p >= B) exhausted = true;
            else {
                const bool warm = io.u_init && (!io.warm || io.warm[p]);
                const double *u_src = (warm ? io.u_init : guess) + p * P.N * 2;
                if (sv.init(io, p, io.ctx != nullptr, u_src, warm)) {
                    if (!CTA_MLP) sv.terminal_of(sv.cur, sv.tcur, true);
                    active = true;
                    fresh = true;
                } else {
                    sv.write_out(io, p);
                }
            }
        }
        if (TC) {
            if (__syncthreads_or(fresh)) {
                float cx[4] = { float(sv.ctx[0]), float(sv.ctx[1]), float(sv.ctx[2]), float(sv.ctx[3]) }, o[6];
                float sN = fresh ? float(sv.w.Z(sv.cur, P.N, IS)) : 0.f, vN = fresh ? float(sv.w.Z(sv.cur, P.N, IV)) : 0.f;
                mlp_tc_eval(*tc, fresh, sN, vN, cx, o);
                if (fresh) term_from_tc(o, sv.tcur);
            }
        }
        if (COOP) {
            const bool want = fresh && sv.gt;
            if (__syncthreads_or(want)) {
                T o[6];
                const T sN = want ? sv.w.Z(sv.cur, P.N, IS) : T(0), vN = want ? sv.w.Z(sv.cur, P.N, IV) : T(0);
                if constexpr (BANK) mlp_coop_eval_bank(bank_io<T>(io).nets, coop_smem, want, want ? bank_io<T>(io).net_idx[p] : 0, sN, vN, sv.ctx, o);
                else mlp_coop_eval(P, coop_smem, want, sN, vN, sv.ctx, o);
                if (want) { sv.tcur.V = o[0]; sv.tcur.gs = o[1]; sv.tcur.gv = o[2]; sv.tcur.Hss = o[3]; sv.tcur.Hsv = o[4]; sv.tcur.Hvv = o[5]; }
            }
        }
        // a warp is finished once its lanes can fetch no more and none of them is busy
        const bool wants_exit = __all_sync(FULL, exhausted && !active);
#ifdef IGT_PHASE_CLOCKS
        cta_rounds++;
        const int cta_busy = __syncthreads_count(active);
        if (clk_on && round_i < 512) {
            long long t_ = clock64();
            g_round_clk[round_i] = t_ - round_t; g_round_n[round_i] = cta_busy; round_t = t_; round_i++;
            if (round_i < 512) for (int i = 0; i < 12; i++) g_round_ph[round_i][i] = 0;
        }
#else
        const int cta_busy = __syncthreads_or(active);
#endif
        if (__syncthreads_and(wants_exit)) break;
        if (!cta_busy) { IGT_TICK(9); continue; }               // (only while other warps still fetch)
        IGT_TICK(0);
        // ---- phase 1: backward pass = CTA-wide node phases between the per-problem sweeps ----
        const bool back = active && sv.need_back;
        node_phase_cta<T, 1, STRIDE, RSTG>(P, ws_base, sv.w.L, back && sv.need_back == 2, bound, sv, nl);
        IGT_TICK(1);
#ifdef IGT_PHASE_CLOCKS
        __shared__ int s_round_i;
        if (clk_on) s_round_i = round_i;
        __syncthreads();
        const int rnd_ = s_round_i;
        const long long ta_ = clock64();
#endif
        const bool p2 = back && sv.backward_pre();              // adjoint sweep, convergence test, barrier update
#ifdef IGT_PHASE_CLOCKS
        if (blockIdx.x == 0 && back && rnd_ < 512) atomicMax(&g_round_mx[rnd_][0], (int)((clock64() - ta_) >> 10));
#endif
        IGT_TICK(2);
        node_phase_cta<T, 2, STRIDE, RSTG>(P, ws_base, sv.w.L, p2, bound, sv, nl);
        IGT_TICK(3);
        if (back && !sv.done) {                                  // Riccati sweep, step bound
#ifdef IGT_PHASE_CLOCKS
            const long long tr_ = clock64();
            int nsw_ = 0;
            for (;;) {
                nsw_++;
                if (sv.riccati_sweep()) break;
                sv.reg = fmax(fmax(sv.reg * P.reg_up, P.reg_min), sv.reg_hint);
                if (sv.reg > P.reg_max) { sv.status = sv.acceptable() ? 6 : 3; sv.done = true; break; }
            }
            const long long ts_ = clock64();
            IGT_TICK(4);
            if (!sv.done) { sv.need_back = 0; sv.ls = 0; sv.step_bound(); }
            if (blockIdx.x == 0 && rnd_ < 512) {
                atomicMax(&g_round_mx[rnd_][1], (int)((ts_ - tr_) >> 10));
                atomicMax(&g_round_mx[rnd_][2], (int)((clock64() - ts_) >> 10));
                atomicMax(&g_round_mx[rnd_][3], nsw_);
            }
            IGT_TICK(5);
#else
            sv.backward_post();
#endif
        }
        __syncthreads();
        IGT_TICK(6);
        // ---- phase 2: one forward trial + acceptance ----
        const bool trying = active && !sv.done;
        int n_try = 0;
        int my_idx = 0;                                          // this owner's position in the trial phase's list
        const int n_spec = trial_phase_cta<T, STRIDE, RSTG>(P, ws_base, sv.w.L, trying, bound, sv, nl, true, n_try, &my_idx);
#ifdef IGT_PHASE_CLOCKS
        if (clk_on) { long long m_ = g_mid_t; clk[7] += m_ - clk_t; if (round_i < 512) g_round_ph[round_i][7] += (int)((m_ - clk_t) >> 10); clk_t = m_; }
#endif
        IGT_TICK(11);
        if (CTA_MLP) {
            // Value terms CTA-wide, lazily: first every problem's first candidate (the one sequential halving tries
            // first, accepted nine times out of ten); the speculative candidates only of the problems whose first
            // was rejected.  Same candidates judged in the same order: same iterates.
            const int left = P.n_alpha - sv.ls, nj = n_spec < left ? n_spec : left;
            tc_candidates<T, COOP, BANK>(P, io, ws_base, sv.w, nl, n_try, 1, tc, coop_smem);
            int tried = 0, jacc = -1;
            if (trying) jacc = sv.judge_trials(0, 1, true, tried);
            const bool more = trying && jacc < 0 && nj > 1;
            if (trying) nl.more[my_idx] = more ? 1 : 0;
            if (__syncthreads_or(more)) {
                // candidates 1 .. n_spec-1: (n_spec - 1) n <= blockDim.x requests, one pass
                tc_candidates<T, COOP, BANK>(P, io, ws_base, sv.w, nl, n_try, n_spec, tc, coop_smem, 1, true);
                if (more) jacc = sv.judge_trials(1, nj, true, tried);
            }
            if (trying) sv.finish_trials(jacc, tried);
        } else if (trying) {
            const int left = P.n_alpha - sv.ls;
            sv.accept_trials(n_spec < left ? n_spec : left, false);
        }
        IGT_TICK(8);
        if (active && sv.done) { sv.write_out(io, p); active = false; }
        IGT_TICK(10);
    }
#ifdef IGT_PHASE_CLOCKS
    if (threadIdx.x == 0 && blockIdx.x < 512) { g_cta_clk[blockIdx.x] = clock64() - cta_t0; g_cta_rounds[blockIdx.x] = cta_rounds; }
    if (clk_on) {
        for (int i = 0; i < 16; i++) g_phase_clk[i] = clk[i];
        for (int i = round_i; i < 512; i++) { g_round_clk[i] = 0; g_round_n[i] = -1; }
    }
#endif
}
#endif

}  // namespace igt
