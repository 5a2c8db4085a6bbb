// igt_abi.cu -- kernels and the extern "C" boundary of libigtmpc.so (see include/igt_mpc.h).
//
// Kernels (all hand-written, sm_100a):
//   solve_kernel<T>       one MPC problem per thread, whole interior-point iLQR on chip + SoA
//                         workspace in HBM (solver_core.cuh); replaces mpc.py:383-406
//   rollout_kernel        fp32 Frenet RK4 rollout + analytic Jacobians (compensated state
//                         accumulation); replaces kinematic_bicycle_model_frenet.py:69-185
//   rollout_euler_kernel  fp32 Cartesian Euler rollout + Jacobians; kinematic_bicycle_model.py:15-50
//   eval_kernel           fp64 cost / max-row-violation of given controls; mpc.py:177-373
//   vjp_kernel            fp64 vector-Jacobian product of a solve through its converged KKT system (sens.cuh)
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <new>
#include <mutex>
#include <atomic>
#include <algorithm>

#include "../../include/igt_mpc.h"
#include "solver_core.cuh"
#include "sens.cuh"
#include "params_host.hpp"
#include "mlp_tc.cuh"

using namespace igt;

// resident solver threads per SM: one CTA of SOLVE_BLOCK threads (255 registers/thread -> 256 threads)
#ifndef SOLVE_BLOCK
#define SOLVE_BLOCK 256
#endif
#define SLOTS_PER_SM SOLVE_BLOCK

// ------------------------------------------------------------------ device constants ----
// Solver parameters live in constant memory, N_CSLOTS copies per precision: every handle owns a slot (handles
// beyond N_CSLOTS per device share one, ordered by events -- see acquire_cslot), kernels get the slot index as an
// argument, and a slot is uploaded only when its content changes.  Handles with different horizons, limits or value
// networks can therefore run concurrently on different streams.
constexpr int N_CSLOTS = 8;
__constant__ DevParams<float> c_Pf[N_CSLOTS];
__constant__ DevParams<double> c_Pd[N_CSLOTS];
static_assert(N_CSLOTS * (sizeof(DevParams<float>) + sizeof(DevParams<double>)) <= 60 * 1024, "constant memory budget");

template <> struct igt::ConstP<float> { static __device__ __forceinline__ const DevParams<float> &get(int s) { return c_Pf[s]; } };
template <> struct igt::ConstP<double> { static __device__ __forceinline__ const DevParams<double> &get(int s) { return c_Pd[s]; } };
#include "episode.cuh"

// ------------------------------------------------------------------ kernels -------------
// cold-start guess: best of five tracking-controller rollouts per problem -> guess[B][N][2]
template <typename T, bool OBCA>
__global__ void __launch_bounds__(128) guess_kernel(ProbIO io, long B, double *guess, int cs)
{
    long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    if (io.u_init && (!io.warm || io.warm[p])) return;            // warm-started problem: no cold-start guess needed
    const DevParams<T> &P = ConstP<T>::get(cs);
    Solver<T, Ws<T, 32, OBCA>> sv(P);
    sv.compute_guess(io, p, guess + p * P.N * 2);
}

#ifndef IGT_RSTG
#define IGT_RSTG 1     // row staging in the node phases of the plain throughput kernels (solver_core.cuh, Ws RSTG)
#endif
// BANK: gt_mpc with the handle's network bank, network io.net_idx[p] per problem (not with TC)
// DUALS: io is a DualsIO, and every problem also writes the final slack and multiplier of each row
template <typename T, bool BANK, bool DUALS>
using SolveIO = typename std::conditional<DUALS, DualsIO<typename std::conditional<BANK, ProbIONet<T>, ProbIO>::type>,
                                          typename std::conditional<BANK, ProbIONet<T>, ProbIO>::type>::type;
template <typename T, bool TC, bool OBCA, bool COOP = false, bool BANK = false, bool DUALS = false>
__global__ void __launch_bounds__(SOLVE_BLOCK, 1) solve_kernel(SolveIO<T, BANK, DUALS> io, T *ws, long n_slots, long B, Sched sc,
                                                               const double *guess, T *mlp_scratch, int mlp_width,
                                                               MlpTcWeights wt, int quota, int cs)
{
    extern __shared__ __align__(16) uint8_t dyn_smem[];
    long slot = (long)blockIdx.x * blockDim.x + threadIdx.x;   // grid is sized to n_slots exactly
    const DevParams<T> &P = ConstP<T>::get(cs);
    MlpTcCtx tc;
    if (TC) mlp_tc_setup(tc, dyn_smem, wt);
    constexpr bool RSTG = IGT_RSTG && !TC && !COOP;                 // (TC fills shared memory itself; with COOP the value term's
                                                                    //  weight reads need the L1 more: measured 120 -> 146 ms per batch)
    // dynamic shared memory: [cooperative value-term buffers (COOP)] [row staging (RSTG)]
    solve_persistent<T, TC, 32, OBCA, COOP, RSTG, BANK, DUALS>(P, io, ws, slot, B, sc, guess,
                            mlp_scratch ? mlp_scratch + slot * 12 * (long)mlp_width : nullptr, mlp_width, &tc, quota, cs, dyn_smem,
                            RSTG ? dyn_smem + (COOP ? mlp_coop_smem_bytes<T>(SOLVE_BLOCK) : 0) : nullptr);
    if (TC) mlp_tc_teardown(tc);
}

// Latency path for batches of at most one problem per SM (the closed-loop step: B = 2): one CTA per problem,
// its whole workspace in shared memory (stride-1 layout), so the sweeps of the problem's one owner thread run at
// shared-memory latency instead of an L2 round trip per stage; the node phases and the line-search candidates
// are dealt out over the CTA's 256 threads as in the throughput kernel.  Same code, same arithmetic, same results.
// GT: gt_mpc, with the value term evaluated by the CTA (COOP: exact cooperative evaluation, its buffers sized for one
// problem's requests and placed before the workspace) or by the owner thread (its [2][6][width] scratch slab in global
// memory, one per CTA); BANK: the network bank, as in solve_kernel.  The tensor-core value term is not offered here.
template <typename IO, typename T>
struct SmallIO : IO {                                     // inputs of a gt_mpc latency solve: IO and the per-thread scratch
    T *mlp_scratch = nullptr;                             // [grid][2][6][mlp_width], null with COOP
    int mlp_width = 0;
};
// (rounded up to 16 bytes: the workspace that follows keeps the alignment of the start of dynamic shared memory, which
// the shared solver functions are compiled for)
template <typename T, bool COOP, bool BANK>
constexpr int small_coop_bytes()
{
    return COOP ? ((BANK ? mlp_coop_bank_smem_bytes<T, COOP_CAP>(SOLVE_BLOCK) : mlp_coop_smem_bytes<T, COOP_CAP>(SOLVE_BLOCK)) + 15) & ~15 : 0;
}
template <typename T, bool OBCA, bool COOP = false, bool BANK = false, bool GT = COOP || BANK>
__global__ void __launch_bounds__(SOLVE_BLOCK, 1) solve_small_kernel(
    typename std::conditional<GT, SmallIO<typename std::conditional<BANK, ProbIONet<T>, ProbIO>::type, T>, ProbIO>::type io,
    long B, Sched sc, const double *guess, int cs)
{
    extern __shared__ __align__(16) uint8_t dyn_smem[];
    const DevParams<T> &P = ConstP<T>::get(cs);
    if constexpr (GT) {
        constexpr int off = small_coop_bytes<T, COOP, BANK>();   // dynamic shared memory: [value term (COOP)] [workspace]
        T *scr = io.mlp_scratch ? io.mlp_scratch + (long)blockIdx.x * 12 * io.mlp_width : nullptr;
        solve_persistent<T, false, 1, OBCA, COOP, false, BANK>(P, io, reinterpret_cast<T *>(dyn_smem + off), 0, B, sc, guess, scr,
                                                               io.mlp_width, nullptr, 1, cs, dyn_smem);
    } else {
        solve_persistent<T, false, 1, OBCA>(P, io, reinterpret_cast<T *>(dyn_smem), 0, B, sc, guess, (T *)nullptr, 0, nullptr, 1, cs);
    }
}

// fp32 rollout with Kahan-compensated accumulation of the RK4 increments (x, y, s reach ~50 m
// while one sub-step adds ~0.1 m; plain fp32 accumulation loses the 1e-5 target on ~0.5 % of
// rollouts, SURVEY 7 item 4).  One problem per thread; outputs are AoS as the ABI promises.
__global__ void __launch_bounds__(128) rollout_kernel(int B, const float *__restrict__ z0,
                                                      const float *__restrict__ U,
                                                      const float *__restrict__ curv_, float *__restrict__ Z,
                                                      float *__restrict__ A, float *__restrict__ Bm, int cs)
{
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    const DevParams<float> &P = c_Pf[cs];
    const int N = P.N;
    float z[NZ], comp[NZ], curv[3] = { curv_[3 * p], curv_[3 * p + 1], curv_[3 * p + 2] };
#pragma unroll
    for (int i = 0; i < NZ; i++) { z[i] = z0[(long)p * NZ + i]; comp[i] = 0.f; Z[(long)p * (N + 1) * NZ + i] = z[i]; }
    const float h = P.h;
    for (int k = 0; k < N; k++) {
        float u[2] = { U[((long)p * N + k) * 2], U[((long)p * N + k) * 2 + 1] };
        if (A) {
            float zn[NZ], Sc[NSENS], S[NZ][NSEED];
            rk4_step_sens(P, z, u, curv, zn, Sc);
            expand_sens(P, Sc, S);
            float *Ak = A + ((long)p * N + k) * NZ * NZ, *Bk = Bm + ((long)p * N + k) * NZ * 2;
#pragma unroll
            for (int i = 0; i < NZ; i++) {
#pragma unroll
                for (int j = 0; j < NZ; j++) Ak[i * NZ + j] = (i == j && j < 3) ? 1.f : 0.f;
                Ak[i * NZ + IEY] = S[i][0]; Ak[i * NZ + IEPSI] = S[i][1]; Ak[i * NZ + IV] = S[i][2]; Ak[i * NZ + IPSI] = S[i][3];
                Bk[i * 2] = S[i][4]; Bk[i * 2 + 1] = S[i][5];
            }
        }
        // compensated value step: the same stage derivatives as rk4_core, Kahan-summed increments.  The pw_const branch
        // of every evaluation (mpc.py:199: K steps at s = b0, b1) is decided in DOUBLE from the compensated arc length
        // (z - comp is the running sum to about fp64 accuracy): in plain fp32 a stage state within 5e-5 m of a break-point
        // takes the other branch than the fp64 reference (0.1 % of rollouts missed the 1e-5 target in round 1).
        const StepK<float> c = step_setup(P, z, u, curv);
        const double b0d = curv[0], b1d = curv[1];
        auto Kof = [&](double sd) { return (sd >= b0d ? curv[2] : 0.f) - (sd >= b1d ? curv[2] : 0.f); };
        for (int it = 0; it < P.n_rk; it++) {
            Deriv<float> k1, k2, k3, k4;
            RhsJac<float> J;
            const float hh = 0.5f * h;
            const double sd = (double)z[IS] - (double)comp[IS];
            stage_deriv<float, false, true>(c, z[IS], z[IEY], z[IEPSI], z[IV], z[IPSI], k1, J, Kof(sd));
            stage_deriv<float, false, true>(c, z[IS] + hh * k1.s, z[IEY] + hh * k1.ey, z[IEPSI] + hh * k1.ep, z[IV] + hh * u[0],
                                            z[IPSI] + hh * k1.ps, k2, J, Kof(sd + (double)hh * (double)k1.s));
            stage_deriv<float, false, true>(c, z[IS] + hh * k2.s, z[IEY] + hh * k2.ey, z[IEPSI] + hh * k2.ep, z[IV] + hh * u[0],
                                            z[IPSI] + hh * k2.ps, k3, J, Kof(sd + (double)hh * (double)k2.s));
            stage_deriv<float, false, true>(c, z[IS] + h * k3.s, z[IEY] + h * k3.ey, z[IEPSI] + h * k3.ep, z[IV] + h * u[0],
                                            z[IPSI] + hh * k3.ps, k4, J, Kof(sd + (double)h * (double)k3.s));      // psi + h/2 k3: the reference's k4 quirk
            float inc[NZ];
            inc[IX] = h / 6.f * (k1.x + 2.f * k2.x + 2.f * k3.x + k4.x);
            inc[IY] = h / 6.f * (k1.y + 2.f * k2.y + 2.f * k3.y + k4.y);
            inc[IS] = h / 6.f * (k1.s + 2.f * k2.s + 2.f * k3.s + k4.s);
            inc[IEY] = h / 6.f * (k1.ey + 2.f * k2.ey + 2.f * k3.ey + k4.ey);
            inc[IEPSI] = h / 6.f * (k1.ep + 2.f * k2.ep + 2.f * k3.ep + k4.ep);
            inc[IV] = h * u[0];
            inc[IPSI] = h / 6.f * (k1.ps + 2.f * k2.ps + 2.f * k3.ps + k4.ps);
#pragma unroll
            for (int i = 0; i < NZ; i++) {
                float y = inc[i] - comp[i];
                float t = z[i] + y;
                comp[i] = (t - z[i]) - y;
                z[i] = t;
            }
        }
#pragma unroll
        for (int i = 0; i < NZ; i++) Z[((long)p * (N + 1) + k + 1) * NZ + i] = z[i];
    }
}

__global__ void __launch_bounds__(128) rollout_euler_kernel(int B, const float *__restrict__ z0,
                                                            const float *__restrict__ U, float *__restrict__ Z,
                                                            float *__restrict__ A, float *__restrict__ Bm, int cs)
{
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    const DevParams<float> &P = c_Pf[cs];
    const int N = P.N;
    float z[4];
    for (int i = 0; i < 4; i++) { z[i] = z0[(long)p * 4 + i]; Z[(long)p * (N + 1) * 4 + i] = z[i]; }
    for (int k = 0; k < N; k++) {
        float u[2] = { U[((long)p * N + k) * 2], U[((long)p * N + k) * 2 + 1] }, zn[4];
        euler_step(P, z, u, zn, A ? A + ((long)p * N + k) * 16 : nullptr, A ? Bm + ((long)p * N + k) * 8 : nullptr);
        for (int i = 0; i < 4; i++) { z[i] = zn[i]; Z[((long)p * (N + 1) + k + 1) * 4 + i] = zn[i]; }
    }
}

// largest row so far.  Unlike fmax, which drops a NaN operand, a NaN row wins and then stays: controls that drive the
// state non-finite must not come back with the violation of the rows before the NaN
__device__ __forceinline__ double row_max(double m, double r) { return (r > m || r != r) ? r : m; }

// fp64 re-roll + cost + max inequality row (reference units) of given controls; BANK: value term of network
// net_idx[p] of the bank (indices checked by the host)
template <bool BANK>
__global__ void __launch_bounds__(128) eval_kernel(long B, const double *__restrict__ x0_, const double *__restrict__ uprev_,
                                                   const double *__restrict__ curv_, const double *__restrict__ obs_,
                                                   const double *__restrict__ ctx_, const double *__restrict__ U,
                                                   double *__restrict__ cost, double *__restrict__ viol,
                                                   double *__restrict__ Zout, double *mlp_scratch, int mlp_width, int cs,
                                                   const double *__restrict__ obs_psi_, const int *__restrict__ net_idx,
                                                   const MlpNet<double> *nets)
{
    long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    const DevParams<double> &P = c_Pd[cs];
    const int N = P.N;
    double z[NZ], curv[3] = { curv_[3 * p], curv_[3 * p + 1], curv_[3 * p + 2] };
    double up[2] = { uprev_[2 * p], uprev_[2 * p + 1] };
    for (int i = 0; i < NZ; i++) z[i] = x0_[p * NZ + i];
    double s0 = z[IS], J = 0, su = 0, m = 0;
    const double *obs = obs_ + p * (N + 1) * 2;
    for (int k = 0; k <= N; k++) {
        if (Zout) for (int i = 0; i < NZ; i++) Zout[(p * (N + 1) + k) * NZ + i] = z[i];
        J += z[IEPSI] * z[IEPSI] + z[IEY] * z[IEY];
        m = row_max(m, fabs(z[IEY]) - P.ey_lim);
        if (k >= 1) {
            if (obs_psi_) {                                      // OBCA rows in dual-eliminated form (obca.cuh)
                double gd[3];
                m = row_max(m, P.d_min + OBCA_MARGIN - obca_rect_sdist(z[IX], z[IY], z[IPSI], obs[2 * k], obs[2 * k + 1], obs_psi_[p * (N + 1) + k], gd));
            } else {
                double dx = z[IX] - obs[2 * k], dy = z[IY] - obs[2 * k + 1];
                m = row_max(m, P.d_min * P.d_min - dx * dx - dy * dy);
            }
        }
        if (k == N) break;
        double u[2] = { U[(p * N + k) * 2], U[(p * N + k) * 2 + 1] };
        su += u[0] * u[0] + u[1] * u[1];
        m = row_max(m, row_max(P.v_min - z[IV], z[IV] - P.v_max));
        m = row_max(m, row_max(P.a_min - u[0], u[0] - P.a_max));
        m = row_max(m, fabs(u[1]) - P.df_max);
        m = row_max(m, fabs(u[0] - up[0]) - P.da_max);
        m = row_max(m, fabs(u[1] - up[1]) - P.ddf_max);
        if (k == N - 1)
            for (int q = 0; q < P.n_cinf; q++) m = row_max(m, P.cinf_A[q][0] * z[IV] + P.cinf_A[q][1] * u[0] - P.cinf_b[q]);
        double zn[NZ];
        rk4_step(P, z, u, curv, zn);
        for (int i = 0; i < NZ; i++) z[i] = zn[i];
        up[0] = u[0]; up[1] = u[1];
    }
    J += P.w_u * su;
    if (ctx_) {
        TermVal<double> t;
        double ctx[4] = { ctx_[4 * p], ctx_[4 * p + 1], ctx_[4 * p + 2], ctx_[4 * p + 3] };
        double *sc = mlp_scratch + p * 12 * (long)mlp_width;
        if (BANK) mlp_eval_thread_net(nets[net_idx[p]], z[IS], z[IV], ctx, sc, sc + 6 * mlp_width, mlp_width, t, false);
        else mlp_eval_thread(P, z[IS], z[IV], ctx, sc, sc + 6 * mlp_width, mlp_width, t, false);
        J -= t.V;
    } else {
        J -= z[IS] - s0;
    }
    cost[p] = J;
    viol[p] = m;
}

// standalone evaluation of the gt_mpc value term (value + tangents in (s_N, v_N)) for B problems:
// tensor-core path (one CTA = 256 problems per pass) and the fp64 CUDA-core path it is checked against
__global__ void __launch_bounds__(256, 1) mlp_tc_kernel(MlpTcWeights wt, long B, const double *sN, const double *vN,
                                                        const double *ctx, double *out)
{
    extern __shared__ uint8_t dyn_smem[];
    MlpTcCtx c;
    mlp_tc_setup(c, dyn_smem, wt);
    for (long base = (long)blockIdx.x * 256; base < B; base += (long)gridDim.x * 256) {
        long p = base + threadIdx.x;
        bool valid = p < B;
        float cx[4] = { 0.f, 0.f, 0.f, 0.f }, o[6];
        float s = 0.f, v = 0.f;
        if (valid) { s = (float)sN[p]; v = (float)vN[p]; for (int i = 0; i < 4; i++) cx[i] = (float)ctx[4 * p + i]; }
        mlp_tc_eval(c, valid, s, v, cx, o);
        if (valid) for (int i = 0; i < 6; i++) out[6 * p + i] = (double)o[i];
    }
    mlp_tc_teardown(c);
}

template <bool BANK>
__global__ void __launch_bounds__(128) mlp_ref_kernel(long B, const double *sN, const double *vN, const double *ctx,
                                                      double *out, double *scratch, int width, int cs, const int *net_idx,
                                                      const MlpNet<double> *nets)
{
    long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    const DevParams<double> &P = c_Pd[cs];
    TermVal<double> t;
    double cx[4] = { ctx[4 * p], ctx[4 * p + 1], ctx[4 * p + 2], ctx[4 * p + 3] };
    double *sc = scratch + p * 12 * (long)width;
    if (BANK) mlp_eval_thread_net(nets[net_idx[p]], sN[p], vN[p], cx, sc, sc + 6 * width, width, t, true);
    else mlp_eval_thread(P, sN[p], vN[p], cx, sc, sc + 6 * width, width, t, true);
    out[6 * p] = t.V; out[6 * p + 1] = t.gs; out[6 * p + 2] = t.gv; out[6 * p + 3] = t.Hss; out[6 * p + 4] = t.Hsv; out[6 * p + 5] = t.Hvv;
}

// the exact cooperative evaluation (mlp_coop.cuh) standalone: one CTA pass per 256 problems; BANK: network net_idx[p]
template <bool BANK>
__global__ void __launch_bounds__(256, 1) mlp_coop_kernel(long B, const double *sN, const double *vN, const double *ctx,
                                                          double *out, int cs, const int *net_idx, const MlpNet<double> *nets)
{
    extern __shared__ __align__(16) uint8_t dyn_smem[];
    const DevParams<double> &P = c_Pd[cs];
    for (long base = (long)blockIdx.x * 256; base < B; base += (long)gridDim.x * 256) {
        const long p = base + threadIdx.x;
        const bool valid = p < B;
        double cx[4] = { 0, 0, 0, 0 }, o[6], s = 0, v = 0;
        int net = 0;
        if (valid) { s = sN[p]; v = vN[p]; for (int i = 0; i < 4; i++) cx[i] = ctx[4 * p + i]; if (BANK) net = net_idx[p]; }
        if (BANK) mlp_coop_eval_bank(nets, dyn_smem, valid, net, s, v, cx, o);
        else mlp_coop_eval(P, dyn_smem, valid, s, v, cx, o);
        if (valid) for (int i = 0; i < 6; i++) out[6 * p + i] = o[i];
    }
}

// VJP of a solve (sens.cuh), one problem per thread; ws: [sens_ws_size(N)][B] (element-major, so that a warp's 32
// problems touch consecutive words); mlp_scratch: [B][2][6][mlp_width] (gt_mpc)
template <bool BANK>
__global__ void __launch_bounds__(128) vjp_kernel(SensIO io, long B, double *ws, double *mlp_scratch, int mlp_width, int cs)
{
    const long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    const DevParams<double> &P = c_Pd[cs];
    const SensWs w = { ws + p, B, P.N };
    vjp_problem<BANK>(P, io, p, w, mlp_scratch ? mlp_scratch + p * 12 * (long)mlp_width : nullptr, mlp_width);
}

// dependent-free FMA chains: the CUDA-core roofline denominator that MEASURED_PEAKS.json lacks
template <typename T>
__global__ void __launch_bounds__(256) fma_peak_kernel(T *out, int iters)
{
    T a0 = T(threadIdx.x) * T(1e-3), a1 = a0 + T(1), a2 = a0 + T(2), a3 = a0 + T(3);
    T a4 = a0 + T(4), a5 = a0 + T(5), a6 = a0 + T(6), a7 = a0 + T(7);
    const T m = T(0.999999), c = T(1e-6);
    for (int i = 0; i < iters; i++) {
        a0 = a0 * m + c; a1 = a1 * m + c; a2 = a2 * m + c; a3 = a3 * m + c;
        a4 = a4 * m + c; a5 = a5 * m + c; a6 = a6 * m + c; a7 = a7 * m + c;
    }
    out[(long)blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// ------------------------------------------------------------------ handle --------------
struct igt_handle {
    igt_params prm;
    DevParams<float> Pf;
    DevParams<double> Pd;
    MlpTcWeights tc = {};              // tensor-core copy of the value network (6-128-128-1 only)
    int use_tc = 0;                    // igt_set_option("tensor_core_mlp", 1): fp32-accurate tcgen05 value term (6-128-128-1 nets)
    int use_small = 1;                 // igt_set_option("latency_path", 0) keeps small batches on the throughput kernel
    // network bank (igt_set_mlp_at): slot 0 is also the network of the calls without net_idx (Pf / Pd, tc); a solve
    // with net_idx reads the device table `bank` = [MAX_MLP_NETS] MlpNet<double>, then [MAX_MLP_NETS] MlpNet<float>
    void *mlp_buf[MAX_MLP_NETS] = {};  // device image of each slot: its weights in both precisions (+ the tensor-core copy)
    MlpNet<double> netd[MAX_MLP_NETS] = {};
    MlpNet<float> netf[MAX_MLP_NETS] = {};
    int net_width[MAX_MLP_NETS] = {};  // widest layer of each slot, 0 = empty
    void *bank = nullptr;
    void *ws = nullptr; size_t ws_bytes = 0;
    void *mlp_scratch = nullptr; size_t mlp_scratch_bytes = 0;
    void *stage = nullptr; size_t stage_bytes = 0;     // device block of the *_host calls (see staged)
    void *guess = nullptr; size_t guess_bytes = 0;     // cold-start controls [B][N][2] + the work counter
    void *sens = nullptr; size_t sens_bytes = 0;       // VJP scratch (vjp_kernel)
    int n_sm = 0;
    int smem_optin = 0;                // shared memory a block may opt in to (the gt_mpc latency path's limit)
    long long launches = 0;
    std::string err;
    int device = 0;
    // concurrency (see the header): calls on one handle are serialised on the device in call order whatever their
    // streams -- the handle's workspace, guess buffer and work counter are shared by its calls
    std::mutex mu;                     // host-side: one call at a time per handle
    cudaStream_t hstream = nullptr;    // the *_host entry points run on a private non-blocking stream
    void *pin = nullptr; size_t pin_bytes = 0;   // pinned staging block of the *_host calls (small batches)
    cudaEvent_t last_use = nullptr;    // recorded after the last kernel of every call
    cudaStream_t last_stream = nullptr;
    bool used = false;
    unsigned long long version[2] = { 1, 1 };   // bumped when Pf / Pd change (igt_set_mlp)
    int cslot[2] = { -1, -1 };
};

// constant-memory slot table, per device and precision (0 = f32, 1 = f64)
struct CSlot { const igt_handle *owner = nullptr; unsigned long long version = 0; cudaEvent_t ev = nullptr; };
constexpr int MAX_DEV = 16;
static std::mutex g_slot_mu;
static CSlot g_slots[MAX_DEV][2][N_CSLOTS];
static unsigned g_slot_rr[MAX_DEV][2];

static std::string g_create_err;
static_assert(IGT_MAX_MLP_NETS == MAX_MLP_NETS, "bank size");

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            h->err = std::string(#call) + ": " + cudaGetErrorString(_e);                           \
            return IGT_ECUDA;                                                                      \
        }                                                                                          \
    } while (0)

// (re)allocation is stream-ordered: the old buffer is released after the work already queued on `st` (which, by
// begin_call, includes every earlier call on this handle), the new one is usable by work queued on `st` afterwards
static int grow(igt_handle *h, void **buf, size_t *have, size_t need, cudaStream_t st)
{
    if (*have >= need) return IGT_OK;
    if (*buf) { CK(cudaFreeAsync(*buf, st)); *buf = nullptr; *have = 0; }
    CK(cudaMallocAsync(buf, need, st));
    *have = need;
    return IGT_OK;
}

// Entry of every call that queues device work for a handle: select its device and order the call after the
// handle's previous call if that one went to a different stream.
static int begin_call(igt_handle *h, cudaStream_t st)
{
    CK(cudaSetDevice(h->device));
    if (!h->last_use) CK(cudaEventCreateWithFlags(&h->last_use, cudaEventDisableTiming));
    if (h->used && h->last_stream != st) CK(cudaStreamWaitEvent(st, h->last_use, 0));
    return IGT_OK;
}

// Constant-memory slot holding this handle's parameters in `prec` (0 = f32, 1 = f64), uploaded if it does not
// hold them yet.  A slot taken over from another handle is first made to wait for that handle's kernels.
static int acquire_cslot(igt_handle *h, int prec, cudaStream_t st, int *slot_out)
{
    std::lock_guard<std::mutex> lk(g_slot_mu);
    const int dev = h->device < MAX_DEV ? h->device : MAX_DEV - 1;
    CSlot *tab = g_slots[dev][prec];
    int sl = h->cslot[prec];
    if (sl < 0 || tab[sl].owner != h) {
        sl = -1;
        for (int i = 0; i < N_CSLOTS && sl < 0; i++) if (!tab[i].owner) sl = i;
        if (sl < 0) sl = (int)(g_slot_rr[dev][prec]++ % N_CSLOTS);       // all taken: share, ordered by the slot's event
        h->cslot[prec] = sl;
    }
    CSlot &c = tab[sl];
    if (c.owner != h || c.version != h->version[prec]) {
        if (c.ev) CK(cudaStreamWaitEvent(st, c.ev, 0));                    // kernels still reading the old content
        if (prec) CK(cudaMemcpyToSymbolAsync(c_Pd, &h->Pd, sizeof(h->Pd), (size_t)sl * sizeof(h->Pd), cudaMemcpyHostToDevice, st));
        else CK(cudaMemcpyToSymbolAsync(c_Pf, &h->Pf, sizeof(h->Pf), (size_t)sl * sizeof(h->Pf), cudaMemcpyHostToDevice, st));
        c.owner = h; c.version = h->version[prec];
    }
    *slot_out = sl;
    return IGT_OK;
}

// Exit of every such call: later users of the handle / of its constant slots wait for these events.
static int end_call(igt_handle *h, cudaStream_t st, int prec_used_mask)
{
    CK(cudaEventRecord(h->last_use, st));
    h->last_stream = st; h->used = true;
    std::lock_guard<std::mutex> lk(g_slot_mu);
    const int dev = h->device < MAX_DEV ? h->device : MAX_DEV - 1;
    for (int prec = 0; prec < 2; prec++)
        if ((prec_used_mask >> prec) & 1) {
            CSlot &c = g_slots[dev][prec][h->cslot[prec]];
            if (!c.ev) CK(cudaEventCreateWithFlags(&c.ev, cudaEventDisableTiming));
            CK(cudaEventRecord(c.ev, st));
        }
    return IGT_OK;
}

// Prologue of every *_host call: one call at a time per handle; the arguments are checked under the lock (bank
// indices are read against the loaded slots, which igt_set_mlp_at changes under it) before anything is allocated or
// copied; then `run` queues its work on the handle's private non-blocking stream.
template <typename Check, typename Run>
static int host_call(igt_handle *h, int B, Check &&check, Run &&run)
{
    if (!h) return IGT_EINVAL;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check();
    if (rc || B == 0) return rc;
    CK(cudaSetDevice(h->device));
    if (!h->hstream) CK(cudaStreamCreateWithFlags(&h->hstream, cudaStreamNonBlocking));
    rc = begin_call(h, h->hstream);
    return rc ? rc : run(h->hstream);
}

// One array of a *_host call: copied in from host memory, copied out to it, or on the device only.  An absent
// (null) host array takes no bytes and gets a null device address.
struct Staged { const void *in; void *out; size_t bytes; void **dev; };
template <typename T, typename D> static Staged input(const T *p, size_t n, D **d) { return { p, nullptr, p ? n * sizeof(T) : 0, (void **)d }; }
template <typename T> static Staged output(T *p, size_t n, T **d) { return { nullptr, p, p ? n * sizeof(T) : 0, (void **)d }; }
template <typename T> static Staged device_only(size_t n, T **d) { return { nullptr, nullptr, n * sizeof(T), (void **)d }; }

// Lays the arrays out in h->stage -- inputs, outputs, device-only arrays, each at a 256-byte boundary -- copies the
// inputs in, calls `run` (which queues the call's kernels on `st`), copies the outputs back and synchronises.
// Inputs and outputs of at most 1 MiB together (the closed-loop step: B = 2) travel in ONE copy each way through the
// pinned block h->pin; larger ones are copied array by array straight from / to the caller's (ideally pinned)
// memory -- packing 100 MB on the host would cost more than the copies.
template <size_t n, typename Run>
static int staged(igt_handle *h, cudaStream_t st, Staged (&a)[n], Run &&run)
{
    size_t off[n], top = 0, end[3];
    for (int kind = 0; kind < 3; kind++) {
        for (size_t i = 0; i < n; i++)
            if ((a[i].in ? 0 : a[i].out ? 1 : 2) == kind) { off[i] = top; top += (a[i].bytes + 255) & ~(size_t)255; }
        end[kind] = top;
    }
    int rc = grow(h, &h->stage, &h->stage_bytes, top, st);
    if (rc) return rc;
    char *d = (char *)h->stage, *pin = nullptr;
    for (size_t i = 0; i < n; i++) *a[i].dev = a[i].bytes ? d + off[i] : nullptr;
    if (end[1] <= (size_t)1 << 20) {
        if (h->pin_bytes < end[1]) {
            if (h->pin) { CK(cudaStreamSynchronize(st)); CK(cudaFreeHost(h->pin)); h->pin = nullptr; h->pin_bytes = 0; }
            CK(cudaHostAlloc(&h->pin, end[1], cudaHostAllocDefault));
            h->pin_bytes = end[1];
        }
        pin = (char *)h->pin;
        for (size_t i = 0; i < n; i++) if (a[i].in && a[i].bytes) memcpy(pin + off[i], a[i].in, a[i].bytes);
        if (end[0]) CK(cudaMemcpyAsync(d, pin, end[0], cudaMemcpyHostToDevice, st));
    } else {
        for (size_t i = 0; i < n; i++)
            if (a[i].in && a[i].bytes) CK(cudaMemcpyAsync(d + off[i], a[i].in, a[i].bytes, cudaMemcpyHostToDevice, st));
    }
    if ((rc = run())) return rc;
    if (pin) {
        if (end[1] > end[0]) CK(cudaMemcpyAsync(pin + end[0], d + end[0], end[1] - end[0], cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        for (size_t i = 0; i < n; i++) if (a[i].out && a[i].bytes) memcpy(a[i].out, pin + off[i], a[i].bytes);
    } else {
        for (size_t i = 0; i < n; i++)
            if (a[i].out && a[i].bytes) CK(cudaMemcpyAsync(a[i].out, d + off[i], a[i].bytes, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    return IGT_OK;
}

// ------------------------------------------------------------------ solver variants -----
// The solver configurations the library is built with, one row each.  A row names its throughput kernel
// solve_kernel<T, TC, OBCA, COOP, BANK>, its cold-start kernel guess_kernel<T, OBCA> and, without TC, its latency
// kernel solve_small_kernel<T, OBCA, COOP, BANK, GT>: these rows are the only instantiations of the three templates.
// TC: tensor-core value term; COOP: the CTA-cooperative exact value term (f64, circle mode, every layer <= MLP_COOP_W);
// BANK: network net_idx[p] of the handle's bank per problem; GT: gt_mpc (a value term at all); DUALS: the row also
// builds solve_kernel<..., DUALS = true>, the throughput kernel that exports every row's final slack and multiplier
// (igt_solve_duals_*: f64 circle mode with the exact value term; these are the inputs of the VJP, sens.cuh).
template <typename T_, bool OBCA_, bool TC_, bool COOP_, bool BANK_, bool GT_, bool DUALS_>
struct Variant {
    using T = T_;
    static constexpr bool OBCA = OBCA_, TC = TC_, COOP = COOP_, BANK = BANK_, GT = GT_, DUALS = DUALS_;
};
template <typename... V> struct VariantList {};
using Variants = VariantList<
    //      T       OBCA   TC     COOP   BANK   GT     DUALS
    Variant<double, false, false, false, false, false, true>,      // 'mpc'
    Variant<float,  false, false, false, false, false, false>,
    Variant<double, true,  false, false, false, false, false>,
    Variant<double, false, false, true,  false, true,  true>,      // gt_mpc, one network
    Variant<double, false, true,  false, false, true,  false>,
    Variant<float,  false, true,  false, false, true,  false>,
    Variant<double, false, false, false, false, true,  true>,
    Variant<double, true,  false, false, false, true,  false>,
    Variant<float,  false, false, false, false, true,  false>,
    Variant<double, false, false, true,  true,  true,  true>,      // gt_mpc, network bank
    Variant<double, false, false, false, true,  true,  true>,
    Variant<double, true,  false, false, true,  true,  false>,
    Variant<float,  false, false, false, true,  true,  false>>;

// f(V()) for the row V with these flags (solve_dev_impl only asks for combinations that have a row)
template <typename F, typename... V>
static int with_variant(igt_handle *h, VariantList<V...>, bool f64, bool obca, bool tc, bool coop, bool bank, bool gt, F &&f)
{
    int rc = IGT_OK;
    const bool hit = ((std::is_same<typename V::T, double>::value == f64 && V::OBCA == obca && V::TC == tc && V::COOP == coop &&
                       V::BANK == bank && V::GT == gt && (rc = f(V()), true)) || ...);
    if (!hit) { h->err = "igt_solve: no solver variant for this combination"; return IGT_EINVAL; }
    return rc;
}

// Widest network the value term of a call may meet: slot 0's, or the widest of the bank (0: nothing loaded).  It sizes
// the per-thread scratch, and the cooperative evaluation applies when it is <= MLP_COOP_W.
static int value_width(const igt_handle *h, bool bank)
{
    int w = h->net_width[0];
    if (bank) for (int k = 1; k < MAX_MLP_NETS; k++) if (h->net_width[k] > w) w = h->net_width[k];
    return w;
}

// Bank calls: every index names a loaded slot (checked on the host before anything is launched, under h->mu, so that
// a concurrent igt_set_mlp_at cannot empty a slot between the check and the launch).
static int check_net_idx(igt_handle *h, int n, const int *net_idx, const char *who)
{
    for (int i = 0; i < n; i++) {
        const int k = net_idx[i];
        if (k < 0 || k >= IGT_MAX_MLP_NETS || h->net_width[k] == 0) {
            h->err = std::string(who) + ": net_idx[" + std::to_string(i) + "] = " + std::to_string(k) + " names no loaded network";
            return IGT_EINVAL;
        }
    }
    return IGT_OK;
}

// arguments of igt_solve_ex_dev / igt_solve_ex_host (host_idx: net_idx is in host memory and is checked here; a device
// index is checked in the kernel: IGT_STATUS_BAD_NET)
static int check_solve(igt_handle *h, int B, const ProbIO &io, const int *net_idx, bool host_idx)
{
    if (B < 0 || !io.x0 || !io.u_prev || !io.curv || !io.obs || !io.x || !io.u || !io.cost || !io.viol || !io.status || !io.iters) {
        h->err = "igt_solve: null argument"; return IGT_EINVAL;
    }
    if (net_idx && !io.ctx) { h->err = "igt_solve: net_idx needs nn_ctx (gt_mpc)"; return IGT_EINVAL; }
    if (net_idx && host_idx) { const int rc = check_net_idx(h, B, net_idx, "igt_solve"); if (rc) return rc; }
    if (io.ctx && value_width(h, net_idx != nullptr) == 0) {
        h->err = net_idx ? "igt_solve: net_idx given but no network was loaded" : "igt_solve: nn_ctx given but igt_set_mlp was never called";
        return IGT_ENOMLP;
    }
    if (io.obs_psi && h->prm.precision != IGT_PREC_F64) { h->err = "igt_solve: the OBCA collision rows (obs_psi) need precision f64"; return IGT_EINVAL; }
    return IGT_OK;
}

// io as the kernels of a row with BANK take it: with the bank's descriptor table in T (the f32 one follows the f64 one)
template <typename T, bool BANK>
static typename std::conditional<BANK, ProbIONet<T>, ProbIO>::type io_for(const ProbIO &io, const int *net_idx, const igt_handle *h)
{
    typename std::conditional<BANK, ProbIONet<T>, ProbIO>::type r;
    static_cast<ProbIO &>(r) = io;
    if constexpr (BANK) {
        r.net_idx = net_idx;
        r.nets = (const MlpNet<T> *)((const char *)h->bank + (sizeof(T) == 8 ? 0 : sizeof(h->netd)));
    }
    return r;
}

// Solve of checked arguments (device pointers) on `st`.  slack / mult [B][M] (both or neither): a dual-exporting solve
// (checked by check_duals), always on the throughput kernel: the latency kernel gives the same bits, so the small
// batches it would take are exported from the throughput kernel without a latency twin of each dual-exporting row.
static int solve_dev_impl(igt_handle *h, int B, const ProbIO &io, const int *net_idx, cudaStream_t st,
                          double *slack = nullptr, double *mult = nullptr)
{
    if (B == 0) return IGT_OK;
    int rc = begin_call(h, st);
    if (rc) return rc;
    const bool f64 = h->prm.precision == IGT_PREC_F64, obca = io.obs_psi != nullptr, gt = io.ctx != nullptr, bank = net_idx != nullptr;
    WsLayout L; L.init(h->prm.N, h->prm.n_cinf, obca ? NGE_OBCA : NGE, obca ? NHE_OBCA : NHE);
    // value term (OBCA + gt_mpc: per-thread value term; a bank: exact evaluation whatever tensor_core_mlp says)
    const int width = value_width(h, bank);
    const bool use_tc = gt && !bank && h->tc.enabled && h->use_tc && !obca;
    const bool use_coop = gt && !use_tc && f64 && width <= MLP_COOP_W && !obca;
    // persistent lanes: one CTA of SOLVE_BLOCK threads per SM.  A batch smaller than the machine is spread
    // over all SMs, a whole number of warps each: `quota` threads per CTA fetch problems, the rest of
    // the CTA only helps in the CTA-wide phases (and adopts stragglers in the tail).
    const int bs = SOLVE_BLOCK;
    long n_cta = ((long)B + 31) / 32;
    if (n_cta > h->n_sm) n_cta = h->n_sm;
    long per_cta = ((long)B + n_cta - 1) / n_cta;
    int quota = (int)((per_cta + 31) / 32 * 32);
    if (quota > bs) quota = bs;
    const long n_slots = n_cta * bs;
    return with_variant(h, Variants(), f64, obca, use_tc, use_coop, bank, gt, [&](auto v) -> int {
        using V = decltype(v);
        using T = typename V::T;
        // latency path: at most one problem per SM and a workspace that fits shared memory next to the work lists; in
        // gt_mpc (not with the tensor-core value term) the kernel's whole shared memory -- static, value-term buffers,
        // workspace -- within the device's opt-in limit per block
        const size_t small_smem = (size_t)L.total * sizeof(T) + small_coop_bytes<T, V::COOP, V::BANK>();
        bool small = false;
        if constexpr (!V::TC) {
            if (h->use_small && B <= h->n_sm && !slack) {
                if constexpr (V::GT) {
                    static std::atomic<int> static_smem{ -1 };   // the latency kernel's static shared memory, read once
                    if (static_smem < 0) {
                        cudaFuncAttributes fa;
                        CK(cudaFuncGetAttributes(&fa, solve_small_kernel<T, V::OBCA, V::COOP, V::BANK, V::GT>));
                        static_smem = (int)fa.sharedSizeBytes;
                    }
                    small = small_smem + (size_t)static_smem <= (size_t)h->smem_optin;
                } else {
                    small = small_smem <= 200 * 1024;
                }
            }
        }
        int rc = small ? IGT_OK : grow(h, &h->ws, &h->ws_bytes, (size_t)L.total * n_slots * sizeof(T), st);
        if (rc) return rc;
        constexpr bool per_thread = V::GT && !V::TC && !V::COOP;      // per-thread value term: activations in HBM
        if (per_thread) {                                                // (one slab per persistent lane, or per CTA on the latency path)
            rc = grow(h, &h->mlp_scratch, &h->mlp_scratch_bytes, (size_t)12 * width * (small ? B : n_slots) * sizeof(T), st);
            if (rc) return rc;
        }
        T *scratch = per_thread ? (T *)h->mlp_scratch : nullptr;
        // scheduler block (the work counter), then the cold-start guesses
        const size_t off_guess = 256;
        rc = grow(h, &h->guess, &h->guess_bytes, off_guess + (size_t)B * h->prm.N * 2 * sizeof(double), st);
        if (rc) return rc;
        char *sb = (char *)h->guess;
        Sched sc;
        sc.counter = (unsigned long long *)sb;
        double *guess = (double *)(sb + off_guess);
        int cs = 0;
        rc = acquire_cslot(h, f64 ? 1 : 0, st, &cs);
        if (rc) return rc;
        CK(cudaMemsetAsync(sb, 0, 256, st));
        if (!io.u_init || io.warm) {
            guess_kernel<T, V::OBCA><<<(B + 127) / 128, 128, 0, st>>>(io, B, guess, cs);
            h->launches++;
        }
        using IO = typename std::conditional<V::BANK, ProbIONet<T>, ProbIO>::type;
        const IO iob = io_for<T, V::BANK>(io, net_idx, h);   // (a bank problem with a bad index gets IGT_STATUS_BAD_NET)
        if constexpr (!V::TC) {
            if (small) {
                typename std::conditional<V::GT, SmallIO<IO, T>, IO>::type ios;
                static_cast<IO &>(ios) = iob;
                if constexpr (V::GT) { ios.mlp_scratch = scratch; ios.mlp_width = width; }
                auto *k = solve_small_kernel<T, V::OBCA, V::COOP, V::BANK, V::GT>;
                CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small_smem));
                k<<<B, bs, small_smem, st>>>(ios, B, sc, guess, cs);
            }
        }
        const int smem = V::TC ? TC_SMEM_BYTES
                       : V::COOP ? (V::BANK ? mlp_coop_bank_smem_bytes<T>(SOLVE_BLOCK) : mlp_coop_smem_bytes<T>(SOLVE_BLOCK))
                       : IGT_RSTG ? RSTG_SLOTS * SOLVE_BLOCK * (int)sizeof(T) : 0;
        if (slack) {
            if constexpr (V::DUALS) {
                SolveIO<T, V::BANK, true> iod;
                static_cast<IO &>(iod) = iob;
                iod.slack = slack; iod.mult = mult;
                auto *k = solve_kernel<T, V::TC, V::OBCA, V::COOP, V::BANK, true>;
                CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
                k<<<(int)(n_slots / bs), bs, smem, st>>>(iod, (T *)h->ws, n_slots, B, sc, guess, scratch, width, h->tc, quota, cs);
            } else {
                h->err = "igt_solve_duals: no dual-exporting solver for this combination";
                return IGT_EINVAL;
            }
        } else if (!small) {
            auto *k = solve_kernel<T, V::TC, V::OBCA, V::COOP, V::BANK>;
            CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            k<<<(int)(n_slots / bs), bs, smem, st>>>(iob, (T *)h->ws, n_slots, B, sc, guess, scratch, width, h->tc, quota, cs);
        }
        h->launches++;
        CK(cudaGetLastError());
        return end_call(h, st, f64 ? 2 : 1);
    });
}

// slot 0's network in the solver parameters (constant memory) of the single-network calls
template <typename T>
static void set_param_net(DevParams<T> &P, const MlpNet<T> &n)
{
    P.n_layers = n.n_layers;
    memcpy(P.dims, n.dims, sizeof(P.dims)); memcpy(P.Wn, n.Wn, sizeof(P.Wn)); memcpy(P.mu_f, n.mu_f, sizeof(P.mu_f));
    P.sigma_t = n.sigma_t; P.mu_t = n.mu_t;
    memcpy(P.W, n.W, sizeof(P.W)); memcpy(P.b, n.b, sizeof(P.b)); memcpy(P.Wt, n.Wt, sizeof(P.Wt));
}

extern "C" {

const char *igt_version(void) { return "igtmpc 0.1 sm_100a"; }

int igt_default_params(igt_params *p, int precision) { return igt::default_params(p, precision); }

int igt_create(const igt_params *p, igt_handle **out)
{
    if (!p || !out) { g_create_err = "null argument"; return IGT_EINVAL; }
    if (p->N < 2 || p->N > 64 || p->n_rk < 1 || p->n_cinf < 0 || p->n_cinf > IGT_MAX_CINF ||
        (p->precision != IGT_PREC_F32 && p->precision != IGT_PREC_F64)) {
        g_create_err = "unsupported N / n_rk / n_cinf / precision";
        return IGT_EINVAL;
    }
    if (p->n_alpha < 1 || p->n_alpha > MAX_ALPHA) { g_create_err = "n_alpha must be in 1..6"; return IGT_EINVAL; }
    igt_handle *h = new (std::nothrow) igt_handle();
    if (!h) { g_create_err = "out of memory"; return IGT_EINVAL; }
    h->prm = *p;
    fill_dev_params(*p, h->Pf);
    fill_dev_params(*p, h->Pd);
    cudaError_t e = cudaGetDevice(&h->device);
    if (e != cudaSuccess) {
        g_create_err = std::string("cudaGetDevice: ") + cudaGetErrorString(e) + " (no CUDA device: this library has no CPU path)";
        delete h;
        return IGT_ECUDA;
    }
    cudaDeviceGetAttribute(&h->n_sm, cudaDevAttrMultiProcessorCount, h->device);
    if (h->n_sm <= 0) h->n_sm = 148;
    cudaDeviceGetAttribute(&h->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device);
    *out = h;
    return IGT_OK;
}

void igt_destroy(igt_handle *h)
{
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->last_use) { cudaEventSynchronize(h->last_use); cudaEventDestroy(h->last_use); }
    {
        std::lock_guard<std::mutex> lk(g_slot_mu);
        const int dev = h->device < MAX_DEV ? h->device : MAX_DEV - 1;
        for (int prec = 0; prec < 2; prec++)
            for (int i = 0; i < N_CSLOTS; i++)
                if (g_slots[dev][prec][i].owner == h) { g_slots[dev][prec][i].owner = nullptr; g_slots[dev][prec][i].version = 0; }
    }
    for (void *b : h->mlp_buf) if (b) cudaFree(b);
    if (h->bank) cudaFree(h->bank);
    if (h->hstream) cudaStreamDestroy(h->hstream);
    if (h->pin) cudaFreeHost(h->pin);
    if (h->ws) cudaFree(h->ws);
    if (h->mlp_scratch) cudaFree(h->mlp_scratch);
    if (h->stage) cudaFree(h->stage);
    if (h->guess) cudaFree(h->guess);
    if (h->sens) cudaFree(h->sens);
    delete h;
}

const char *igt_last_error(const igt_handle *h) { return h ? h->err.c_str() : g_create_err.c_str(); }

long long igt_launch_count(const igt_handle *h) { return h ? h->launches : 0; }

int igt_set_mlp_at(igt_handle *h, int net, int n_layers, const int *dims, const double *const *W, const double *const *b,
                   const double *Wn, const double *mu_f, double sigma_t, double mu_t)
{
    if (!h) return IGT_EINVAL;
    if (net < 0 || net >= IGT_MAX_MLP_NETS) { h->err = "igt_set_mlp: net must be in 0..IGT_MAX_MLP_NETS-1"; return IGT_EINVAL; }
    if (n_layers < 1 || n_layers > IGT_MAX_MLP_LAYERS || !dims || !W || !b || !Wn || !mu_f || dims[0] != 6 ||
        dims[n_layers] != 1) { h->err = "igt_set_mlp: bad layer description"; return IGT_EINVAL; }
    int width = 6;
    for (int l = 0; l <= n_layers; l++) { if (dims[l] < 1 || dims[l] > 1024) { h->err = "igt_set_mlp: bad width"; return IGT_EINVAL; } if (dims[l] > width) width = dims[l]; }
    for (int l = 0; l < n_layers; l++) if (!W[l] || !b[l]) { h->err = "igt_set_mlp: null layer"; return IGT_EINVAL; }
    // the slot's device image, built here and uploaded in one copy: per layer W, b in f64 and f32 and the transposed
    // copies [in][out] for the cooperative evaluation (mlp_coop.cuh); for slot 0 of shape 6-128-128-1 also the
    // tensor-core copy.  Every array starts at a 256-byte boundary, as a cudaMalloc of its own would.
    std::vector<uint8_t> img;
    auto put = [&img](const void *src, size_t bytes) {
        const size_t o = img.size();
        img.resize((o + bytes + 255) & ~(size_t)255);
        memcpy(img.data() + o, src, bytes);
        return o;
    };
    size_t o_net[IGT_MAX_MLP_LAYERS][6];
    for (int l = 0; l < n_layers; l++) {
        const size_t nw = (size_t)dims[l] * dims[l + 1], nb = dims[l + 1];
        std::vector<float> wf(nw), bf(nb);
        for (size_t i = 0; i < nw; i++) wf[i] = (float)W[l][i];
        for (size_t i = 0; i < nb; i++) bf[i] = (float)b[l][i];
        std::vector<double> wtd(nw); std::vector<float> wtf(nw);
        for (int o = 0; o < dims[l + 1]; o++)
            for (int i = 0; i < dims[l]; i++) { wtd[(size_t)i * dims[l + 1] + o] = W[l][(size_t)o * dims[l] + i]; wtf[(size_t)i * dims[l + 1] + o] = (float)W[l][(size_t)o * dims[l] + i]; }
        o_net[l][0] = put(W[l], nw * 8); o_net[l][1] = put(b[l], nb * 8);
        o_net[l][2] = put(wf.data(), nw * 4); o_net[l][3] = put(bf.data(), nb * 4);
        o_net[l][4] = put(wtd.data(), nw * 8); o_net[l][5] = put(wtf.data(), nw * 4);
    }
    const bool tc = net == 0 && n_layers == 3 && dims[1] == MLP_H && dims[2] == MLP_H;
    size_t o_tc[5] = {};
    if (tc) {
        // tensor-core copy: W1eff = W1 Wn, b1eff = b1 - W1eff mu_f (fp32), W2 as bf16 hi/mid/lo in UMMA core-matrix order
        std::vector<float> w1eff(MLP_H * 6), b1eff(MLP_H), b2(MLP_H), w3(MLP_H);
        for (int o = 0; o < MLP_H; o++) {
            double bacc = b[0][o];
            for (int j = 0; j < 6; j++) {
                double acc = 0;
                for (int i = 0; i < 6; i++) acc += W[0][o * 6 + i] * Wn[i * 6 + j];
                w1eff[o * 6 + j] = (float)acc;
                bacc -= acc * mu_f[j];
            }
            b1eff[o] = (float)bacc; b2[o] = (float)b[1][o]; w3[o] = (float)W[2][o];
        }
        std::vector<uint8_t> blob(3 * TC_TILE_BYTES);
        for (int n = 0; n < MLP_H; n++)
            for (int k = 0; k < MLP_H; k++) {
                float x = (float)W[1][n * MLP_H + k];
                __nv_bfloat16 hi = __float2bfloat16_rn(x);
                float r1 = x - __bfloat162float(hi);
                __nv_bfloat16 mid = __float2bfloat16_rn(r1);
                __nv_bfloat16 lo = __float2bfloat16_rn(r1 - __bfloat162float(mid));
                int off = tc_elem_offset(n, k);
                memcpy(&blob[off], &hi, 2); memcpy(&blob[TC_TILE_BYTES + off], &mid, 2); memcpy(&blob[2 * TC_TILE_BYTES + off], &lo, 2);
            }
        o_tc[0] = put(blob.data(), blob.size()); o_tc[1] = put(w1eff.data(), w1eff.size() * 4);
        o_tc[2] = put(b1eff.data(), MLP_H * 4); o_tc[3] = put(b2.data(), MLP_H * 4); o_tc[4] = put(w3.data(), MLP_H * 4);
    }
    std::lock_guard<std::mutex> lk(h->mu);
    CK(cudaSetDevice(h->device));
    if (h->last_use && h->used) CK(cudaEventSynchronize(h->last_use));   // no kernel of this handle reads the old network
    if (!h->bank) CK(cudaMalloc(&h->bank, MAX_MLP_NETS * (sizeof(MlpNet<double>) + sizeof(MlpNet<float>))));
    h->version[0]++; h->version[1]++;
    if (h->mlp_buf[net]) { cudaFree(h->mlp_buf[net]); h->mlp_buf[net] = nullptr; }
    h->net_width[net] = 0;
    if (net == 0) h->tc.enabled = 0;
    MlpNet<double> &nd = h->netd[net];
    MlpNet<float> &nf = h->netf[net];
    nd = MlpNet<double>(); nf = MlpNet<float>();
    CK(cudaMalloc(&h->mlp_buf[net], img.size()));
    CK(cudaMemcpy(h->mlp_buf[net], img.data(), img.size(), cudaMemcpyHostToDevice));
    const uint8_t *base = (const uint8_t *)h->mlp_buf[net];
    nf.n_layers = nd.n_layers = n_layers;
    for (int l = 0; l <= n_layers; l++) nf.dims[l] = nd.dims[l] = dims[l];
    for (int l = 0; l < n_layers; l++) {
        nd.W[l] = (const double *)(base + o_net[l][0]); nd.b[l] = (const double *)(base + o_net[l][1]);
        nf.W[l] = (const float *)(base + o_net[l][2]); nf.b[l] = (const float *)(base + o_net[l][3]);
        nd.Wt[l] = (const double *)(base + o_net[l][4]); nf.Wt[l] = (const float *)(base + o_net[l][5]);
    }
    for (int i = 0; i < 36; i++) { nd.Wn[i] = Wn[i]; nf.Wn[i] = (float)Wn[i]; }
    for (int i = 0; i < 6; i++) { nd.mu_f[i] = mu_f[i]; nf.mu_f[i] = (float)mu_f[i]; }
    nd.sigma_t = sigma_t; nd.mu_t = mu_t; nf.sigma_t = (float)sigma_t; nf.mu_t = (float)mu_t;
    h->net_width[net] = width;
    // the whole descriptor table (empty slots: n_layers = 0); bank launches pass it to the kernels (ProbIONet::nets)
    CK(cudaMemcpy(h->bank, h->netd, sizeof(h->netd), cudaMemcpyHostToDevice));
    CK(cudaMemcpy((char *)h->bank + sizeof(h->netd), h->netf, sizeof(h->netf), cudaMemcpyHostToDevice));
    if (net != 0) return IGT_OK;
    // slot 0 is the handle's network of the single-network calls: in DevParams (constant memory) and the tcgen05 copy
    set_param_net(h->Pd, nd);
    set_param_net(h->Pf, nf);
    if (tc) {
        h->tc.w2_splits = base + o_tc[0]; h->tc.w1eff = (const float *)(base + o_tc[1]); h->tc.b1eff = (const float *)(base + o_tc[2]);
        h->tc.b2 = (const float *)(base + o_tc[3]); h->tc.w3 = (const float *)(base + o_tc[4]);
        h->tc.b3 = (float)b[2][0]; h->tc.sigma_t = (float)sigma_t; h->tc.mu_t = (float)mu_t;
        h->tc.enabled = 1;
        CK(cudaFuncSetAttribute(mlp_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_BYTES));
    }
    return IGT_OK;
}

int igt_set_mlp(igt_handle *h, int n_layers, const int *dims, const double *const *W, const double *const *b,
                const double *Wn, const double *mu_f, double sigma_t, double mu_t)
{
    return igt_set_mlp_at(h, 0, n_layers, dims, W, b, Wn, mu_f, sigma_t, mu_t);
}

static int check_rollout(igt_handle *h, int B, const float *z0, const float *u, const float *curv, const float *z,
                         const float *A, const float *Bm, int model)
{
    if (B < 0 || !z0 || !u || !z || (model == 0 && !curv) || ((A == nullptr) != (Bm == nullptr)) ||
        (model != 0 && model != 1)) { h->err = "igt_rollout: bad argument"; return IGT_EINVAL; }
    return IGT_OK;
}

static int rollout_dev_impl(igt_handle *h, int B, const float *z0, const float *u, const float *curv, float *z,
                            float *A, float *Bm, int model, cudaStream_t st)
{
    int rc = begin_call(h, st), cs = 0;
    if (rc) return rc;
    rc = acquire_cslot(h, 0, st, &cs);
    if (rc) return rc;
    int bs = 128, gs = (B + bs - 1) / bs;
    if (model == 0) rollout_kernel<<<gs, bs, 0, st>>>(B, z0, u, curv, z, A, Bm, cs);
    else rollout_euler_kernel<<<gs, bs, 0, st>>>(B, z0, u, z, A, Bm, cs);
    h->launches++;
    CK(cudaGetLastError());
    return end_call(h, st, 1);
}

int igt_rollout_dev(igt_handle *h, int B, const float *z0, const float *u, const float *curv, float *z,
                    float *A, float *Bm, int model, void *stream)
{
    if (!h) return IGT_EINVAL;
    std::lock_guard<std::mutex> lk(h->mu);
    const int rc = check_rollout(h, B, z0, u, curv, z, A, Bm, model);
    if (rc || B == 0) return rc;
    return rollout_dev_impl(h, B, z0, u, curv, z, A, Bm, model, (cudaStream_t)stream);
}

int igt_rollout_host(igt_handle *h, int B, const float *z0, const float *u, const float *curv, float *z,
                     float *A, float *Bm, int model)
{
    return host_call(h, B, [&] { return check_rollout(h, B, z0, u, curv, z, A, Bm, model); }, [&](cudaStream_t st) {
        const size_t N = h->prm.N, nb = B, nz = model == 0 ? 7 : 4;
        const float *dz0, *du, *dc;
        float *dz, *dA, *dB;
        Staged a[] = { input(z0, nb * nz, &dz0), input(u, nb * N * 2, &du), input(model == 0 ? curv : nullptr, nb * 3, &dc),
                       output(z, nb * (N + 1) * nz, &dz), output(A, nb * N * nz * nz, &dA), output(Bm, nb * N * nz * 2, &dB) };
        return staged(h, st, a, [&] { return rollout_dev_impl(h, B, dz0, du, dc, dz, dA, dB, model, st); });
    });
}

int igt_solve_ex_dev(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                     const double *obs_xy, const double *obs_psi, const double *nn_ctx, const int *net_idx, const double *u_init,
                     double *x, double *u, double *cost, double *viol, int *status, int *iters, void *stream)
{
    if (!h) return IGT_EINVAL;
    const ProbIO io = { x0, u_prev, curv, obs_xy, nn_ctx, u_init, x, u, cost, viol, status, iters, obs_psi };
    std::lock_guard<std::mutex> lk(h->mu);
    const int rc = check_solve(h, B, io, net_idx, false);
    return rc ? rc : solve_dev_impl(h, B, io, net_idx, (cudaStream_t)stream);
}

int igt_solve_dev(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                  const double *obs_xy, const double *obs_psi, const double *nn_ctx, const double *u_init, double *x,
                  double *u, double *cost, double *viol, int *status, int *iters, void *stream)
{
    return igt_solve_ex_dev(h, B, x0, u_prev, curv, obs_xy, obs_psi, nn_ctx, nullptr, u_init, x, u, cost, viol, status, iters, stream);
}

int igt_solve_ex_host(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                      const double *obs_xy, const double *obs_psi, const double *nn_ctx, const int *net_idx, const double *u_init,
                      double *x, double *u, double *cost, double *viol, int *status, int *iters)
{
    const ProbIO io = { x0, u_prev, curv, obs_xy, nn_ctx, u_init, x, u, cost, viol, status, iters, obs_psi };
    return host_call(h, B, [&] { return check_solve(h, B, io, net_idx, true); }, [&](cudaStream_t st) {
        const size_t N = h->prm.N, nb = B;
        ProbIO d = {};
        const int *dnet;
        Staged a[] = { input(x0, nb * 7, &d.x0), input(u_prev, nb * 2, &d.u_prev), input(curv, nb * 3, &d.curv),
                       input(obs_xy, nb * (N + 1) * 2, &d.obs), input(nn_ctx, nb * 4, &d.ctx), input(u_init, nb * N * 2, &d.u_init),
                       input(obs_psi, nb * (N + 1), &d.obs_psi), input(net_idx, nb, &dnet),
                       output(x, nb * (N + 1) * 7, &d.x), output(u, nb * N * 2, &d.u), output(cost, nb, &d.cost), output(viol, nb, &d.viol),
                       output(status, nb, &d.status), output(iters, nb, &d.iters) };
        return staged(h, st, a, [&] { return solve_dev_impl(h, B, d, dnet, st); });
    });
}

int igt_solve_host(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                   const double *obs_xy, const double *obs_psi, const double *nn_ctx, const double *u_init, double *x,
                   double *u, double *cost, double *viol, int *status, int *iters)
{
    return igt_solve_ex_host(h, B, x0, u_prev, curv, obs_xy, obs_psi, nn_ctx, nullptr, u_init, x, u, cost, viol, status, iters);
}

int igt_row_count(const igt_handle *h) { return h ? row_total(h->prm.N, h->prm.n_cinf) : IGT_EINVAL; }

// the further conditions of a dual-exporting solve (after check_solve)
static int check_duals(igt_handle *h, const ProbIO &io, const double *slack, const double *mult)
{
    if (!slack || !mult) { h->err = "igt_solve_duals: null argument"; return IGT_EINVAL; }
    if (h->prm.precision != IGT_PREC_F64) { h->err = "igt_solve_duals: needs precision f64"; return IGT_EINVAL; }
    if (io.obs_psi) { h->err = "igt_solve_duals: not in the OBCA collision mode (obs_psi)"; return IGT_EINVAL; }
    if (io.ctx && h->use_tc) { h->err = "igt_solve_duals: not with the tensor-core value term (tensor_core_mlp = 1)"; return IGT_EINVAL; }
    return IGT_OK;
}

int igt_solve_duals_ex_dev(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                           const double *obs_xy, const double *obs_psi, const double *nn_ctx, const int *net_idx,
                           const double *u_init, double *x, double *u, double *cost, double *viol, int *status, int *iters,
                           double *slack, double *mult, void *stream)
{
    if (!h) return IGT_EINVAL;
    const ProbIO io = { x0, u_prev, curv, obs_xy, nn_ctx, u_init, x, u, cost, viol, status, iters, obs_psi };
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = check_solve(h, B, io, net_idx, false);
    if (!rc) rc = check_duals(h, io, slack, mult);
    return rc ? rc : solve_dev_impl(h, B, io, net_idx, (cudaStream_t)stream, slack, mult);
}

int igt_solve_duals_ex_host(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                            const double *obs_xy, const double *obs_psi, const double *nn_ctx, const int *net_idx,
                            const double *u_init, double *x, double *u, double *cost, double *viol, int *status, int *iters,
                            double *slack, double *mult)
{
    const ProbIO io = { x0, u_prev, curv, obs_xy, nn_ctx, u_init, x, u, cost, viol, status, iters, obs_psi };
    return host_call(h, B, [&] { int rc = check_solve(h, B, io, net_idx, true); return rc ? rc : check_duals(h, io, slack, mult); },
                     [&](cudaStream_t st) {
        const size_t N = h->prm.N, nb = B, M = row_total(h->prm.N, h->prm.n_cinf);
        ProbIO d = {};
        const int *dnet;
        double *dy, *ds;
        Staged a[] = { input(x0, nb * 7, &d.x0), input(u_prev, nb * 2, &d.u_prev), input(curv, nb * 3, &d.curv),
                       input(obs_xy, nb * (N + 1) * 2, &d.obs), input(nn_ctx, nb * 4, &d.ctx), input(u_init, nb * N * 2, &d.u_init),
                       input(net_idx, nb, &dnet),
                       output(x, nb * (N + 1) * 7, &d.x), output(u, nb * N * 2, &d.u), output(cost, nb, &d.cost), output(viol, nb, &d.viol),
                       output(status, nb, &d.status), output(iters, nb, &d.iters), output(slack, nb * M, &dy), output(mult, nb * M, &ds) };
        return staged(h, st, a, [&] { return solve_dev_impl(h, B, d, dnet, st, dy, ds); });
    });
}

// arguments of igt_solve_vjp_dev / _host (host_idx: as in check_solve)
static int check_vjp(igt_handle *h, int B, const SensIO &io, bool host_idx)
{
    if (B < 0 || !io.x0 || !io.u_prev || !io.curv || !io.obs || !io.u || !io.slack || !io.mult || !io.status || !io.gx0 ||
        !io.gu_prev || !io.gobs || !io.ok) { h->err = "igt_solve_vjp: null argument"; return IGT_EINVAL; }
    if (h->prm.precision != IGT_PREC_F64) { h->err = "igt_solve_vjp: needs precision f64"; return IGT_EINVAL; }
    if (io.ctx && h->use_tc) { h->err = "igt_solve_vjp: not with the tensor-core value term (tensor_core_mlp = 1)"; return IGT_EINVAL; }
    if (io.net_idx && !io.ctx) { h->err = "igt_solve_vjp: net_idx needs nn_ctx (gt_mpc)"; return IGT_EINVAL; }
    if (io.net_idx && host_idx) { const int rc = check_net_idx(h, B, io.net_idx, "igt_solve_vjp"); if (rc) return rc; }
    if (io.ctx && value_width(h, io.net_idx != nullptr) == 0) { h->err = "igt_solve_vjp: nn_ctx given but no network was loaded"; return IGT_ENOMLP; }
    return IGT_OK;
}

static int vjp_dev_impl(igt_handle *h, int B, SensIO io, cudaStream_t st)
{
    if (B == 0) return IGT_OK;
    int rc = begin_call(h, st), cs = 0;
    if (rc) return rc;
    const int width = value_width(h, io.net_idx != nullptr);
    const size_t ws = (size_t)B * sens_ws_size(h->prm.N), scr = io.ctx ? (size_t)B * 12 * width : 0;
    if ((rc = grow(h, &h->sens, &h->sens_bytes, (ws + scr) * sizeof(double), st))) return rc;
    if ((rc = acquire_cslot(h, 1, st, &cs))) return rc;
    io.nets = (const MlpNet<double> *)h->bank;
    double *base = (double *)h->sens;
    auto *k = io.net_idx ? vjp_kernel<true> : vjp_kernel<false>;
    k<<<(B + 127) / 128, 128, 0, st>>>(io, B, base, io.ctx ? base + ws : nullptr, width, cs);
    h->launches++;
    CK(cudaGetLastError());
    return end_call(h, st, 2);
}

int igt_solve_vjp_dev(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv, const double *obs_xy,
                      const double *nn_ctx, const int *net_idx, const double *u, const double *slack, const double *mult,
                      const int *status, const double *gx, const double *gu, const double *gcost, double *gx0, double *gu_prev,
                      double *gobs, int *ok, void *stream)
{
    if (!h) return IGT_EINVAL;
    SensIO io = { x0, u_prev, curv, obs_xy, nn_ctx, net_idx, nullptr, u, slack, mult, status, gx, gu, gcost, gx0, gu_prev, gobs, ok };
    std::lock_guard<std::mutex> lk(h->mu);
    const int rc = check_vjp(h, B, io, false);
    return rc ? rc : vjp_dev_impl(h, B, io, (cudaStream_t)stream);
}

int igt_solve_vjp_host(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv, const double *obs_xy,
                       const double *nn_ctx, const int *net_idx, const double *u, const double *slack, const double *mult,
                       const int *status, const double *gx, const double *gu, const double *gcost, double *gx0, double *gu_prev,
                       double *gobs, int *ok)
{
    const SensIO io = { x0, u_prev, curv, obs_xy, nn_ctx, net_idx, nullptr, u, slack, mult, status, gx, gu, gcost, gx0, gu_prev, gobs, ok };
    return host_call(h, B, [&] { return check_vjp(h, B, io, true); }, [&](cudaStream_t st) {
        const size_t N = h->prm.N, nb = B, M = row_total(h->prm.N, h->prm.n_cinf);
        SensIO d = {};
        Staged a[] = { input(x0, nb * 7, &d.x0), input(u_prev, nb * 2, &d.u_prev), input(curv, nb * 3, &d.curv),
                       input(obs_xy, nb * (N + 1) * 2, &d.obs), input(nn_ctx, nb * 4, &d.ctx), input(net_idx, nb, &d.net_idx),
                       input(u, nb * N * 2, &d.u), input(slack, nb * M, &d.slack), input(mult, nb * M, &d.mult),
                       input(status, nb, &d.status), input(gx, nb * (N + 1) * 7, &d.gx), input(gu, nb * N * 2, &d.gu),
                       input(gcost, nb, &d.gcost),
                       output(gx0, nb * 7, &d.gx0), output(gu_prev, nb * 2, &d.gu_prev), output(gobs, nb * (N + 1) * 2, &d.gobs),
                       output(ok, nb, &d.ok) };
        return staged(h, st, a, [&] { return vjp_dev_impl(h, B, d, st); });
    });
}

int igt_eval_ex_host(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                     const double *obs_xy, const double *obs_psi, const double *nn_ctx, const int *net_idx, const double *u,
                     double *cost, double *viol, double *z)
{
    auto check = [&]() -> int {
        if (B < 0 || !x0 || !u_prev || !curv || !obs_xy || !u || !cost || !viol) { h->err = "igt_eval: null argument"; return IGT_EINVAL; }
        if (net_idx && !nn_ctx) { h->err = "igt_eval: net_idx needs nn_ctx (gt_mpc)"; return IGT_EINVAL; }
        if (nn_ctx && !net_idx && value_width(h, false) == 0) { h->err = "igt_eval: nn_ctx given but igt_set_mlp was never called"; return IGT_ENOMLP; }
        return net_idx ? check_net_idx(h, B, net_idx, "igt_eval") : IGT_OK;
    };
    return host_call(h, B, check, [&](cudaStream_t st) {
        const size_t N = h->prm.N, nb = B;
        const double *dx0, *dup, *dc, *dob, *dctx, *du, *dop;
        const int *dnet;
        double *dcost, *dviol, *dz;
        Staged a[] = { input(x0, nb * 7, &dx0), input(u_prev, nb * 2, &dup), input(curv, nb * 3, &dc), input(obs_xy, nb * (N + 1) * 2, &dob),
                       input(nn_ctx, nb * 4, &dctx), input(u, nb * N * 2, &du), input(obs_psi, nb * (N + 1), &dop), input(net_idx, nb, &dnet),
                       output(cost, nb, &dcost), output(viol, nb, &dviol), output(z, nb * (N + 1) * 7, &dz) };
        return staged(h, st, a, [&] {
            const int width = value_width(h, net_idx != nullptr);
            if (nn_ctx) { const int rc = grow(h, &h->mlp_scratch, &h->mlp_scratch_bytes, (size_t)12 * width * nb * 8, st); if (rc) return rc; }
            int cs = 0;
            const int rc = acquire_cslot(h, 1, st, &cs);
            if (rc) return rc;
            auto *k = net_idx ? eval_kernel<true> : eval_kernel<false>;
            k<<<(B + 127) / 128, 128, 0, st>>>(B, dx0, dup, dc, dob, dctx, du, dcost, dviol, dz, nn_ctx ? (double *)h->mlp_scratch : nullptr,
                                               width, cs, dop, dnet, (const MlpNet<double> *)h->bank);
            h->launches++;
            CK(cudaGetLastError());
            return end_call(h, st, 2);
        });
    });
}

int igt_eval_host(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                  const double *obs_xy, const double *obs_psi, const double *nn_ctx, const double *u, double *cost,
                  double *viol, double *z)
{
    return igt_eval_ex_host(h, B, x0, u_prev, curv, obs_xy, obs_psi, nn_ctx, nullptr, u, cost, viol, z);
}

int igt_measure_fma_peak(igt_handle *h, int precision, double *tflops)
{
    if (!h || !tflops) return IGT_EINVAL;
    const int blocks = h->n_sm * 8, threads = 256, iters = 1 << 16;
    std::lock_guard<std::mutex> lk(h->mu);
    int rc = begin_call(h, nullptr);
    if (rc) return rc;
    rc = grow(h, &h->stage, &h->stage_bytes, (size_t)blocks * threads * 8, nullptr);
    if (rc) return rc;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        CK(cudaEventRecord(e0));
        if (precision == IGT_PREC_F64) fma_peak_kernel<double><<<blocks, threads>>>((double *)h->stage, iters);
        else fma_peak_kernel<float><<<blocks, threads>>>((float *)h->stage, iters);
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        float ms;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0 && ms < best) best = ms;
        h->launches++;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    rc = end_call(h, nullptr, 0);
    if (rc) return rc;
    *tflops = 2.0 * 8.0 * iters * (double)blocks * threads / (best * 1e-3) / 1e12;
    return IGT_OK;
}

int igt_mlp_value_ex_host(igt_handle *h, int B, const double *sN, const double *vN, const double *nn_ctx, const int *net_idx,
                          double *out, int use_tensor_cores)
{
    const int mode = use_tensor_cores;
    auto check = [&]() -> int {
        if (B < 0 || !sN || !vN || !nn_ctx || !out) { h->err = "igt_mlp_value: null argument"; return IGT_EINVAL; }
        if (net_idx && mode != 0 && mode != 2) {
            h->err = "igt_mlp_value: with net_idx the mode must be 0 (per thread) or 2 (cooperative)"; return IGT_EINVAL;
        }
        const int width = value_width(h, net_idx != nullptr);
        if (width == 0) { h->err = "igt_mlp_value: igt_set_mlp was never called"; return IGT_ENOMLP; }
        if (mode == 1 && !h->tc.enabled) { h->err = "igt_mlp_value: tensor-core path needs a 6-128-128-1 network"; return IGT_EINVAL; }
        if (mode == 2 && width > MLP_COOP_W) { h->err = "igt_mlp_value: the cooperative evaluation needs layers <= 128 wide"; return IGT_EINVAL; }
        return net_idx ? check_net_idx(h, B, net_idx, "igt_mlp_value") : IGT_OK;
    };
    return host_call(h, B, check, [&](cudaStream_t st) {
        const size_t nb = B;
        const double *ds, *dv, *dc;
        const int *dnet;
        double *dout;
        Staged a[] = { input(sN, nb, &ds), input(vN, nb, &dv), input(nn_ctx, nb * 4, &dc), input(net_idx, nb, &dnet), output(out, nb * 6, &dout) };
        return staged(h, st, a, [&] {
            const int grid = (int)std::min<size_t>((nb + 255) / 256, (size_t)h->n_sm);
            const MlpNet<double> *nets = (const MlpNet<double> *)h->bank;
            int cs = 0, rc;
            if (mode == 2) {
                if ((rc = acquire_cslot(h, 1, st, &cs))) return rc;
                const int sm = net_idx ? mlp_coop_bank_smem_bytes<double>(256) : mlp_coop_smem_bytes<double>(256);
                auto *k = net_idx ? mlp_coop_kernel<true> : mlp_coop_kernel<false>;
                CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, sm));
                k<<<grid, 256, sm, st>>>(B, ds, dv, dc, dout, cs, dnet, nets);
            } else if (mode) {
                mlp_tc_kernel<<<grid, 256, TC_SMEM_BYTES, st>>>(h->tc, B, ds, dv, dc, dout);
            } else {
                const int width = value_width(h, net_idx != nullptr);
                if ((rc = grow(h, &h->mlp_scratch, &h->mlp_scratch_bytes, (size_t)12 * width * nb * 8, st))) return rc;
                if ((rc = acquire_cslot(h, 1, st, &cs))) return rc;
                auto *k = net_idx ? mlp_ref_kernel<true> : mlp_ref_kernel<false>;
                k<<<(int)((nb + 127) / 128), 128, 0, st>>>(B, ds, dv, dc, dout, (double *)h->mlp_scratch, width, cs, dnet, nets);
            }
            h->launches++;
            CK(cudaGetLastError());
            return end_call(h, st, mode == 1 ? 0 : 2);
        });
    });
}

int igt_mlp_value_host(igt_handle *h, int B, const double *sN, const double *vN, const double *nn_ctx, double *out,
                       int use_tensor_cores)
{
    return igt_mlp_value_ex_host(h, B, sN, vN, nn_ctx, nullptr, out, use_tensor_cores);
}


#ifdef IGT_PHASE_CLOCKS
/* debug builds only: cycle counters of thread 0 of CTA 0 of the last solve launch */
int igt_debug_phase_clocks(igt_handle *h, long long *out16)
{
    if (!h || !out16) return IGT_EINVAL;
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpyFromSymbol(out16, g_phase_clk, 16 * sizeof(long long)));
    return IGT_OK;
}
int igt_debug_round_clocks(igt_handle *h, long long *clk512, int *n512)
{
    if (!h || !clk512 || !n512) return IGT_EINVAL;
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpyFromSymbol(clk512, g_round_clk, 512 * sizeof(long long)));
    CK(cudaMemcpyFromSymbol(n512, g_round_n, 512 * sizeof(int)));
    return IGT_OK;
}
int igt_debug_round_max(igt_handle *h, int *mx512x4)
{
    if (!h || !mx512x4) return IGT_EINVAL;
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpyFromSymbol(mx512x4, g_round_mx, 512 * 4 * sizeof(int)));
    int z[512 * 4] = { 0 };
    CK(cudaMemcpyToSymbol(g_round_mx, z, sizeof(z)));
    return IGT_OK;
}
int igt_debug_cta_clocks(igt_handle *h, long long *clk512, int *rounds512)
{
    if (!h || !clk512 || !rounds512) return IGT_EINVAL;
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpyFromSymbol(clk512, g_cta_clk, 512 * sizeof(long long)));
    CK(cudaMemcpyFromSymbol(rounds512, g_cta_rounds, 512 * sizeof(int)));
    return IGT_OK;
}
int igt_debug_round_phases(igt_handle *h, int *ph512x12)
{
    if (!h || !ph512x12) return IGT_EINVAL;
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpyFromSymbol(ph512x12, g_round_ph, 512 * 12 * sizeof(int)));
    return IGT_OK;
}
#endif

int igt_episode_run_ex_host(igt_handle *h, int E, int steps, int mode, const double *route_desc, const double *curv,
                            const double *z0, const double *u_prev0, const double *enc, const int *net_idx, double *z_cl,
                            double *u_cl, int *solved, float *step_ms)
{
    const int gt_mpc = (mode & IGT_EPISODE_GT_MPC) != 0;
    const bool obca = (mode & IGT_EPISODE_OBCA) != 0;
    auto check = [&]() -> int {
        if (E < 0 || steps < 1 || !route_desc || !curv || !z0 || !u_prev0 || !enc || !z_cl || !u_cl || !solved) {
            h->err = "igt_episode_run: bad argument"; return IGT_EINVAL;
        }
        if (mode & ~(IGT_EPISODE_GT_MPC | IGT_EPISODE_OBCA)) {
            h->err = "igt_episode_run: unknown mode bits (IGT_EPISODE_GT_MPC | IGT_EPISODE_OBCA)"; return IGT_EINVAL;
        }
        if (h->prm.precision != IGT_PREC_F64) { h->err = "igt_episode_run: needs precision f64"; return IGT_EINVAL; }
        if (net_idx && !gt_mpc) { h->err = "igt_episode_run: net_idx needs the IGT_EPISODE_GT_MPC mode bit"; return IGT_EINVAL; }
        if (gt_mpc && !net_idx && value_width(h, false) == 0) { h->err = "igt_episode_run: gt_mpc needs igt_set_mlp"; return IGT_ENOMLP; }
        return net_idx ? check_net_idx(h, E, net_idx, "igt_episode_run") : IGT_OK;
    };
    std::vector<cudaEvent_t> ev;
    const int rc = host_call(h, E, check, [&](cudaStream_t st) {
        const int N = h->prm.N, B = 2 * E, T = steps;
        const size_t nb = B;
        std::vector<int> veh_net;   // both vehicles of episode e plan with network net_idx[e]: expanded once, the glue kernels never see it
        if (net_idx) { veh_net.resize(nb); for (int b = 0; b < B; b++) veh_net[b] = net_idx[b / 2]; }
        // one device block: state, records, solver inputs and two sets of solver outputs (the plans of t and t-1)
        EpisodeBufs eb;
        const int *dnet;
        double *px[2], *pu[2], *pcost[2], *pviol[2];
        int *pst[2], *pit[2];
        Staged a[] = { input(z0, nb * 7, &eb.z), input(u_prev0, nb * 2, &eb.u_prev), input(curv, nb * 3, &eb.curv),
                       input(route_desc, nb * ROUTE_DESC, &eb.rd), input(enc, nb, &eb.enc), input(net_idx ? veh_net.data() : nullptr, nb, &dnet),
                       output(z_cl, nb * (T + 1) * 7, &eb.z_cl), output(u_cl, nb * T * 2, &eb.u_cl), output(solved, nb * T, &eb.solved),
                       device_only(nb * (N + 1) * 2, &eb.obs), device_only(nb * 4, &eb.ctx), device_only(nb * N * 2, &eb.u_init),
                       device_only(obca ? nb * (N + 1) : 0, &eb.obs_psi), device_only(nb, &eb.warm), device_only(nb, &eb.prev_ok),
                       device_only(nb * (N + 1) * 7, &px[0]), device_only(nb * N * 2, &pu[0]), device_only(nb, &pcost[0]), device_only(nb, &pviol[0]),
                       device_only(nb * (N + 1) * 7, &px[1]), device_only(nb * N * 2, &pu[1]), device_only(nb, &pcost[1]), device_only(nb, &pviol[1]),
                       device_only(nb, &pst[0]), device_only(nb, &pit[0]), device_only(nb, &pst[1]), device_only(nb, &pit[1]) };
        return staged(h, st, a, [&] {
            CK(cudaMemsetAsync(eb.prev_ok, 0, nb * 4, st));
            // z_cl[:, :, 0] = z0
            CK(cudaMemcpy2DAsync(eb.z_cl, (size_t)(T + 1) * 7 * 8, eb.z, 7 * 8, 7 * 8, nb, cudaMemcpyDeviceToDevice, st));
            if (step_ms) { ev.resize(T + 1); for (auto &e : ev) CK(cudaEventCreate(&e)); CK(cudaEventRecord(ev[0], st)); }
            const int bs = 128, gs = (B + bs - 1) / bs;
            int cs = 0, rc;
            for (int t = 0; t < T; t++) {
                const int cur = t & 1, prv = cur ^ 1;
                if (obca) episode_pre_kernel<true><<<gs, bs, 0, st>>>(eb, B, N, h->prm.dt, t, gt_mpc, px[prv], pu[prv]);
                else episode_pre_kernel<false><<<gs, bs, 0, st>>>(eb, B, N, h->prm.dt, t, gt_mpc, px[prv], pu[prv]);
                h->launches++;
                const ProbIO io = { eb.z, eb.u_prev, eb.curv, eb.obs, gt_mpc ? eb.ctx : nullptr, eb.u_init, px[cur], pu[cur],
                                    pcost[cur], pviol[cur], pst[cur], pit[cur], eb.obs_psi, eb.warm };
                if ((rc = solve_dev_impl(h, B, io, dnet, st))) return rc;
                if ((rc = acquire_cslot(h, 1, st, &cs))) return rc;
                episode_post_kernel<<<gs, bs, 0, st>>>(eb, B, N, T, t, h->prm.a_min, px[cur], pu[cur], pst[cur], cs);
                h->launches++;
                if (step_ms) CK(cudaEventRecord(ev[t + 1], st));
            }
            CK(cudaGetLastError());
            return end_call(h, st, 2);
        });
    });
    if (rc || ev.empty()) return rc;
    for (int t = 0; t < steps; t++) CK(cudaEventElapsedTime(&step_ms[t], ev[t], ev[t + 1]));
    for (auto &e : ev) cudaEventDestroy(e);
    return IGT_OK;
}

int igt_episode_run_host(igt_handle *h, int E, int steps, int mode, const double *route_desc, const double *curv,
                         const double *z0, const double *u_prev0, const double *enc, double *z_cl, double *u_cl,
                         int *solved, float *step_ms)
{
    return igt_episode_run_ex_host(h, E, steps, mode, route_desc, curv, z0, u_prev0, enc, nullptr, z_cl, u_cl, solved, step_ms);
}

int igt_set_option(igt_handle *h, const char *name, double value)
{
    if (!h || !name) return IGT_EINVAL;
    if (strcmp(name, "tensor_core_mlp") == 0) { h->use_tc = value != 0.0; return IGT_OK; }
    if (strcmp(name, "latency_path") == 0) { h->use_small = value != 0.0; return IGT_OK; }
    h->err = std::string("igt_set_option: unknown option ") + name;
    return IGT_EINVAL;
}

}  // extern "C"
