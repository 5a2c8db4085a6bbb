// igt_abi.cu -- kernels and the extern "C" boundary of libigtmpc.so (see include/igt_mpc.h).
//
// Kernels (all hand-written, sm_100a):
//   solve_kernel<T>       one MPC problem per thread, whole interior-point iLQR on chip + SoA
//                         workspace in HBM (solver_core.cuh); replaces mpc.py:383-406
//   rollout_kernel        fp32 Frenet RK4 rollout + analytic Jacobians (compensated state
//                         accumulation); replaces kinematic_bicycle_model_frenet.py:69-185
//   rollout_euler_kernel  fp32 Cartesian Euler rollout + Jacobians; kinematic_bicycle_model.py:15-50
//   eval_kernel           fp64 cost / max-row-violation of given controls; mpc.py:177-373
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <new>
#include <mutex>

#include "../../include/igt_mpc.h"
#include "solver_core.cuh"
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
template <typename T, bool TC, bool OBCA, bool COOP = false, bool BANK = false>
__global__ void __launch_bounds__(SOLVE_BLOCK, 1) solve_kernel(typename std::conditional<BANK, ProbIONet<T>, ProbIO>::type io, T *ws, long n_slots, long B, Sched sc,
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
    solve_persistent<T, TC, 32, OBCA, COOP, RSTG, BANK>(P, io, ws, slot, B, sc, guess,
                            mlp_scratch ? mlp_scratch + slot * 12 * (long)mlp_width : nullptr, mlp_width, &tc, quota, cs, dyn_smem,
                            RSTG ? dyn_smem + (COOP ? mlp_coop_smem_bytes<T>(SOLVE_BLOCK) : 0) : nullptr);
    if (TC) mlp_tc_teardown(tc);
}

// Latency path for batches of at most one problem per SM (the closed-loop step: B = 2): one CTA per problem,
// its whole workspace in shared memory (stride-1 layout), so the sweeps of the problem's one owner thread run at
// shared-memory latency instead of an L2 round trip per stage; the node phases and the line-search candidates
// are dealt out over the CTA's 256 threads as in the throughput kernel.  Same code, same arithmetic, same results.
template <typename T, bool OBCA>
__global__ void __launch_bounds__(SOLVE_BLOCK, 1) solve_small_kernel(ProbIO io, long B, Sched sc, const double *guess, int cs)
{
    extern __shared__ __align__(16) uint8_t dyn_smem[];
    const DevParams<T> &P = ConstP<T>::get(cs);
    solve_persistent<T, false, 1, OBCA>(P, io, reinterpret_cast<T *>(dyn_smem), 0, B, sc, guess, (T *)nullptr, 0, nullptr, 1, cs);
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
        m = fmax(m, fabs(z[IEY]) - P.ey_lim);
        if (k >= 1) {
            if (obs_psi_) {                                      // OBCA rows in dual-eliminated form (obca.cuh)
                double gd[3];
                m = fmax(m, P.d_min + OBCA_MARGIN - obca_rect_sdist(z[IX], z[IY], z[IPSI], obs[2 * k], obs[2 * k + 1], obs_psi_[p * (N + 1) + k], gd));
            } else {
                double dx = z[IX] - obs[2 * k], dy = z[IY] - obs[2 * k + 1];
                m = fmax(m, P.d_min * P.d_min - dx * dx - dy * dy);
            }
        }
        if (k == N) break;
        double u[2] = { U[(p * N + k) * 2], U[(p * N + k) * 2 + 1] };
        su += u[0] * u[0] + u[1] * u[1];
        m = fmax(m, fmax(P.v_min - z[IV], z[IV] - P.v_max));
        m = fmax(m, fmax(P.a_min - u[0], u[0] - P.a_max));
        m = fmax(m, fabs(u[1]) - P.df_max);
        m = fmax(m, fabs(u[0] - up[0]) - P.da_max);
        m = fmax(m, fabs(u[1] - up[1]) - P.ddf_max);
        if (k == N - 1)
            for (int q = 0; q < P.n_cinf; q++) m = fmax(m, P.cinf_A[q][0] * z[IV] + P.cinf_A[q][1] * u[0] - P.cinf_b[q]);
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
    bool has_mlp = false;
    MlpTcWeights tc = {};              // tensor-core copy of the value network (6-128-128-1 only)
    int use_tc = 0;                    // igt_set_option("tensor_core_mlp", 1): fp32-accurate tcgen05 value term (6-128-128-1 nets)
    bool coop_ok = false;              // every layer <= MLP_COOP_W wide: the exact CTA-cooperative evaluation applies
    int use_small = 1;                 // igt_set_option("latency_path", 0) keeps small batches on the throughput kernel
    int mlp_width = 0;
    // network bank (igt_set_mlp_at): slot 0 is also the network above (Pf / Pd, tc); a solve with net_idx reads the
    // device table `bank` = [MAX_MLP_NETS] MlpNet<double>, then [MAX_MLP_NETS] MlpNet<float>
    std::vector<void *> mlp_bufs[MAX_MLP_NETS];   // device weight buffers of each slot (both precisions)
    MlpNet<double> netd[MAX_MLP_NETS] = {};
    MlpNet<float> netf[MAX_MLP_NETS] = {};
    int net_width[MAX_MLP_NETS] = {};  // widest layer of each slot, 0 = empty
    void *bank = nullptr;
    void *ws = nullptr; size_t ws_bytes = 0;
    void *mlp_scratch = nullptr; size_t mlp_scratch_bytes = 0;
    void *stage = nullptr; size_t stage_bytes = 0;     // device staging for *_host calls
    void *guess = nullptr; size_t guess_bytes = 0;     // cold-start controls [B][N][2] + the work counter
    void *episode = nullptr; size_t episode_bytes = 0; // igt_episode_run_host: state, records, solver inputs / outputs
    int n_sm = 0;
    long long launches = 0;
    std::string err;
    int device = 0;
    // concurrency (see the header): calls on one handle are serialised on the device in call order whatever their
    // streams -- the handle's workspace, guess buffer and work counter are shared by its calls
    std::mutex mu;                     // host-side: one call at a time per handle
    cudaStream_t hstream = nullptr;    // the *_host entry points run on a private non-blocking stream
    void *pin = nullptr; size_t pin_bytes = 0;   // pinned staging block of igt_solve_host (small batches)
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
    for (auto &v : h->mlp_bufs) for (void *b : v) cudaFree(b);
    if (h->bank) cudaFree(h->bank);
    if (h->hstream) cudaStreamDestroy(h->hstream);
    if (h->pin) cudaFreeHost(h->pin);
    if (h->ws) cudaFree(h->ws);
    if (h->mlp_scratch) cudaFree(h->mlp_scratch);
    if (h->stage) cudaFree(h->stage);
    if (h->guess) cudaFree(h->guess);
    if (h->episode) cudaFree(h->episode);
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
    std::lock_guard<std::mutex> lk(h->mu);
    CK(cudaSetDevice(h->device));
    if (h->last_use && h->used) CK(cudaEventSynchronize(h->last_use));   // no kernel of this handle reads the old network
    if (!h->bank) CK(cudaMalloc(&h->bank, MAX_MLP_NETS * (sizeof(MlpNet<double>) + sizeof(MlpNet<float>))));
    h->version[0]++; h->version[1]++;
    for (void *q : h->mlp_bufs[net]) cudaFree(q);
    h->mlp_bufs[net].clear();
    h->net_width[net] = 0;
    MlpNet<double> &nd = h->netd[net];
    MlpNet<float> &nf = h->netf[net];
    nd = MlpNet<double>(); nf = MlpNet<float>();
    std::vector<void *> &bufs = h->mlp_bufs[net];
    nf.n_layers = nd.n_layers = n_layers;
    for (int l = 0; l <= n_layers; l++) nf.dims[l] = nd.dims[l] = dims[l];
    for (int l = 0; l < n_layers; l++) {
        size_t nw = (size_t)dims[l] * dims[l + 1], nb = dims[l + 1];
        std::vector<float> wf(nw), bf(nb);
        for (size_t i = 0; i < nw; i++) wf[i] = (float)W[l][i];
        for (size_t i = 0; i < nb; i++) bf[i] = (float)b[l][i];
        void *dWd, *dbd, *dWf, *dbf;
        CK(cudaMalloc(&dWd, nw * 8)); bufs.push_back(dWd);
        CK(cudaMalloc(&dbd, nb * 8)); bufs.push_back(dbd);
        CK(cudaMalloc(&dWf, nw * 4)); bufs.push_back(dWf);
        CK(cudaMalloc(&dbf, nb * 4)); bufs.push_back(dbf);
        CK(cudaMemcpy(dWd, W[l], nw * 8, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(dbd, b[l], nb * 8, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(dWf, wf.data(), nw * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(dbf, bf.data(), nb * 4, cudaMemcpyHostToDevice));
        nd.W[l] = (const double *)dWd; nd.b[l] = (const double *)dbd;
        nf.W[l] = (const float *)dWf; nf.b[l] = (const float *)dbf;
        // transposed copies [in][out] for the cooperative evaluation (mlp_coop.cuh)
        std::vector<double> wtd(nw); std::vector<float> wtf(nw);
        for (int o = 0; o < dims[l + 1]; o++)
            for (int i = 0; i < dims[l]; i++) { wtd[(size_t)i * dims[l + 1] + o] = W[l][(size_t)o * dims[l] + i]; wtf[(size_t)i * dims[l + 1] + o] = (float)W[l][(size_t)o * dims[l] + i]; }
        void *dTd, *dTf;
        CK(cudaMalloc(&dTd, nw * 8)); bufs.push_back(dTd);
        CK(cudaMalloc(&dTf, nw * 4)); bufs.push_back(dTf);
        CK(cudaMemcpy(dTd, wtd.data(), nw * 8, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(dTf, wtf.data(), nw * 4, cudaMemcpyHostToDevice));
        nd.Wt[l] = (const double *)dTd; nf.Wt[l] = (const float *)dTf;
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
    h->mlp_width = width;
    h->Pf.n_layers = h->Pd.n_layers = n_layers;
    for (int l = 0; l <= n_layers; l++) h->Pf.dims[l] = h->Pd.dims[l] = dims[l];
    for (int l = 0; l < n_layers; l++) {
        h->Pd.W[l] = nd.W[l]; h->Pd.b[l] = nd.b[l]; h->Pd.Wt[l] = nd.Wt[l];
        h->Pf.W[l] = nf.W[l]; h->Pf.b[l] = nf.b[l]; h->Pf.Wt[l] = nf.Wt[l];
    }
    h->coop_ok = width <= MLP_COOP_W;
    for (int i = 0; i < 36; i++) { h->Pd.Wn[i] = Wn[i]; h->Pf.Wn[i] = (float)Wn[i]; }
    for (int i = 0; i < 6; i++) { h->Pd.mu_f[i] = mu_f[i]; h->Pf.mu_f[i] = (float)mu_f[i]; }
    h->Pd.sigma_t = sigma_t; h->Pd.mu_t = mu_t; h->Pf.sigma_t = (float)sigma_t; h->Pf.mu_t = (float)mu_t;
    h->has_mlp = true;
    h->tc.enabled = 0;
    if (n_layers == 3 && dims[1] == MLP_H && dims[2] == MLP_H) {
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
        void *dblob, *dw1, *db1, *db2, *dw3;
        CK(cudaMalloc(&dblob, blob.size())); bufs.push_back(dblob);
        CK(cudaMalloc(&dw1, w1eff.size() * 4)); bufs.push_back(dw1);
        CK(cudaMalloc(&db1, MLP_H * 4)); bufs.push_back(db1);
        CK(cudaMalloc(&db2, MLP_H * 4)); bufs.push_back(db2);
        CK(cudaMalloc(&dw3, MLP_H * 4)); bufs.push_back(dw3);
        CK(cudaMemcpy(dblob, blob.data(), blob.size(), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(dw1, w1eff.data(), w1eff.size() * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(db1, b1eff.data(), MLP_H * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(db2, b2.data(), MLP_H * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(dw3, w3.data(), MLP_H * 4, cudaMemcpyHostToDevice));
        h->tc.w2_splits = (const uint8_t *)dblob; h->tc.w1eff = (const float *)dw1; h->tc.b1eff = (const float *)db1;
        h->tc.b2 = (const float *)db2; h->tc.w3 = (const float *)dw3;
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

// Bank calls: every index names a loaded slot (checked on the host before anything is launched, under h->mu, so that
// a concurrent igt_set_mlp_at cannot empty a slot between the check and the launch); the widest network
// of the bank sizes the per-thread scratch, and the cooperative evaluation applies when every slot is <= 128 wide.
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
static ProbIONet<float> iob_f32(const ProbIONet<double> &io, const igt_handle *h)
{
    ProbIONet<float> r;
    static_cast<ProbIO &>(r) = io;
    r.net_idx = io.net_idx;
    r.nets = (const MlpNet<float> *)((const char *)h->bank + sizeof(h->netd));
    return r;
}
static int bank_width(const igt_handle *h)
{
    int w = 0;
    for (int k = 0; k < MAX_MLP_NETS; k++) if (h->net_width[k] > w) w = h->net_width[k];
    return w;
}

static int rollout_dev_impl(igt_handle *h, int B, const float *z0, const float *u, const float *curv, float *z,
                            float *A, float *Bm, int model, cudaStream_t st)
{
    if (B < 0 || !z0 || !u || !z || (model == 0 && !curv) || ((A == nullptr) != (Bm == nullptr)) ||
        (model != 0 && model != 1)) { h->err = "igt_rollout: bad argument"; return IGT_EINVAL; }
    if (B == 0) return IGT_OK;
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
    return rollout_dev_impl(h, B, z0, u, curv, z, A, Bm, model, (cudaStream_t)stream);
}

int igt_rollout_host(igt_handle *h, int B, const float *z0, const float *u, const float *curv, float *z,
                     float *A, float *Bm, int model)
{
    if (!h) return IGT_EINVAL;
    if (B < 0 || !z0 || !u || !z || (model == 0 && !curv)) { h->err = "igt_rollout: bad argument"; return IGT_EINVAL; }
    if (B == 0) return IGT_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    { int rc0 = begin_call(h, nullptr); if (rc0) return rc0; }
    const int N = h->prm.N, nz = model == 0 ? 7 : 4;
    size_t n_z0 = (size_t)B * nz, n_u = (size_t)B * N * 2, n_c = (size_t)B * 3, n_z = (size_t)B * (N + 1) * nz;
    size_t n_A = A ? (size_t)B * N * nz * nz : 0, n_B = A ? (size_t)B * N * nz * 2 : 0;
    size_t total = (n_z0 + n_u + n_c + n_z + n_A + n_B) * sizeof(float);
    int rc = grow(h, &h->stage, &h->stage_bytes, total, nullptr);
    if (rc) return rc;
    float *d = (float *)h->stage;
    float *dz0 = d, *du = dz0 + n_z0, *dc = du + n_u, *dz = dc + n_c, *dA = dz + n_z, *dB = dA + n_A;
    CK(cudaMemcpy(dz0, z0, n_z0 * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(du, u, n_u * 4, cudaMemcpyHostToDevice));
    if (model == 0) CK(cudaMemcpy(dc, curv, n_c * 4, cudaMemcpyHostToDevice));
    rc = rollout_dev_impl(h, B, dz0, du, dc, dz, A ? dA : nullptr, A ? dB : nullptr, model, nullptr);
    if (rc) return rc;
    CK(cudaMemcpy(z, dz, n_z * 4, cudaMemcpyDeviceToHost));
    if (A) { CK(cudaMemcpy(A, dA, n_A * 4, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(Bm, dB, n_B * 4, cudaMemcpyDeviceToHost)); }
    return IGT_OK;
}

static int solve_dev_impl(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                          const double *obs_xy, const double *obs_psi, const double *nn_ctx, const double *u_init,
                          double *x, double *u, double *cost, double *viol, int *status, int *iters, cudaStream_t st,
                          const int *warm = nullptr, const int *net_idx = nullptr)
{
    if (B < 0 || !x0 || !u_prev || !curv || !obs_xy || !x || !u || !cost || !viol || !status || !iters) {
        h->err = "igt_solve: null argument"; return IGT_EINVAL;
    }
    const bool bank = net_idx != nullptr;
    if (bank && !nn_ctx) { h->err = "igt_solve: net_idx needs nn_ctx (gt_mpc)"; return IGT_EINVAL; }
    if (bank && bank_width(h) == 0) { h->err = "igt_solve: net_idx given but no network was loaded"; return IGT_ENOMLP; }
    if (nn_ctx && !bank && !h->has_mlp) { h->err = "igt_solve: nn_ctx given but igt_set_mlp was never called"; return IGT_ENOMLP; }
    const bool f64 = h->prm.precision == IGT_PREC_F64, obca = obs_psi != nullptr;
    if (obca && !f64) { h->err = "igt_solve: the OBCA collision rows (obs_psi) need precision f64"; return IGT_EINVAL; }
    if (B == 0) return IGT_OK;
    int rc = begin_call(h, st), cs = 0;
    if (rc) return rc;
    WsLayout L; L.init(h->prm.N, h->prm.n_cinf, obca ? NGE_OBCA : NGE, obca ? NHE_OBCA : NHE);
    size_t esz = f64 ? 8 : 4;
    // latency path: at most one problem per SM and a workspace that fits shared memory next to the work lists
    const size_t small_smem = (size_t)L.total * esz;
    const bool small = h->use_small && !nn_ctx && B <= h->n_sm && small_smem <= 200 * 1024;
    // persistent lanes: one CTA of SOLVE_BLOCK threads per SM.  A batch smaller than the machine is spread
    // over all SMs, a whole number of warps each: `quota` threads per CTA fetch problems, the rest of
    // the CTA only helps in the CTA-wide phases (and adopts stragglers in the tail).
    const int bs = SOLVE_BLOCK;
    long n_cta = ((long)B + 31) / 32;
    if (n_cta > h->n_sm) n_cta = h->n_sm;
    long per_cta = ((long)B + n_cta - 1) / n_cta;
    int quota = (int)((per_cta + 31) / 32 * 32);
    if (quota > bs) quota = bs;
    long n_slots = n_cta * bs;
    rc = small ? IGT_OK : grow(h, &h->ws, &h->ws_bytes, (size_t)L.total * n_slots * esz, st);
    if (rc) return rc;
    // (OBCA + gt_mpc: per-thread value term; a bank: exact evaluation whatever tensor_core_mlp says)
    const bool use_tc = nn_ctx && !bank && h->tc.enabled && h->use_tc && !obca;
    const int width = bank ? bank_width(h) : h->mlp_width;
    const bool use_coop = nn_ctx && !use_tc && f64 && (bank ? width <= MLP_COOP_W : h->coop_ok) && !obca;
    if (nn_ctx && !use_tc && !use_coop) {                                 // per-thread evaluation: activations in HBM
        rc = grow(h, &h->mlp_scratch, &h->mlp_scratch_bytes, (size_t)12 * width * n_slots * esz, st);
        if (rc) return rc;
    }
    // scheduler block (the work counter), then the cold-start guesses
    const size_t off_guess = 256;
    rc = grow(h, &h->guess, &h->guess_bytes, off_guess + (size_t)B * h->prm.N * 2 * sizeof(double), st);
    if (rc) return rc;
    char *sb = (char *)h->guess;
    Sched sc;
    sc.counter = (unsigned long long *)sb;
    double *guess = (double *)(sb + off_guess);
    rc = acquire_cslot(h, f64 ? 1 : 0, st, &cs);
    if (rc) return rc;
    CK(cudaMemsetAsync(sb, 0, 256, st));
    ProbIO io = { x0, u_prev, curv, obs_xy, nn_ctx, u_init, x, u, cost, viol, status, iters };
    io.obs_psi = obs_psi;
    io.warm = warm;
    ProbIONet<double> iob;   // (the bank kernels' inputs: the f32 one reinterprets nets, same layout)
    static_cast<ProbIO &>(iob) = io;
    iob.net_idx = net_idx;
    iob.nets = (const MlpNet<double> *)h->bank;
    if (!u_init || warm) {
        int gbs = 128, ggs = (B + gbs - 1) / gbs;
        if (obca) guess_kernel<double, true><<<ggs, gbs, 0, st>>>(io, B, guess, cs);
        else if (f64) guess_kernel<double, false><<<ggs, gbs, 0, st>>>(io, B, guess, cs);
        else guess_kernel<float, false><<<ggs, gbs, 0, st>>>(io, B, guess, cs);
        h->launches++;
    }
    int gs = (int)(n_slots / bs);
    if (small) {
        if (obca) {
            CK(cudaFuncSetAttribute(solve_small_kernel<double, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small_smem));
            solve_small_kernel<double, true><<<B, bs, small_smem, st>>>(io, B, sc, guess, cs);
        } else if (f64) {
            CK(cudaFuncSetAttribute(solve_small_kernel<double, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small_smem));
            solve_small_kernel<double, false><<<B, bs, small_smem, st>>>(io, B, sc, guess, cs);
        } else {
            CK(cudaFuncSetAttribute(solve_small_kernel<float, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small_smem));
            solve_small_kernel<float, false><<<B, bs, small_smem, st>>>(io, B, sc, guess, cs);
        }
    } else if (bank) {
        // gt_mpc with the network bank: the same kernels' BANK instantiations (problems with a bad index get
        // IGT_STATUS_BAD_NET); cooperative value term where every network fits it, else per thread
        double *scr = (double *)h->mlp_scratch;
        const int rsm = IGT_RSTG ? RSTG_SLOTS * SOLVE_BLOCK * (int)esz : 0;
        if (use_coop) {
            const int sm = mlp_coop_bank_smem_bytes<double>(SOLVE_BLOCK);
            CK(cudaFuncSetAttribute(solve_kernel<double, false, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm));
            solve_kernel<double, false, false, true, true><<<gs, bs, sm, st>>>(iob, (double *)h->ws, n_slots, B, sc, guess, nullptr, width, h->tc, quota, cs);
        } else if (obca) {
            CK(cudaFuncSetAttribute(solve_kernel<double, false, true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, rsm));
            solve_kernel<double, false, true, false, true><<<gs, bs, rsm, st>>>(iob, (double *)h->ws, n_slots, B, sc, guess, scr, width, h->tc, quota, cs);
        } else if (f64) {
            CK(cudaFuncSetAttribute(solve_kernel<double, false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, rsm));
            solve_kernel<double, false, false, false, true><<<gs, bs, rsm, st>>>(iob, (double *)h->ws, n_slots, B, sc, guess, scr, width, h->tc, quota, cs);
        } else {
            CK(cudaFuncSetAttribute(solve_kernel<float, false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, rsm));
            solve_kernel<float, false, false, false, true><<<gs, bs, rsm, st>>>(iob_f32(iob, h), (float *)h->ws, n_slots, B, sc, guess, (float *)h->mlp_scratch, width, h->tc, quota, cs);
        }
    } else if (use_tc) {
        if (f64) {
            CK(cudaFuncSetAttribute(solve_kernel<double, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_BYTES));
            solve_kernel<double, true, false><<<gs, bs, TC_SMEM_BYTES, st>>>(io, (double *)h->ws, n_slots, B, sc, guess, nullptr, h->mlp_width, h->tc, quota, cs);
        } else {
            CK(cudaFuncSetAttribute(solve_kernel<float, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_BYTES));
            solve_kernel<float, true, false><<<gs, bs, TC_SMEM_BYTES, st>>>(io, (float *)h->ws, n_slots, B, sc, guess, nullptr, h->mlp_width, h->tc, quota, cs);
        }
    } else if (use_coop) {
        // gt_mpc, exact value term: CTA-cooperative evaluation, one warp per evaluation (mlp_coop.cuh)
        const int sm = mlp_coop_smem_bytes<double>(SOLVE_BLOCK);
        CK(cudaFuncSetAttribute(solve_kernel<double, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm));
        solve_kernel<double, false, false, true><<<gs, bs, sm, st>>>(io, (double *)h->ws, n_slots, B, sc, guess, nullptr, h->mlp_width, h->tc, quota, cs);
    } else if (obca) {
        const int rsm = IGT_RSTG ? RSTG_SLOTS * SOLVE_BLOCK * 8 : 0;
        CK(cudaFuncSetAttribute(solve_kernel<double, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, rsm));
        solve_kernel<double, false, true><<<gs, bs, rsm, st>>>(io, (double *)h->ws, n_slots, B, sc, guess,
                                                               nn_ctx ? (double *)h->mlp_scratch : nullptr, h->mlp_width, h->tc, quota, cs);
    } else if (f64) {
        const int rsm = IGT_RSTG ? RSTG_SLOTS * SOLVE_BLOCK * 8 : 0;
        CK(cudaFuncSetAttribute(solve_kernel<double, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, rsm));
        solve_kernel<double, false, false><<<gs, bs, rsm, st>>>(io, (double *)h->ws, n_slots, B, sc, guess,
                                                                nn_ctx ? (double *)h->mlp_scratch : nullptr, h->mlp_width, h->tc, quota, cs);
    } else {
        const int rsm = IGT_RSTG ? RSTG_SLOTS * SOLVE_BLOCK * 4 : 0;
        CK(cudaFuncSetAttribute(solve_kernel<float, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, rsm));
        solve_kernel<float, false, false><<<gs, bs, rsm, st>>>(io, (float *)h->ws, n_slots, B, sc, guess,
                                                               nn_ctx ? (float *)h->mlp_scratch : nullptr, h->mlp_width, h->tc, quota, cs);
    }
    h->launches++;
    CK(cudaGetLastError());
    return end_call(h, st, f64 ? 2 : 1);
}

int igt_solve_ex_dev(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                     const double *obs_xy, const double *obs_psi, const double *nn_ctx, const int *net_idx, const double *u_init,
                     double *x, double *u, double *cost, double *viol, int *status, int *iters, void *stream)
{
    if (!h) return IGT_EINVAL;
    std::lock_guard<std::mutex> lk(h->mu);
    return solve_dev_impl(h, B, x0, u_prev, curv, obs_xy, obs_psi, nn_ctx, u_init, x, u, cost, viol, status, iters,
                          (cudaStream_t)stream, nullptr, net_idx);
}

int igt_solve_dev(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                  const double *obs_xy, const double *obs_psi, const double *nn_ctx, const double *u_init, double *x,
                  double *u, double *cost, double *viol, int *status, int *iters, void *stream)
{
    return igt_solve_ex_dev(h, B, x0, u_prev, curv, obs_xy, obs_psi, nn_ctx, nullptr, u_init, x, u, cost, viol, status, iters, stream);
}

// Host-pointer solve.  All inputs travel in ONE host-to-device copy and all outputs in ONE device-to-host copy on
// the handle's own non-blocking stream: small batches (a closed-loop step solves B = 2) are packed into pinned
// staging blocks first; large batches are copied array by array straight from the caller's (ideally pinned)
// memory -- packing 100 MB on the host would cost more than the copies.
int igt_solve_ex_host(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                      const double *obs_xy, const double *obs_psi, const double *nn_ctx, const int *net_idx, const double *u_init,
                      double *x, double *u, double *cost, double *viol, int *status, int *iters)
{
    if (!h) return IGT_EINVAL;
    if (B < 0 || !x0 || !u_prev || !curv || !obs_xy || !x || !u || !cost || !viol || !status || !iters) {
        h->err = "igt_solve: null argument"; return IGT_EINVAL;
    }
    if (net_idx && !nn_ctx) { h->err = "igt_solve: net_idx needs nn_ctx (gt_mpc)"; return IGT_EINVAL; }
    if (B == 0) return IGT_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    if (net_idx) { const int rc0 = check_net_idx(h, B, net_idx, "igt_solve"); if (rc0) return rc0; }
    CK(cudaSetDevice(h->device));
    if (!h->hstream) CK(cudaStreamCreateWithFlags(&h->hstream, cudaStreamNonBlocking));
    cudaStream_t st = h->hstream;
    int rc = begin_call(h, st);
    if (rc) return rc;
    const int N = h->prm.N;
    size_t nb = (size_t)B;
    size_t n_x0 = nb * 7, n_up = nb * 2, n_c = nb * 3, n_o = nb * (N + 1) * 2, n_ctx = nn_ctx ? nb * 4 : 0;
    size_t n_ui = u_init ? nb * N * 2 : 0, n_x = nb * (N + 1) * 7, n_u = nb * N * 2, n_op = obs_psi ? nb * (N + 1) : 0;
    size_t n_in = n_x0 + n_up + n_c + n_o + n_ctx + n_ui + n_op, n_out = n_x + n_u + 2 * nb;
    size_t in_bytes = n_in * 8, out_bytes = n_out * 8 + 2 * nb * 4, total = in_bytes + out_bytes;
    rc = grow(h, &h->stage, &h->stage_bytes, total + (net_idx ? nb * 4 : 0), st);
    if (rc) return rc;
    int *dnet = (int *)((char *)h->stage + total);                     // net_idx: after the outputs, copied on its own
    if (net_idx) CK(cudaMemcpyAsync(dnet, net_idx, nb * 4, cudaMemcpyHostToDevice, st));
    double *d = (double *)h->stage;
    double *dx0 = d, *dup = dx0 + n_x0, *dc = dup + n_up, *dob = dc + n_c, *dctx = dob + n_o, *dui = dctx + n_ctx;
    double *dop = dui + n_ui;
    double *dx = dop + n_op, *du = dx + n_x, *dcost = du + n_u, *dviol = dcost + nb;
    int *dst = (int *)(dviol + nb), *dit = dst + nb;
    const bool packed = total <= (size_t)1 << 20;
    if (packed) {
        if (h->pin_bytes < total) {
            if (h->pin) { CK(cudaStreamSynchronize(st)); CK(cudaFreeHost(h->pin)); h->pin = nullptr; h->pin_bytes = 0; }
            CK(cudaHostAlloc(&h->pin, total, cudaHostAllocDefault));
            h->pin_bytes = total;
        }
        double *p = (double *)h->pin;
        memcpy(p, x0, n_x0 * 8); p += n_x0;
        memcpy(p, u_prev, n_up * 8); p += n_up;
        memcpy(p, curv, n_c * 8); p += n_c;
        memcpy(p, obs_xy, n_o * 8); p += n_o;
        if (nn_ctx) { memcpy(p, nn_ctx, n_ctx * 8); p += n_ctx; }
        if (u_init) { memcpy(p, u_init, n_ui * 8); p += n_ui; }
        if (obs_psi) { memcpy(p, obs_psi, n_op * 8); p += n_op; }
        CK(cudaMemcpyAsync(dx0, h->pin, in_bytes, cudaMemcpyHostToDevice, st));
    } else {
        CK(cudaMemcpyAsync(dx0, x0, n_x0 * 8, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(dup, u_prev, n_up * 8, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(dc, curv, n_c * 8, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(dob, obs_xy, n_o * 8, cudaMemcpyHostToDevice, st));
        if (nn_ctx) CK(cudaMemcpyAsync(dctx, nn_ctx, n_ctx * 8, cudaMemcpyHostToDevice, st));
        if (u_init) CK(cudaMemcpyAsync(dui, u_init, n_ui * 8, cudaMemcpyHostToDevice, st));
        if (obs_psi) CK(cudaMemcpyAsync(dop, obs_psi, n_op * 8, cudaMemcpyHostToDevice, st));
    }
    rc = solve_dev_impl(h, B, dx0, dup, dc, dob, obs_psi ? dop : nullptr, nn_ctx ? dctx : nullptr, u_init ? dui : nullptr,
                        dx, du, dcost, dviol, dst, dit, st, nullptr, net_idx ? dnet : nullptr);
    if (rc) return rc;
    if (packed) {
        char *q = (char *)h->pin + in_bytes;
        CK(cudaMemcpyAsync(q, dx, out_bytes, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        memcpy(x, q, n_x * 8); q += n_x * 8;
        memcpy(u, q, n_u * 8); q += n_u * 8;
        memcpy(cost, q, nb * 8); q += nb * 8;
        memcpy(viol, q, nb * 8); q += nb * 8;
        memcpy(status, q, nb * 4); q += nb * 4;
        memcpy(iters, q, nb * 4);
    } else {
        CK(cudaMemcpyAsync(x, dx, n_x * 8, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(u, du, n_u * 8, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(cost, dcost, nb * 8, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(viol, dviol, nb * 8, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(status, dst, nb * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(iters, dit, nb * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    return IGT_OK;
}

int igt_solve_host(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                   const double *obs_xy, const double *obs_psi, const double *nn_ctx, const double *u_init, double *x,
                   double *u, double *cost, double *viol, int *status, int *iters)
{
    return igt_solve_ex_host(h, B, x0, u_prev, curv, obs_xy, obs_psi, nn_ctx, nullptr, u_init, x, u, cost, viol, status, iters);
}

int igt_eval_ex_host(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                     const double *obs_xy, const double *obs_psi, const double *nn_ctx, const int *net_idx, const double *u,
                     double *cost, double *viol, double *z)
{
    if (!h) return IGT_EINVAL;
    if (B < 0 || !x0 || !u_prev || !curv || !obs_xy || !u || !cost || !viol) { h->err = "igt_eval: null argument"; return IGT_EINVAL; }
    if (net_idx && !nn_ctx) { h->err = "igt_eval: net_idx needs nn_ctx (gt_mpc)"; return IGT_EINVAL; }
    if (nn_ctx && !net_idx && !h->has_mlp) { h->err = "igt_eval: nn_ctx given but igt_set_mlp was never called"; return IGT_ENOMLP; }
    if (B == 0) return IGT_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    if (net_idx) { const int rc0 = check_net_idx(h, B, net_idx, "igt_eval"); if (rc0) return rc0; }
    int cs = 0;
    { int rc0 = begin_call(h, nullptr); if (rc0) return rc0; }
    const int N = h->prm.N;
    size_t nb = (size_t)B;
    size_t n_x0 = nb * 7, n_up = nb * 2, n_c = nb * 3, n_o = nb * (N + 1) * 2, n_ctx = nn_ctx ? nb * 4 : 0;
    size_t n_u = nb * N * 2, n_z = nb * (N + 1) * 7, n_op = obs_psi ? nb * (N + 1) : 0;
    size_t total = (n_x0 + n_up + n_c + n_o + n_ctx + n_u + n_z + 2 * nb + n_op) * 8;
    int rc = grow(h, &h->stage, &h->stage_bytes, total + (net_idx ? nb * 4 : 0), nullptr);
    if (rc) return rc;
    const int width = net_idx ? bank_width(h) : h->mlp_width;
    if (nn_ctx) { rc = grow(h, &h->mlp_scratch, &h->mlp_scratch_bytes, (size_t)12 * width * B * 8, nullptr); if (rc) return rc; }
    int *dnet = (int *)((char *)h->stage + total);
    if (net_idx) CK(cudaMemcpy(dnet, net_idx, nb * 4, cudaMemcpyHostToDevice));
    double *d = (double *)h->stage;
    double *dx0 = d, *dup = dx0 + n_x0, *dc = dup + n_up, *dob = dc + n_c, *dctx = dob + n_o, *du = dctx + n_ctx;
    double *dz = du + n_u, *dcost = dz + n_z, *dviol = dcost + nb, *dop = dviol + nb;
    if (obs_psi) CK(cudaMemcpy(dop, obs_psi, n_op * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dx0, x0, n_x0 * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dup, u_prev, n_up * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dc, curv, n_c * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dob, obs_xy, n_o * 8, cudaMemcpyHostToDevice));
    if (nn_ctx) CK(cudaMemcpy(dctx, nn_ctx, n_ctx * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(du, u, n_u * 8, cudaMemcpyHostToDevice));
    rc = acquire_cslot(h, 1, nullptr, &cs);
    if (rc) return rc;
    int bs = 128, gs = (B + bs - 1) / bs;
    if (net_idx)
        eval_kernel<true><<<gs, bs>>>(B, dx0, dup, dc, dob, dctx, du, dcost, dviol, dz, (double *)h->mlp_scratch, width, cs,
                                      obs_psi ? dop : nullptr, dnet, (const MlpNet<double> *)h->bank);
    else
        eval_kernel<false><<<gs, bs>>>(B, dx0, dup, dc, dob, nn_ctx ? dctx : nullptr, du, dcost, dviol, dz,
                                       nn_ctx ? (double *)h->mlp_scratch : nullptr, h->mlp_width, cs, obs_psi ? dop : nullptr, nullptr, nullptr);
    h->launches++;
    CK(cudaGetLastError());
    rc = end_call(h, nullptr, 2);
    if (rc) return rc;
    CK(cudaMemcpy(cost, dcost, nb * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(viol, dviol, nb * 8, cudaMemcpyDeviceToHost));
    if (z) CK(cudaMemcpy(z, dz, n_z * 8, cudaMemcpyDeviceToHost));
    return IGT_OK;
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
    if (!h) return IGT_EINVAL;
    if (B < 0 || !sN || !vN || !nn_ctx || !out) { h->err = "igt_mlp_value: null argument"; return IGT_EINVAL; }
    if (net_idx && use_tensor_cores != 0 && use_tensor_cores != 2) {
        h->err = "igt_mlp_value: with net_idx the mode must be 0 (per thread) or 2 (cooperative)"; return IGT_EINVAL;
    }
    std::lock_guard<std::mutex> lk(h->mu);   // (the bank state below is read under the lock: igt_set_mlp_at takes it)
    const int width = net_idx ? bank_width(h) : h->mlp_width;
    if (net_idx ? width == 0 : !h->has_mlp) { h->err = "igt_mlp_value: igt_set_mlp was never called"; return IGT_ENOMLP; }
    if (use_tensor_cores == 1 && !h->tc.enabled) { h->err = "igt_mlp_value: tensor-core path needs a 6-128-128-1 network"; return IGT_EINVAL; }
    if (use_tensor_cores == 2 && (net_idx ? width > MLP_COOP_W : !h->coop_ok)) {
        h->err = "igt_mlp_value: the cooperative evaluation needs layers <= 128 wide"; return IGT_EINVAL;
    }
    if (B == 0) return IGT_OK;
    if (net_idx) { const int rc0 = check_net_idx(h, B, net_idx, "igt_mlp_value"); if (rc0) return rc0; }
    int cs = 0;
    int rc = begin_call(h, nullptr);
    if (rc) return rc;
    size_t nb = (size_t)B, total = (nb * 2 + nb * 4 + nb * 6) * 8;
    rc = grow(h, &h->stage, &h->stage_bytes, total + (net_idx ? nb * 4 : 0), nullptr);
    if (rc) return rc;
    double *ds = (double *)h->stage, *dv = ds + nb, *dc = dv + nb, *dout = dc + nb * 4;
    int *dnet = (int *)((char *)h->stage + total);
    if (net_idx) CK(cudaMemcpy(dnet, net_idx, nb * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ds, sN, nb * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dv, vN, nb * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dc, nn_ctx, nb * 32, cudaMemcpyHostToDevice));
    if (use_tensor_cores == 2) {
        rc = acquire_cslot(h, 1, nullptr, &cs);
        if (rc) return rc;
        int grid = (int)((nb + 255) / 256);
        if (grid > h->n_sm) grid = h->n_sm;
        if (net_idx) {
            const int sm = mlp_coop_bank_smem_bytes<double>(256);
            CK(cudaFuncSetAttribute(mlp_coop_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm));
            mlp_coop_kernel<true><<<grid, 256, sm>>>(B, ds, dv, dc, dout, cs, dnet, (const MlpNet<double> *)h->bank);
        } else {
            const int sm = mlp_coop_smem_bytes<double>(256);
            CK(cudaFuncSetAttribute(mlp_coop_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm));
            mlp_coop_kernel<false><<<grid, 256, sm>>>(B, ds, dv, dc, dout, cs, nullptr, nullptr);
        }
    } else if (use_tensor_cores) {
        int grid = (int)((nb + 255) / 256);
        if (grid > h->n_sm) grid = h->n_sm;
        mlp_tc_kernel<<<grid, 256, TC_SMEM_BYTES>>>(h->tc, B, ds, dv, dc, dout);
    } else {
        rc = grow(h, &h->mlp_scratch, &h->mlp_scratch_bytes, (size_t)12 * width * nb * 8, nullptr);
        if (rc) return rc;
        rc = acquire_cslot(h, 1, nullptr, &cs);
        if (rc) return rc;
        if (net_idx) mlp_ref_kernel<true><<<(int)((nb + 127) / 128), 128>>>(B, ds, dv, dc, dout, (double *)h->mlp_scratch, width, cs, dnet, (const MlpNet<double> *)h->bank);
        else mlp_ref_kernel<false><<<(int)((nb + 127) / 128), 128>>>(B, ds, dv, dc, dout, (double *)h->mlp_scratch, width, cs, nullptr, nullptr);
    }
    h->launches++;
    CK(cudaGetLastError());
    rc = end_call(h, nullptr, use_tensor_cores == 1 ? 0 : 2);
    if (rc) return rc;
    CK(cudaMemcpy(out, dout, nb * 48, cudaMemcpyDeviceToHost));
    return IGT_OK;
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
    if (!h) return IGT_EINVAL;
    if (E < 0 || steps < 1 || !route_desc || !curv || !z0 || !u_prev0 || !enc || !z_cl || !u_cl || !solved) {
        h->err = "igt_episode_run: bad argument"; return IGT_EINVAL;
    }
    if (mode & ~(IGT_EPISODE_GT_MPC | IGT_EPISODE_OBCA)) {
        h->err = "igt_episode_run: unknown mode bits (IGT_EPISODE_GT_MPC | IGT_EPISODE_OBCA)"; return IGT_EINVAL;
    }
    const int gt_mpc = (mode & IGT_EPISODE_GT_MPC) != 0;
    const bool obca = (mode & IGT_EPISODE_OBCA) != 0;
    if (h->prm.precision != IGT_PREC_F64) { h->err = "igt_episode_run: needs precision f64"; return IGT_EINVAL; }
    if (net_idx && !gt_mpc) { h->err = "igt_episode_run: net_idx needs the IGT_EPISODE_GT_MPC mode bit"; return IGT_EINVAL; }
    if (gt_mpc && !net_idx && !h->has_mlp) { h->err = "igt_episode_run: gt_mpc needs igt_set_mlp"; return IGT_ENOMLP; }
    if (E == 0) return IGT_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    if (net_idx) { const int rc0 = check_net_idx(h, E, net_idx, "igt_episode_run"); if (rc0) return rc0; }
    CK(cudaSetDevice(h->device));
    if (!h->hstream) CK(cudaStreamCreateWithFlags(&h->hstream, cudaStreamNonBlocking));
    cudaStream_t st = h->hstream;
    int rc = begin_call(h, st);
    if (rc) return rc;
    const int N = h->prm.N, B = 2 * E, T = steps;
    const size_t nb = (size_t)B;
    // one device block: state, records, solver inputs and two sets of solver outputs (the plans of t and t-1)
    const size_t n_z = nb * 7, n_up = nb * 2, n_cv = nb * 3, n_rd = nb * ROUTE_DESC, n_en = nb, n_obs = nb * (N + 1) * 2,
                 n_ctx = nb * 4, n_ui = nb * N * 2, n_zcl = nb * (T + 1) * 7, n_ucl = nb * T * 2, n_x = nb * (N + 1) * 7,
                 n_u = nb * N * 2, n_op = obca ? nb * (N + 1) : 0;
    const size_t n_dbl = n_z + n_up + n_cv + n_rd + n_en + n_obs + n_ctx + n_ui + n_zcl + n_ucl + 2 * (n_x + n_u + 2 * nb) + n_op;
    const size_t n_int = nb /*warm*/ + nb /*prev_ok*/ + nb * T /*solved*/ + 2 * 2 * nb /*status, iters x2*/ + (net_idx ? nb : 0);
    rc = grow(h, &h->episode, &h->episode_bytes, n_dbl * 8 + n_int * 4, st);
    if (rc) return rc;
    double *d = (double *)h->episode;
    EpisodeBufs eb;
    eb.z = d; d += n_z; eb.u_prev = d; d += n_up;
    double *dcv = d; d += n_cv; double *drd = d; d += n_rd; double *den = d; d += n_en;
    eb.curv = dcv; eb.rd = drd; eb.enc = den;
    eb.obs = d; d += n_obs; eb.ctx = d; d += n_ctx; eb.u_init = d; d += n_ui;
    eb.z_cl = d; d += n_zcl; eb.u_cl = d; d += n_ucl;
    double *px[2], *pu[2], *pcost[2], *pviol[2];
    for (int i = 0; i < 2; i++) { px[i] = d; d += n_x; pu[i] = d; d += n_u; pcost[i] = d; d += nb; pviol[i] = d; d += nb; }
    eb.obs_psi = obca ? d : nullptr; d += n_op;
    int *ip = (int *)d;
    eb.warm = ip; ip += nb; eb.prev_ok = ip; ip += nb; eb.solved = ip; ip += nb * T;
    int *pst[2], *pit[2];
    for (int i = 0; i < 2; i++) { pst[i] = ip; ip += nb; pit[i] = ip; ip += nb; }
    int *dnet = net_idx ? ip : nullptr;
    std::vector<int> veh_net;
    if (net_idx) {   // both vehicles of episode e plan with network net_idx[e]: expanded once, the glue kernels never see it
        veh_net.resize(nb);
        for (int b = 0; b < B; b++) veh_net[b] = net_idx[b / 2];
        CK(cudaMemcpyAsync(dnet, veh_net.data(), nb * 4, cudaMemcpyHostToDevice, st));
    }
    CK(cudaMemcpyAsync(eb.z, z0, n_z * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(eb.u_prev, u_prev0, n_up * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(dcv, curv, n_cv * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(drd, route_desc, n_rd * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(den, enc, n_en * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(eb.prev_ok, 0, nb * 4, st));
    // z_cl[:, :, 0] = z0
    CK(cudaMemcpy2DAsync(eb.z_cl, (size_t)(T + 1) * 7 * 8, eb.z, 7 * 8, 7 * 8, nb, cudaMemcpyDeviceToDevice, st));
    std::vector<cudaEvent_t> ev;
    if (step_ms) { ev.resize(T + 1); for (auto &e : ev) CK(cudaEventCreate(&e)); CK(cudaEventRecord(ev[0], st)); }
    const int bs = 128, gs = (B + bs - 1) / bs;
    int cs = 0;
    for (int t = 0; t < T; t++) {
        const int cur = t & 1, prv = cur ^ 1;
        if (obca) episode_pre_kernel<true><<<gs, bs, 0, st>>>(eb, B, N, h->prm.dt, t, gt_mpc, px[prv], pu[prv]);
        else episode_pre_kernel<false><<<gs, bs, 0, st>>>(eb, B, N, h->prm.dt, t, gt_mpc, px[prv], pu[prv]);
        h->launches++;
        rc = solve_dev_impl(h, B, eb.z, eb.u_prev, eb.curv, eb.obs, eb.obs_psi, gt_mpc ? eb.ctx : nullptr, eb.u_init, px[cur], pu[cur],
                            pcost[cur], pviol[cur], pst[cur], pit[cur], st, eb.warm, dnet);
        if (rc) return rc;
        rc = acquire_cslot(h, 1, st, &cs);
        if (rc) return rc;
        episode_post_kernel<<<gs, bs, 0, st>>>(eb, B, N, T, t, h->prm.a_min, px[cur], pu[cur], pst[cur], cs);
        h->launches++;
        if (step_ms) CK(cudaEventRecord(ev[t + 1], st));
    }
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(z_cl, eb.z_cl, n_zcl * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(u_cl, eb.u_cl, n_ucl * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(solved, eb.solved, nb * T * 4, cudaMemcpyDeviceToHost, st));
    rc = end_call(h, st, 2);
    if (rc) return rc;
    CK(cudaStreamSynchronize(st));
    if (step_ms) {
        for (int t = 0; t < T; t++) CK(cudaEventElapsedTime(&step_ms[t], ev[t], ev[t + 1]));
        for (auto &e : ev) cudaEventDestroy(e);
    }
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

