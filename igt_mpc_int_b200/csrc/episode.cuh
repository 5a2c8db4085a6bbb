// episode.cuh -- the per-timestep glue of the reference's closed loop on the device (SURVEY 8(f) N1), so that E
// two-vehicle episodes x T steps run without the host in the loop: one batched solve per 0.1 s step, one small kernel
// before it (forecasts, obstacle, value-network context, warm start) and one after it (plant, brake fallback, records).
//
//   predict            constant-acceleration forecast                       common/constant_acceleration_model.py:18-82
//   share forecasts    a vehicle that solved at t-1 is forecast by its plan   common/utils.py:339-352
//   filter_preds       obstacle behind the ego -> (-20, -20)                  common/utils.py:365-388
//   warm start         previous inputs shifted by one                         common/utils.py:354-363
//   plant              next state = x_sol[:, 1]                               evaluate.py:491-510
//   brake fallback     a = a_min if v > 0 else 0, previous steering           evaluate.py:511-545
//   OBCA mode          the obstacle's heading forecast as well                mpc.py:250-253 (MPC_Planner.update_predictions)
// Same arithmetic as igt_mpc_int_b200/episode.py (the host-side numpy driver this replaces for large E).
#pragma once
#include "solver_core.cuh"

namespace igt {

constexpr int ROUTE_DESC = 12;   // x0, y0, t0x, t0y, sgn, b0, b1, r, exit_axis (0: x, 1: y, -1: none), exit_coord, th0, flip

// lane-centre (x, y) at arc length s (igt_mpc_int_b200/geometry.frenet2global_xy; closed form of common/utils.py:532-586)
__host__ __device__ inline void route_xy(const double *rd, double s, double *x, double *y)
{
    const double x0 = rd[0], y0 = rd[1], t0x = rd[2], t0y = rd[3], sgn = rd[4], b0 = rd[5], b1 = rd[6], r = rd[7];
    if (sgn == 0.0 || s < b0) { *x = x0 + s * t0x; *y = y0 + s * t0y; return; }
    const double n0x = -t0y, n0y = t0x;
    const double cx = x0 + b0 * t0x + sgn * r * n0x, cy = y0 + b0 * t0y + sgn * r * n0y;
    if (s <= b1) {
        const double phi = (s - b0) / r, sp = sin(phi), cp = cos(phi);
        *x = cx + r * (sp * t0x - sgn * cp * n0x);
        *y = cy + r * (sp * t0y - sgn * cp * n0y);
        return;
    }
    const double t1x = sgn * n0x, t1y = sgn * n0y;
    *x = cx + r * t0x + (s - b1) * t1x;
    *y = cy + r * t0y + (s - b1) * t1y;
    if (rd[8] == 0.0) *x = rd[9];
    else if (rd[8] == 1.0) *y = rd[9];
}

// path heading at arc length s (the third output of igt_mpc_int_b200/geometry.frenet2global; geometry.route_heading):
// th0 before the arc, th0 + sgn phi on it, th0 + sgn pi/2 after it.  th0 = rd[10] is stored rather than recovered from
// (t0x, t0y) with atan2, so host and device headings are the same bits.
__host__ __device__ inline double route_heading(const double *rd, double s)
{
    const double th0 = rd[10], sgn = rd[4], b0 = rd[5], b1 = rd[6], r = rd[7];
    if (sgn == 0.0 || s < b0) return th0;
    if (s <= b1) return th0 + sgn * ((s - b0) / r);
    return th0 + sgn * (M_PI / 2);
}

struct EpisodeBufs {
    double *z, *u_prev;            // [B,7] [B,2] current state and last applied input
    const double *curv, *rd, *enc; // [B,3] [B,ROUTE_DESC] [B]
    double *obs, *ctx, *u_init;    // solver inputs built by the pre-step kernel: [B,N+1,2] [B,4] [B,N,2]
    int *warm;                     // [B]
    int *prev_ok;                  // [B] the solve of the previous step succeeded
    double *z_cl, *u_cl;           // records [E,2,T+1,7] [E,2,T,2]
    int *solved;                   // [E,2,T]
    double *obs_psi;               // [B,N+1] obstacle heading forecast (OBCA mode only, else null)
};

#ifdef __CUDACC__
// one constant-acceleration predictor step (constant_acceleration_model.py:69-71; fourwayint.yaml:23-24 clip)
__device__ inline void ca_step(double s, double v, double a, double dt, double *s1, double *v1)
{
    *s1 = s + v * dt + 0.5 * a * dt * dt;
    *v1 = fmin(fmax(v + a * dt, -2.0), 20.0);
}

// before the solve of step t: thread b builds vehicle b's obstacle forecast (= forecast of vehicle b ^ 1), value-network
// context, warm start.  px / pu: the plans of step t-1 (solver outputs [B,N+1,7] / [B,N,2]).
// OBCA: also the obstacle's heading forecast eb.obs_psi[b, 0..N] (igt_mpc_int_b200/episode.py states the convention):
// constant acceleration -- k = 0 the current psi, k >= 1 the route heading at s_k; V2V -- k < N the plan's psi at k + 1,
// k = N the route heading at the extra step's s; abs() on routes 32 / 41 (rd[11]); 0 for a filtered obstacle.
template <bool OBCA>
__global__ void episode_pre_kernel(EpisodeBufs eb, int B, int N, double dt, int t, int gt, const double *px, const double *pu)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int o = b ^ 1;
    const double *zo = eb.z + 7 * o, *zb = eb.z + 7 * b, *rdo = eb.rd + ROUTE_DESC * o;
    double *obs = eb.obs + (long)b * (N + 1) * 2;
    double *psi = OBCA ? eb.obs_psi + (long)b * (N + 1) : nullptr;
    double sN, vN;
    if (t > 0 && eb.prev_ok[o]) {                                  // V2V: the other vehicle's plan of t-1, shifted by one
        const double *pxo = px + (long)o * (N + 1) * 7, *puo = pu + (long)o * N * 2;
        for (int k = 0; k < N; k++) { obs[2 * k] = pxo[(k + 1) * 7 + IX]; obs[2 * k + 1] = pxo[(k + 1) * 7 + IY]; }
        if (OBCA) for (int k = 0; k < N; k++) psi[k] = pxo[(k + 1) * 7 + IPSI];
        double s1, v1;
        ca_step(pxo[N * 7 + IS], pxo[N * 7 + IV], puo[(N - 1) * 2], dt, &s1, &v1);
        if (v1 > 5.0) ca_step(pxo[N * 7 + IS], pxo[N * 7 + IV], 0.0, dt, &s1, &v1);
        route_xy(rdo, s1, &obs[2 * N], &obs[2 * N + 1]);
        if (OBCA) psi[N] = route_heading(rdo, s1);
        sN = s1; vN = v1;
    } else {                                                       // constant acceleration from the current state
        double a0 = eb.u_prev[2 * o];
        if (gt && t == 0) a0 = 0.09 * ((o & 1) + 1);               // evaluate.py:207-210
        double s = zo[IS], v = zo[IV];
        obs[0] = zo[IX]; obs[1] = zo[IY];
        if (OBCA) psi[0] = zo[IPSI];
        for (int k = 0; k < N; k++) {
            ca_step(s, v, a0, dt, &s, &v);
            route_xy(rdo, s, &obs[2 * (k + 1)], &obs[2 * (k + 1) + 1]);
            if (OBCA) psi[k + 1] = route_heading(rdo, s);
        }
        sN = s; vN = v;
    }
    // filter_preds: the other vehicle is behind the ego (utils.py:365-388)
    const double dx = obs[0] - zb[IX], dy = obs[1] - zb[IY];
    if (dx * cos(zb[IPSI]) + dy * sin(zb[IPSI]) < 0.0) {
        for (int k = 0; k <= N; k++) { obs[2 * k] = -20.0; obs[2 * k + 1] = -20.0; }
        if (OBCA) for (int k = 0; k <= N; k++) psi[k] = 0.0;
    } else if (OBCA && rdo[11] != 0.0) {
        for (int k = 0; k <= N; k++) psi[k] = fabs(psi[k]);                          // mpc.py:250-253
    }
    eb.ctx[4 * b] = sN; eb.ctx[4 * b + 1] = vN; eb.ctx[4 * b + 2] = eb.enc[o]; eb.ctx[4 * b + 3] = eb.enc[b];   // mpc.py:326-337
    const int warm = t > 0 && eb.prev_ok[b] && (gt ? t > 1 : 1);   // evaluate.py:232-235 / :478-481
    eb.warm[b] = warm;
    if (warm) {
        const double *pub = pu + (long)b * N * 2;
        double *ui = eb.u_init + (long)b * N * 2;
        for (int k = 0; k < N - 1; k++) { ui[2 * k] = pub[2 * (k + 1)]; ui[2 * k + 1] = pub[2 * (k + 1) + 1]; }
        ui[2 * (N - 1)] = pub[2 * (N - 1)]; ui[2 * (N - 1) + 1] = pub[2 * (N - 1) + 1];                      // utils.py:362
    }
}

// after the solve of step t: plant update, brake fallback, records
__global__ void episode_post_kernel(EpisodeBufs eb, int B, int N, int T, int t, double a_brake, const double *x, const double *u,
                                    const int *status, int cs)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const DevParams<double> &P = ConstP<double>::get(cs);
    double *z = eb.z + 7 * b, *up = eb.u_prev + 2 * b;
    const int ok = status[b] == 0 || status[b] == 6;               // IGT_STATUS_CONVERGED / _ACCEPTABLE
    double zn[NZ], ua[2];
    if (ok) {
        for (int i = 0; i < NZ; i++) zn[i] = x[((long)b * (N + 1) + 1) * 7 + i];                             // evaluate.py:493
        ua[0] = u[(long)b * N * 2]; ua[1] = u[(long)b * N * 2 + 1];
    } else if (z[IV] < 0.0) {                                                                               // evaluate.py:524-528
        for (int i = 0; i < NZ; i++) zn[i] = z[i];
        zn[IV] = 0.0; ua[0] = 0.0; ua[1] = up[1];
    } else {
        ua[0] = z[IV] > 0.0 ? a_brake : 0.0; ua[1] = up[1];                                                  // evaluate.py:516
        const double curv[3] = { eb.curv[3 * b], eb.curv[3 * b + 1], eb.curv[3 * b + 2] };
        rk4_step(P, z, ua, curv, zn);
    }
    for (int i = 0; i < NZ; i++) z[i] = zn[i];
    up[0] = ua[0]; up[1] = ua[1];
    eb.prev_ok[b] = ok;
    const long e = b >> 1, i = b & 1;
    for (int j = 0; j < NZ; j++) eb.z_cl[((e * 2 + i) * (T + 1) + t + 1) * 7 + j] = zn[j];
    eb.u_cl[((e * 2 + i) * T + t) * 2] = ua[0]; eb.u_cl[((e * 2 + i) * T + t) * 2 + 1] = ua[1];
    eb.solved[(e * 2 + i) * T + t] = ok;
}
#endif

}  // namespace igt
