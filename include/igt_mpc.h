/* igt_mpc.h -- C ABI of the B200-native batched MPC solver (libigtmpc.so).
 *
 * Drop-in boundary for the solver behind the reference's MPC_Planner
 * (reference mpc.py:21-406).  The reference has no FFI of its own -- mpc.py talks to CasADi's
 * Python API -- so each entry point below names the reference call site(s) it replaces.  The
 * Python host (igt_mpc_int_b200/planner.py) binds these with ctypes; INTEGRATION.md shows the
 * stub a maintainer would add to the reference's mpc.py.
 *
 * Conventions: plain pointers and sizes only; every array is contiguous, batch-major
 * ("problem b" first).  `*_dev` entry points take DEVICE pointers and enqueue work on `stream`
 * (a cudaStream_t passed as void*; NULL = legacy default stream) without synchronising;
 * `*_host` entry points take HOST pointers, copy in, run, copy out and synchronise; they run on a
 * private non-blocking stream of the handle, not on the legacy default stream.
 * Every function returns 0 on success or a negative IGT_E* code; igt_last_error() gives text.
 * No C++ exception crosses this boundary.
 *
 * Concurrency.  Different handles are independent: they may be used from different host threads and on different
 * streams at the same time, whatever their horizons, limits or value networks (each handle keeps its parameters
 * in its own constant-memory slot and owns its workspace).  Calls on ONE handle may come from any thread and any
 * stream, but they are serialised: a per-handle mutex on the host, and on the device every call waits (stream
 * event) for the handle's previous call before it touches the handle's workspace.  `*_dev` calls never block the
 * host: buffers grow with the stream-ordered allocator.  Each call selects the handle's device (cudaSetDevice).
 *
 * Layouts (reference mpc.py:163-164):  state z = [x, y, s, ey, epsi, v, psi], input u = [a, df].
 */
#ifndef IGT_MPC_H
#define IGT_MPC_H

#ifdef __cplusplus
extern "C" {
#endif

#define IGT_MAX_CINF 128
#define IGT_MAX_MLP_LAYERS 5
#define IGT_MAX_MLP_NETS 8   /* value networks per handle (igt_set_mlp_at) */

#define IGT_OK 0
#define IGT_EINVAL (-1)   /* bad argument (NULL, size, unsupported horizon ...) */
#define IGT_ECUDA (-2)    /* CUDA runtime error */
#define IGT_ENOMLP (-3)   /* gt_mpc solve requested before igt_set_mlp */

/* per-problem status written by igt_solve_* (reference mpc.py:402-406 maps any failure to
 * (None, None, False); the Python host maps status != 0 the same way) */
#define IGT_STATUS_CONVERGED 0
#define IGT_STATUS_MAXITER 1
#define IGT_STATUS_X0_INFEASIBLE 2   /* x0 violates rows that involve x0 only (mpc.py:298-299,316-317 at k=0) */
#define IGT_STATUS_REG_LIMIT 3
#define IGT_STATUS_LINESEARCH 4
#define IGT_STATUS_STALLED 5         /* still infeasible (|c + slack| > stall_rp) after stall_iter iterations */
#define IGT_STATUS_ACCEPTABLE 6      /* failed to converge tightly, but the final point is within the reference's IPOPT tolerances (see acc_tol):
                                        a success for the host (IPOPT returns Solve_Succeeded there), reported apart */
#define IGT_STATUS_BAD_NET 7         /* *_ex_dev with net_idx: the index is outside 0..IGT_MAX_MLP_NETS-1 or names an empty
                                        slot; no solve, NaN outputs, the other problems are unaffected */

#define IGT_PREC_F32 0
#define IGT_PREC_F64 1

typedef struct igt_handle igt_handle;

typedef struct {
    /* ---- problem constants: effective values of mpc.py:47-62, mpc.yaml, fourwayint.yaml ---- */
    int N;            /* horizon, mpc.yaml:6 (10, 20 or 40 ... any 2 <= N <= 64) */
    int n_rk;         /* RK4 sub-steps per MPC step, evaluate.py:109 */
    double dt;        /* mpc.yaml:7 */
    double l_r, l_f;  /* mpc.py:50-51 */
    double v_min, v_max, a_min, a_max, df_max, ey_lim;   /* mpc.py:56-61 */
    double da_max, ddf_max;   /* dt*jerk_limit, dt*steering_rate_limit: mpc.py:54-55, :301-312 */
    double d_min;     /* 2*ca_radius, mpc.py:45 */
    double w_u;       /* 0.05, mpc.py:362 */
    int n_cinf;       /* rows of the terminal invariant set, mpc.py:88-104,:177-180 */
    double cinf_A[IGT_MAX_CINF][2];
    double cinf_b[IGT_MAX_CINF];
    /* ---- solver options (stand in for the IPOPT options of mpc.py:130-146) ---- */
    double tol;        /* stationarity: |grad_u Lagrangian|_inf <= tol * max(1, |mult|_inf) */
    double tol_rp;     /* primal residual |c + slack|_inf (bounds the row violation) */
    double tol_comp;   /* complementarity max(mult*slack) */
    double mu0, mu_floor, kappa_eps, kappa_mu, theta_mu, y_init_min, tau_min;
    double mu0_warm, y_init_min_warm;   /* used instead of mu0 / y_init_min when u_init is given.  Defaults 1e-3 / 1e-2: the
                                           reference restarts IPOPT from the shifted primal plan only (mpc.py:386-389; IPOPT's
                                           mu_init stays 0.1), and a hard warm start (1e-4 / 1e-3) cannot move a shifted plan
                                           that sits on its rows: over the 64 reference episodes it fails 7.5 % of the solves
                                           and deadlocks 13 episodes, the softer one 4.7 % and 6, for 3 more iterations */
    double reg_min, reg_up, reg_down, reg_max;
    double reg_jump;   /* after a Riccati stage whose Quu + reg I is not positive definite: reg >= reg_jump * (-lambda_min(Quu))
                          of that stage (besides reg * reg_up), so the inertia correction takes 1-2 retries, not 6 */
    double eps_phi, gamma_theta, theta_small;
    int max_iter;      /* iteration cap -> IGT_STATUS_MAXITER (mpc.py:137 gives IPOPT 100*N).  Default 60.  A batch is one
                          wave of problems, so its run time follows its slowest problem: a cap of 40 keeps 98.8 % of the
                          converged solves and is 18 % faster, but costs closed-loop episodes extra brake fallbacks
                          (DESIGN.md section 4) */
    int n_alpha;       /* step halvings per line search (1..6: one iterate buffer per halving) */
    int second_order;  /* add the dt*Hess(lambda.f) curvature term to the Riccati pass */
    int stall_iter;    /* local-infeasibility exit: iteration >= stall_iter and ... */
    double stall_rp;   /* ... primal residual still above stall_rp -> IGT_STATUS_STALLED */
    int max_trials;    /* optional budget of forward passes (accepted or not) per solve -> IGT_STATUS_MAXITER, for
                          giving up early on problems that burn all n_alpha halvings iteration after iteration
                          (the reference's counterpart is IPOPT's max_wall_time, mpc.py:139); 0 = no budget (default) */
    int precision;     /* IGT_PREC_F32 / IGT_PREC_F64: arithmetic of the solver kernels */
    /* Reference-tolerance exit -> IGT_STATUS_ACCEPTABLE.  When a solve ends in a failure (the iteration cap, the
     * regularisation limit, the budget of forward passes) at a point that already
     * satisfies the reference's own IPOPT tolerances (mpc.py:133-135: tol = dual_inf_tol = constr_viol_tol = 1e-3;
     * IPOPT's default compl_inf_tol = 1e-4), the point is returned as acceptable instead of failed -- IPOPT itself
     * would have stopped there with Solve_Succeeded.  stationarity <= acc_tol * max(1, |mult|_inf), primal residual
     * <= acc_rp (default 1e-6: the north star's violation bound, not the reference's 1e-3), max(mult * slack) <=
     * acc_comp.  acc_tol = 0 disables. */
    double acc_tol, acc_rp, acc_comp;
    double x0_tol;     /* tolerance of the rows that involve x0 only (IGT_STATUS_X0_INFEASIBLE); default 1e-6, so that the
                          x[:,1] of a converged plan (rows met to tol_rp) is a valid x0 of the next closed-loop step */
} igt_params;

/* Fill `p` with the reference's effective constants (N=40, dt=0.1, n_rk=4, limits of
 * mpc.py:47-62) and default solver options for `precision`.  The C_inf table is left empty
 * (n_cinf = 0): the host computes it (igt_mpc_int_b200/terminal_set.py restates
 * common/utils.py:588-627) and stores it here before igt_create. */
int igt_default_params(igt_params *p, int precision);

/* Replaces MPC_Planner.__init__ (mpc.py:21-160): builds the immutable solver object. */
int igt_create(const igt_params *p, igt_handle **out);
void igt_destroy(igt_handle *h);
const char *igt_last_error(const igt_handle *h);   /* h may be NULL: last create error */

/* Replaces mpc.py:105-127 (loading the value network and its normalisation).
 * n_layers linear layers with tanh between them (model.py:14-51); W[l] is row-major
 * [dims[l+1], dims[l]], dims[0] == 6, dims[n_layers] == 1.  Wn = 6x6 whitening matrix
 * (mpc.py:116), mu_f[6] feature mean, sigma_t / mu_t target scaling (mpc.py:117-118). */
int igt_set_mlp(igt_handle *h, int n_layers, const int *dims, const double *const *W,
                const double *const *b, const double *Wn, const double *mu_f, double sigma_t,
                double mu_t);

/* Network bank, mpc.py:105-127 once per network: the reference ships one value network per scenario (V_GT_sc{1..8}.pt)
 * and evaluate.py:123 loads network k for scenario k.  Loads a network as igt_set_mlp does into slot `net`
 * (0..IGT_MAX_MLP_NETS-1) of the handle's bank; the *_ex entry points below pick a slot per problem (net_idx).
 * net = 0 is exactly igt_set_mlp: slot 0 is also the network of every call without net_idx.  All arguments are
 * checked before anything is replaced; only slot `net`'s buffers are freed.  A bank solve always evaluates the value
 * term exactly (fp64 / the solver's precision): the "tensor_core_mlp" option applies to single-network calls only. */
int igt_set_mlp_at(igt_handle *h, int net, int n_layers, const int *dims, const double *const *W,
                   const double *const *b, const double *Wn, const double *mu_f, double sigma_t, double mu_t);

/* Replaces KinematicBicycleModelFrenet.__call__ (common/kinematic_bicycle_model_frenet.py:
 * 69-185; model 0) and KinematicBicycleModel.__call__ (common/kinematic_bicycle_model.py:
 * 15-50; model 1) rolled over the horizon, plus the Jacobians CasADi derives by AD.
 * fp32 device arrays.  model 0: z0[B,7], u[B,N,2], curv[B,3] = (b0, b1, Kval) of the pw_const
 * curvature (mpc.py:183-200), z[B,N+1,7], A[B,N,7,7], Bm[B,N,7,2].
 * model 1: z0[B,4] = (x, y, psi, v), z[B,N+1,4], A[B,N,4,4], Bm[B,N,4,2], curv ignored.
 * A and Bm may both be NULL. */
int igt_rollout_dev(igt_handle *h, int B, const float *z0, const float *u, const float *curv,
                    float *z, float *A, float *Bm, int model, void *stream);
int igt_rollout_host(igt_handle *h, int B, const float *z0, const float *u, const float *curv,
                     float *z, float *A, float *Bm, int model);

/* Cost (mpc.py:356-373) and the largest inequality-row value, rows exactly as written in
 * mpc.py:177-180,:223-226,:296-321 (collision in squared-distance units), of given controls.
 * The state trajectory is re-rolled on the device.  fp64 arrays: x0[B,7], u_prev[B,2],
 * curv[B,3], obs_xy[B,N+1,2], obs_psi[B,N+1] or NULL (see igt_solve_*), nn_ctx[B,4] = (s_tv, v_tv, e_tv, e_ego) or
 * NULL ('mpc' cost), u[B,N,2] -> cost[B], viol[B], z[B,N+1,7] (z may be NULL).
 * viol[b] = max(0, largest row); a NaN row makes it NaN, so controls with a NaN, or controls that drive the state
 * non-finite, never report a violation that looks feasible (their cost is non-finite as well). */
int igt_eval_host(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                  const double *obs_xy, const double *obs_psi, const double *nn_ctx, const double *u,
                  double *cost, double *viol, double *z);
/* The same with net_idx[B] (int32, needs nn_ctx) or NULL: problem b's value term uses bank slot net_idx[b]
 * (evaluate.py:198-312 per scenario).  Every index must name a loaded slot, else IGT_EINVAL before any launch. */
int igt_eval_ex_host(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                     const double *obs_xy, const double *obs_psi, const double *nn_ctx, const int *net_idx,
                     const double *u, double *cost, double *viol, double *z);

/* Replaces MPC_Planner.update_initial_condition / update_predictions / solve
 * (mpc.py:280-294, :241-278, :383-406) for a batch of independent problems.
 * In : x0[B,7]; u_prev[B,2]; curv[B,3]; obs_xy[B,N+1,2] (row 0 unused, mpc.py:224);
 *      obs_psi[B,N+1] or NULL -- non-NULL selects collision_avoidance_type 'obca' (mpc.py:42-43, :170-175, :211-221):
 *      the obstacle's heading forecast (preds row 6, mpc.py:250-260); the rows are enforced in dual-eliminated
 *      form, margin 1e-6 + d_min - signed distance between the two 4.47 x 2.0 rectangles <= 0 (csrc/obca.cuh), with
 *      d_min = 0 as the reference sets it for this mode; viol[] then reports that row.  f64 only.
 *      nn_ctx[B,4] or NULL -- non-NULL selects the gt_mpc terminal cost (mpc.py:367-369);
 *      u_init[B,N,2] or NULL -- warm start (mpc.py:386-389); NULL = cold-start rule.
 * Out: x[B,N+1,7], u[B,N,2], cost[B], viol[B] (max inequality row, reference units),
 *      status[B] (IGT_STATUS_*), iters[B].  All fp64 / int32. */
int igt_solve_dev(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                  const double *obs_xy, const double *obs_psi, const double *nn_ctx, const double *u_init,
                  double *x, double *u, double *cost, double *viol, int *status, int *iters, void *stream);
int igt_solve_host(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                   const double *obs_xy, const double *obs_psi, const double *nn_ctx, const double *u_init,
                   double *x, double *u, double *cost, double *viol, int *status, int *iters);
/* The gt_mpc branch of evaluate.py:198-312 for many scenarios in one batch (evaluate.py:123: scenario k plans with
 * network k): igt_solve_* plus net_idx[B] (int32) or NULL.  Problem b's value term uses bank slot net_idx[b]
 * (igt_set_mlp_at); net_idx needs nn_ctx, else IGT_EINVAL.  NULL is exactly igt_solve_*.
 * _host checks the indices and returns IGT_EINVAL before any launch if one names no loaded slot; _dev checks them in
 * the kernel: such a problem gets IGT_STATUS_BAD_NET.  Bank solves use the exact value term (cooperative if every
 * loaded network is <= 128 wide and the solve is fp64 circle mode; per thread otherwise). */
int igt_solve_ex_dev(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                     const double *obs_xy, const double *obs_psi, const double *nn_ctx, const int *net_idx,
                     const double *u_init, double *x, double *u, double *cost, double *viol, int *status, int *iters,
                     void *stream);
int igt_solve_ex_host(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                      const double *obs_xy, const double *obs_psi, const double *nn_ctx, const int *net_idx,
                      const double *u_init, double *x, double *u, double *cost, double *viol, int *status, int *iters);

/* Gradients through the solve (csrc/sens.cuh; DESIGN.md section 10).
 *
 * Inequality rows of one problem, M = igt_row_count(h) = 8 + 13 (N - 1) + n_cinf + 3 of them, in the solver's order:
 *   node 0:            a <= a_max, a >= a_min, df <= df_max, df >= -df_max, the four rate rows (a - a_prev <= da_max,
 *                      a_prev - a <= da_max, df - df_prev <= ddf_max, df_prev - df <= ddf_max)          -- 8 rows
 *   node k = 1..N-1:   v <= v_max, v >= v_min, ey <= ey_lim, ey >= -ey_lim, collision (d_min - |p - o| <= 0), then
 *                      the 8 input rows of node 0's order                                                -- 13 rows
 *   after node N-1:    the n_cinf terminal-set rows C_inf.A [v_{N-1}; a_{N-1}] <= C_inf.b
 *   node N:            ey <= ey_lim, ey >= -ey_lim, collision                                            -- 3 rows
 * Each row is c(u) <= 0 with slack y = -c > 0 and multiplier s > 0 at the returned point. */
int igt_row_count(const igt_handle *h);

/* igt_solve_ex_* that also writes the final slack[B,M] and multiplier mult[B,M] of every row (the iterate the solve
 * returned; NaN for a problem that was never solved, status 2 / 7).  x, u, cost, viol, status, iters are the same bits as
 * igt_solve_ex_*.  Supported: precision f64, circle rows, 'mpc' and gt_mpc with one network or a bank, exact value term.
 * IGT_EINVAL: obs_psi (OBCA: Gauss-Newton rows with a piecewise Hessian), precision f32, and gt_mpc with
 * tensor_core_mlp = 1 (it perturbs the merit at 1e-7).  Always runs the throughput kernel, whatever latency_path says
 * (the latency kernel gives the same bits). */
int igt_solve_duals_ex_dev(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                           const double *obs_xy, const double *obs_psi, const double *nn_ctx, const int *net_idx,
                           const double *u_init, double *x, double *u, double *cost, double *viol, int *status, int *iters,
                           double *slack, double *mult, void *stream);
int igt_solve_duals_ex_host(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                            const double *obs_xy, const double *obs_psi, const double *nn_ctx, const int *net_idx,
                            const double *u_init, double *x, double *u, double *cost, double *viol, int *status, int *iters,
                            double *slack, double *mult);

/* Vector-Jacobian product of a solve through its converged KKT system: the implicit function theorem on
 * grad_u L = 0, c + y = 0, s_i y_i = const_i at the returned (u, y, s), theta = (x0, u_prev, obs_xy), the rollout
 * included, with the exact Hessian of the Lagrangian (stage cost, value term, circle rows, second derivatives of the
 * discrete RK4 step).  One problem per thread, fp64.
 * In : the solve's inputs x0, u_prev, curv, obs_xy, nn_ctx (or NULL), net_idx (or NULL; as in igt_solve_ex_*) and its
 *      outputs u[B,N,2], slack[B,M], mult[B,M], status[B] (igt_solve_duals_ex_*); cotangents gx[B,N+1,7], gu[B,N,2],
 *      gcost[B] on x, u, cost, each may be NULL (zero).
 * Out: gx0[B,7], gu_prev[B,2], gobs[B,N+1,2] (row 0 is 0: mpc.py:224 does not use it), ok[B] (int32).
 *      ok = 0 with exact zero gradients (never NaN) when status != 0, when a slack or multiplier is not positive, when a
 *      stage's Quu of the Riccati sweep is not positive definite (no regularisation), or when a result is not finite.
 * Needs precision f64; gt_mpc with tensor_core_mlp = 1 is IGT_EINVAL.  A device net_idx naming no loaded slot gives
 * ok = 0; the _host call checks the indices as igt_solve_ex_host does.  _dev and _host give the same bits. */
int igt_solve_vjp_dev(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                      const double *obs_xy, const double *nn_ctx, const int *net_idx, const double *u, const double *slack,
                      const double *mult, const int *status, const double *gx, const double *gu, const double *gcost,
                      double *gx0, double *gu_prev, double *gobs, int *ok, void *stream);
int igt_solve_vjp_host(igt_handle *h, int B, const double *x0, const double *u_prev, const double *curv,
                       const double *obs_xy, const double *nn_ctx, const int *net_idx, const double *u, const double *slack,
                       const double *mult, const int *status, const double *gx, const double *gu, const double *gcost,
                       double *gx0, double *gu_prev, double *gobs, int *ok);

/* Replaces the per-timestep loop of evaluate.py:451-564 ('mpc') / :198-312 ('gt_mpc') for E independent two-vehicle
 * episodes: `steps` closed-loop steps entirely on the device -- per step one kernel for the glue before the solve
 * (constant-acceleration forecast constant_acceleration_model.py:18-82, shared plans utils.py:339-352, filter_preds
 * utils.py:365-388, warm start utils.py:354-363, value-network context mpc.py:326-337), one batched solve of all 2E
 * vehicles (per-problem warm / cold start), one kernel after it (plant evaluate.py:491-510, brake fallback :511-545).
 * Vehicle b = 2 e + i is agent i of episode e.
 * mode: a bit set.  0 = the 'mpc' branch with circle rows;
 *   IGT_EPISODE_GT_MPC -- the 'gt_mpc' branch (value-network terminal cost; the handle needs igt_set_mlp);
 *   IGT_EPISODE_OBCA   -- collision_avoidance_type 'obca' (mpc.py:42-43): the glue also forecasts the other vehicle's
 *                         heading (k = 0 its current psi; k >= 1 the route heading at the forecast arc length, or its
 *                         previous plan's psi in the shared-plan case; abs() on routes 32 / 41, mpc.py:250-253; 0 for
 *                         a filtered obstacle) and every solve gets it as obs_psi (see igt_solve_*).  The handle's
 *                         d_min should be 0, as the reference sets it for this mode.
 *   Any other bit: IGT_EINVAL.
 * Host fp64 arrays:
 *   route_desc[2E,12] = (x0, y0, t0x, t0y, turn sign, b0, b1, r, exit axis (0 x, 1 y, -1 none), exit coordinate,
 *                       th0, flip): the closed-form lane centre of the vehicle's route (igt_mpc_int_b200/geometry.py);
 *                       th0 = start heading, flip = 1.0 on routes 32 and 41, else 0.0 -- read in OBCA mode only;
 *   curv[2E,3]; z0[2E,7] initial states; u_prev0[2E,2]; enc[2E] scenario codes (utils.py:141-169, gt_mpc only);
 *   out: z_cl[E,2,steps+1,7], u_cl[E,2,steps,2], solved[E,2,steps] (int32), step_ms[steps] (device time per step; may
 *   be NULL).  The handle's horizon N, limits and (gt_mpc) value network apply; precision must be f64. */
#define IGT_EPISODE_GT_MPC 1
#define IGT_EPISODE_OBCA 2
int igt_episode_run_host(igt_handle *h, int E, int steps, int mode, const double *route_desc, const double *curv,
                         const double *z0, const double *u_prev0, const double *enc, double *z_cl, double *u_cl,
                         int *solved, float *step_ms);
/* The same with net_idx[E] (int32) or NULL: both vehicles of episode e plan with bank slot net_idx[e], so episodes
 * of all scenarios run in one loop, each with its own network (evaluate.py:123, :198-312).  Needs the
 * IGT_EPISODE_GT_MPC bit (with or without IGT_EPISODE_OBCA); indices are checked as in igt_solve_ex_host. */
int igt_episode_run_ex_host(igt_handle *h, int E, int steps, int mode, const double *route_desc, const double *curv,
                            const double *z0, const double *u_prev0, const double *enc, const int *net_idx, double *z_cl,
                            double *u_cl, int *solved, float *step_ms);

/* Number of kernels this library has launched on `h` so far (bench.py's gpu_launches). */
long long igt_launch_count(const igt_handle *h);

/* The gt_mpc value term alone (mpc.py:367-369, model.py:53-67): V(W (x_N - mu_f)) sigma_t + mu_t and its
 * first / second derivatives in (s_N, v_N), out[B,6] = (V, dV/ds, dV/dv, d2V/dss, d2V/dsv, d2V/dvv).
 * use_tensor_cores = 1: tcgen05 kernel (6-128-128-1 networks); 0: fp64 per-thread kernel; 2: the exact fp64
 * CTA-cooperative evaluation the solver uses (csrc/mlp_coop.cuh; any network with layers <= 128 wide).  Host fp64 arrays. */
int igt_mlp_value_host(igt_handle *h, int B, const double *sN, const double *vN, const double *nn_ctx,
                       double *out, int use_tensor_cores);
/* The same with net_idx[B] (int32) or NULL: row b uses bank slot net_idx[b] (mpc.py:367-369 with network k of
 * evaluate.py:123).  Modes 0 and 2 only (1 with net_idx: IGT_EINVAL); indices checked as in igt_solve_ex_host. */
int igt_mlp_value_ex_host(igt_handle *h, int B, const double *sN, const double *vN, const double *nn_ctx,
                          const int *net_idx, double *out, int use_tensor_cores);

/* Run-time switches.
 * "tensor_core_mlp" (default 0).  The gt_mpc value term is evaluated exactly (fp64) by default, CTA-cooperatively
 * (csrc/mlp_coop.cuh: waves of 16 evaluations, weights streamed through shared memory, any network up to 128 wide -- all eight shipped V_GT_sc*.pt).  1 = the
 * tcgen05 kernel (csrc/mlp_tc.cuh; 6-128-128-1 networks, bf16x3 = fp32-accurate): measured no faster than the exact
 * path on a B200 (DESIGN.md section 4) and it perturbs the merit at 1e-7, so closed-loop outcomes can differ from the
 * fp64 oracle's; kept as an option.
 * "latency_path" (default 1): batches of at most one problem per SM (a closed-loop step solves the two vehicles of an
 * episode) run one CTA per problem with the workspace in shared memory; 0 = throughput kernel.  'mpc' mode, and gt_mpc
 * with one network or a bank (net_idx): exact cooperative value term in circle mode (fp64, layers <= 128 wide), per-thread
 * value term in OBCA mode, in fp32 and for wider networks.  Not with the tensor-core value term (tensor_core_mlp = 1),
 * and only while the kernel's shared memory fits a block: with the cooperative value term up to N = 45 (a bank: N = 44)
 * at n_cinf = 74 on a B200; longer horizons take the throughput kernel.  Results are the same bits either way. */
int igt_set_option(igt_handle *h, const char *name, double value);

/* Measured throughput (TFLOP/s, FMA = 2 flops) of dependent-free FMA chains in `precision` on
 * this device: the CUDA-core roofline denominator bench.py reports the solver against. */
int igt_measure_fma_peak(igt_handle *h, int precision, double *tflops);

/* Library build info: returns e.g. "igtmpc 0.1 sm_100a". */
const char *igt_version(void);

#ifdef __cplusplus
}
#endif
#endif /* IGT_MPC_H */
