"""Batched closed-loop episode driver (SURVEY 8(f) N1): E independent two-vehicle episodes advance
together, one batched MPC solve per 0.1 s step for all 2E vehicles.

Mirrors the per-timestep glue of the reference's `evaluate.py`, 'mpc' branch (evaluate.py:451-564) and
'gt_mpc' branch (evaluate.py:198-312; differences listed at `run_closed_loop`):
  predict            constant-acceleration forecast      common/constant_acceleration_model.py:18-82
  share forecasts    a vehicle that solved at t-1 is forecast by its own plan   common/utils.py:339-352
  filter_preds       obstacles behind the ego -> (-20, -20)                     common/utils.py:365-388
  warm start         previous input sequence shifted by one                     common/utils.py:354-363
  solve              both vehicles read forecasts made BEFORE the agent loop (Jacobi), evaluate.py:455-482
  plant              next state = x_sol[:, 1] (perfect model), evaluate.py:491-510
  brake fallback     a = a_min if v > 0 else 0, previous steering, one model step; v < 0 -> hold pose, v = 0
                     evaluate.py:511-545
  outcome            deadlock = (#vehicles with final s <= 30) >= 2, evaluate.py:566-569; collision
                     (min centre distance < d_min; in OBCA mode: the two 4.47 x 2.0 rectangles overlap at a
                     recorded step) and goal (final s > 30) are derived here.

Collision avoidance (`ca_type`, the reference's mpc.yaml collision_avoidance_type): 'circle' (default) or 'obca'
(mpc.py:42-43, :170-175, :211-221; the solver must have d_min = 0).  OBCA needs the obstacle's heading forecast
obs_psi[b, k], k = 0..N, built with the convention of MPC_Planner.update_predictions (mpc.py:250-253):
  constant acceleration   k = 0 the other vehicle's current psi, k >= 1 the route heading at the forecast s_k
  V2V                     k < N its previous plan's psi at k + 1, k = N the route heading at the extra step's s
  flip                    abs() of every point if the other vehicle's route is 32 or 41
  filter_preds            0.0 for an obstacle moved to (-20, -20)
(csrc/episode.cuh episode_pre_kernel builds the same numbers on the device.)

The solver is any object with the BatchSolver methods `solve_batch` and `evaluate`; tests drive the
same loop with the CPU oracle wrapped in that interface to compare outcomes.
"""
from dataclasses import dataclass, field
import time

import numpy as np

from . import _lib

from . import geometry as G

A_MIN_BRAKE = -4.0     # mpc.yaml:8 a_min, evaluate.py:516
V_PRED_MIN, V_PRED_MAX = -2.0, 20.0   # fourwayint.yaml:23-24 (predictor clip)


@dataclass
class EpisodeSpec:
    routes: list                 # [route_0, route_1], e.g. ['13', '23']
    s0: tuple                    # start offsets along the routes (evaluate.py:91-94, :404-418)
    scenario: int = 0            # reference scenario 1..8 (0: not from reference_episode_specs)


@dataclass
class EpisodeResult:
    z_cl: np.ndarray             # [E, 2, T+1, 7] closed-loop states (x, y, s, ey, epsi, v, psi)
    u_cl: np.ndarray             # [E, 2, T, 2]
    solved: np.ndarray           # [E, 2, T] bool
    deadlock: np.ndarray         # [E] bool  (evaluate.py:566-569)
    collision: np.ndarray        # [E] bool
    goal: np.ndarray             # [E, 2] bool
    num_infeasible: np.ndarray   # [E, 2]
    min_distance: np.ndarray     # [E]
    step_latency_ms: list = field(default_factory=list)


def reference_episode_specs(scenarios=range(1, 9), sample=0, seed=2026):
    """All (rotation, order) variants of each scenario with the start offsets the reference draws:
    default_rng(2026).random() * max_start in region order 1, 2, 3, 4 per sample (evaluate.py:56,
    :91-94).  The reference picks rotation and order with an unseeded random.choice
    (utils.py:177-179), so every variant is enumerated."""
    max_start = (G.ROAD_LENGTH - G.ROAD_WIDTH) / 2 - (G.ROAD_WIDTH - G.CA_RADIUS)
    rng = np.random.default_rng(seed)
    draws = rng.random(4 * (sample + 1))[4 * sample:]
    offs = {str(r + 1): draws[r] * max_start for r in range(4)}
    specs = []
    for sc in scenarios:
        for rot in range(4):
            for order in range(2):
                routes = G.scenario_routes(sc, rot, order)
                specs.append(EpisodeSpec(routes=routes, s0=tuple(offs[r[0]] for r in routes), scenario=sc))
    return specs


def _outcome(z_cl, u_cl, solved, d_min, ca_type, lat):
    """deadlock (evaluate.py:566-569), collision, goal.  min_distance is the centre distance in both modes."""
    dist = np.sqrt(np.sum((z_cl[:, 0, :, :2] - z_cl[:, 1, :, :2]) ** 2, axis=-1))
    if ca_type == "obca":
        collision = G.rectangles_overlap(z_cl[:, 0][..., [0, 1, 6]], z_cl[:, 1][..., [0, 1, 6]]).any(axis=1)
    else:
        collision = dist.min(axis=1) < d_min - 1e-6
    final_s = z_cl[:, :, -1, 2]
    return EpisodeResult(z_cl=z_cl, u_cl=u_cl, solved=solved, deadlock=np.sum(final_s <= 30, axis=1) >= 2,
                         collision=collision, goal=final_s > 30, num_infeasible=(~solved).sum(axis=2),
                         min_distance=dist.min(axis=1), step_latency_ms=lat)


def _vehicle_nets(net_idx, E):
    """per-episode bank slots [E] -> per-vehicle [2E] (both vehicles of an episode plan with its network)"""
    a = np.asarray(net_idx, dtype=np.int32)
    if a.shape != (E,):
        raise ValueError("net_idx: one bank slot per episode, expected shape (%d,), got %s" % (E, a.shape))
    return np.repeat(a, 2)


def run_closed_loop(solver, specs, steps=150, N=40, dt=0.1, d_min=5.6, record_latency=False, mode="mpc",
                    ca_type="circle", net_idx=None):
    """mode 'gt_mpc' (the solver must have been given the value network): previous input (0, 0) instead of
    (0.1, 0) (evaluate.py:171 / :419); the first forecast assumes a = 0.09 (i + 1) for vehicle i
    (evaluate.py:207-210); warm starts only from t = 2 on (evaluate.py:232-235); every solve gets
    nn_ctx = (s_tv, v_tv, e_tv, e_ego): the other vehicle's forecast at step N (mpc.py:330) and the
    scenario codes of utils.scenario_encoding (mpc.py:336-337).
    ca_type 'obca': every solve also gets obs_psi (module docstring); the solver must have been made with d_min = 0.
    Circle mode calls solve_batch without obs_psi, so solvers that do not know the keyword still work.
    net_idx[E] (gt_mpc): the solver's network-bank slot of each episode (evaluate.py:123, network k for scenario k), so
    that episodes of several scenarios run in one loop; passed to solve_batch only when given."""
    assert mode in ("mpc", "gt_mpc") and ca_type in ("circle", "obca")
    if net_idx is not None and mode != "gt_mpc":
        raise ValueError("net_idx selects value networks: mode 'gt_mpc' only")
    gt = mode == "gt_mpc"
    obca = ca_type == "obca"
    E = len(specs)
    B = 2 * E
    veh_net = None if net_idx is None else _vehicle_nets(net_idx, E)
    routes = [sp.routes for sp in specs]
    curv = np.array([G.curvature_params(r) for sp in specs for r in sp.routes])           # [B, 3]
    z = np.zeros((B, 7))
    for e, sp in enumerate(specs):
        for i in range(2):
            x, y, th = G.frenet2global(sp.s0[i], sp.routes[i])
            if sp.routes[i] in ('32', '41'):
                th = abs(th)                                                               # mpc.py:282-283
            z[2 * e + i] = (x, y, sp.s0[i], 0.0, 0.0, 0.0, th)                             # evaluate.py:404-418, v0 = 0
    u_prev = np.tile([0.0, 0.0] if gt else [0.1, 0.0], (B, 1))                             # evaluate.py:171 / :419
    enc = np.array([G.scenario_encoding(sp.routes) for sp in specs], dtype=np.float64).reshape(B)   # e of every vehicle
    z_cl = np.zeros((E, 2, steps + 1, 7)); u_cl = np.zeros((E, 2, steps, 2))
    solved = np.zeros((E, 2, steps), dtype=bool)
    z_cl[:, :, 0] = z.reshape(E, 2, 7)
    prev_x = np.zeros((B, N + 1, 7)); prev_u = np.zeros((B, N, 2)); prev_ok = np.zeros(B, dtype=bool)
    lat = []
    route_of = [routes[b // 2][b % 2] for b in range(B)]
    groups = {r: np.array([b for b in range(B) if route_of[b] == r]) for r in sorted(set(route_of))}

    def route_xy(s):
        """lane-centre (x, y) of every vehicle's arc length(s): s[B] or s[B, K]"""
        x = np.empty_like(s); y = np.empty_like(s)
        for r, idx in groups.items():
            x[idx], y[idx] = G.frenet2global_xy(s[idx], r, exit_coord=G.EXIT_COORD.get(r))
        return x, y

    def route_psi(s):
        """route heading of every vehicle's arc length(s): s[B] or s[B, K]"""
        th = np.empty_like(s)
        for r, idx in groups.items():
            th[idx] = G.route_heading(s[idx], r)
        return th

    flip = np.array([r in ('32', '41') for r in route_of])                                  # mpc.py:250-253

    def ca_step(s, v, a):
        """one constant-acceleration predictor step, constant_acceleration_model.py:69-71 (vectorised)"""
        return s + v * dt + 0.5 * a * dt * dt, np.minimum(np.maximum(v + a * dt, V_PRED_MIN), V_PRED_MAX)

    for t in range(steps):
        # ---- forecasts of every vehicle (N+1 points: x, y, s, v), all vehicles at once ----
        fc = np.zeros((B, N + 1, 4))
        # constant-acceleration forecast from the current state (constant_acceleration_model.py:18-82)
        a0 = u_prev[:, 0].copy()
        if gt and t == 0:
            a0 = 0.09 * (np.arange(B) % 2 + 1)                                             # evaluate.py:207-210
        sk = np.empty((B, N + 1)); vk = np.empty((B, N + 1))
        sk[:, 0], vk[:, 0] = z[:, 2], z[:, 5]
        for k in range(N):
            sk[:, k + 1], vk[:, k + 1] = ca_step(sk[:, k], vk[:, k], a0)
        fc[:, :, 0], fc[:, :, 1] = route_xy(sk)
        fc[:, 0, 0], fc[:, 0, 1] = z[:, 0], z[:, 1]
        fc[:, :, 2], fc[:, :, 3] = sk, vk
        if obca:
            fpsi = np.empty((B, N + 1))
            fpsi[:, 0] = z[:, 6]
            fpsi[:, 1:] = route_psi(sk[:, 1:])
        if t > 0 and prev_ok.any():
            # V2V: a vehicle that solved at t-1 is forecast by its previous plan shifted by one + one
            # constant-acceleration step (redone with a = 0 if that exceeds v = 5), utils.py:339-352
            v2v = np.where(prev_ok)[0]
            fc[v2v, :N, 0] = prev_x[v2v, 1:, 0]; fc[v2v, :N, 1] = prev_x[v2v, 1:, 1]
            fc[v2v, :N, 2] = prev_x[v2v, 1:, 2]; fc[v2v, :N, 3] = prev_x[v2v, 1:, 5]
            sN, vN = prev_x[:, N, 2], prev_x[:, N, 5]
            s1, v1 = ca_step(sN, vN, prev_u[:, N - 1, 0])
            s1b, v1b = ca_step(sN, vN, 0.0)
            over = v1 > 5
            s1, v1 = np.where(over, s1b, s1), np.where(over, v1b, v1)
            x1, y1 = route_xy(s1)
            fc[v2v, N, 0], fc[v2v, N, 1], fc[v2v, N, 2], fc[v2v, N, 3] = x1[v2v], y1[v2v], s1[v2v], v1[v2v]
            if obca:
                fpsi[v2v, :N] = prev_x[v2v, 1:, 6]
                fpsi[v2v, N] = route_psi(s1)[v2v]
        # ---- per-vehicle obstacle = the other vehicle's forecast; all of it moves to (-20, -20) if the other
        #      vehicle is behind the ego (negative dot product with the ego heading), utils.py:365-388 ----
        other = np.arange(B) ^ 1
        obs = fc[other][:, :, :2].copy()
        dx, dy = obs[:, 0, 0] - fc[:, 0, 0], obs[:, 0, 1] - fc[:, 0, 1]
        behind = dx * np.cos(z[:, 6]) + dy * np.sin(z[:, 6]) < 0
        obs[behind] = -20.0
        if obca:
            obs_psi = fpsi[other]
            obs_psi[flip[other]] = np.abs(obs_psi[flip[other]])
            obs_psi[behind] = 0.0
        # ---- solve: warm-started vehicles and cold ones in two batched calls ----
        t0 = time.perf_counter()
        u_init = np.concatenate([prev_u[:, 1:], prev_u[:, -1:]], axis=1)                   # utils.py:362
        out = dict(x=np.zeros((B, N + 1, 7)), u=np.zeros((B, N, 2)), status=np.ones(B, dtype=np.int32))
        nn_ctx = None
        if gt:
            other = np.arange(B) ^ 1
            nn_ctx = np.stack([fc[other, N, 2], fc[other, N, 3], enc[other], enc], axis=1)  # mpc.py:326-337
        warm_ok = prev_ok & (t > 1) if gt else prev_ok                                     # evaluate.py:232-235 / :478-481
        for mask, warm in ((warm_ok, True), (~warm_ok, False)):
            idx = np.where(mask)[0]
            if len(idx) == 0:
                continue
            kw = dict(nn_ctx=nn_ctx[idx]) if gt else {}
            if obca:
                kw["obs_psi"] = obs_psi[idx]
            if veh_net is not None:
                kw["net_idx"] = veh_net[idx]
            r = solver.solve_batch(z[idx], u_prev[idx], curv[idx], obs[idx], u_init=u_init[idx] if warm else None, **kw)
            out["x"][idx], out["u"][idx], out["status"][idx] = r["x"], r["u"], r["status"]
        if record_latency:
            lat.append(1e3 * (time.perf_counter() - t0))
        ok = np.isin(out["status"], _lib.STATUS_OK)        # converged or within the reference's own tolerances
        # ---- plant update ----
        z_next = z.copy(); u_app = np.zeros((B, 2))
        z_next[ok] = out["x"][ok, 1]                                                       # evaluate.py:493
        u_app[ok] = out["u"][ok, 0]
        bad = np.where(~ok)[0]
        if len(bad):
            ub = np.zeros((len(bad), N, 2))
            ub[:, :, 0] = np.where(z[bad, 5] > 0, A_MIN_BRAKE, 0.0)[:, None]               # evaluate.py:516
            ub[:, :, 1] = u_prev[bad, 1][:, None]
            roll = solver.evaluate(z[bad], u_prev[bad], curv[bad], np.full((len(bad), N + 1, 2), -20.0), ub)["x"][:, 1]
            for j, b in enumerate(bad):
                if z[b, 5] < 0:                                                            # evaluate.py:524-528
                    z_next[b] = z[b]; z_next[b, 5] = 0.0
                    u_app[b] = (0.0, u_prev[b, 1])
                else:
                    z_next[b] = roll[j]
                    u_app[b] = ub[j, 0]
        prev_x[ok], prev_u[ok] = out["x"][ok], out["u"][ok]
        prev_ok = ok
        z, u_prev = z_next, u_app
        z_cl[:, :, t + 1] = z.reshape(E, 2, 7); u_cl[:, :, t] = u_app.reshape(E, 2, 2)
        solved[:, :, t] = ok.reshape(E, 2)
    return _outcome(z_cl, u_cl, solved, d_min, ca_type, lat)


def run_closed_loop_device(solver, specs, steps=150, N=40, d_min=5.6, mode="mpc", record_latency=False, ca_type="circle",
                           net_idx=None):
    """The same closed loop with the per-timestep glue on the GPU (csrc/episode.cuh, igt_episode_run_host): all E
    episodes advance `steps` steps without the host in the loop -- per step one glue kernel, one batched solve of all 2E
    vehicles (per-problem warm / cold start), one plant kernel.  `solver` is a planner.BatchSolver (fp64) with horizon N.
    Returns an EpisodeResult; step_latency_ms = device time per step (all episodes together).
    ca_type 'obca' builds the obstacle heading forecast on the device as well (module docstring) and needs a solver
    made with d_min = 0 (mpc.py:42-43): with the circle gap of 5.6 m the rectangles would be kept that far apart.
    net_idx[E] (gt_mpc): bank slot of each episode, as in run_closed_loop (igt_episode_run_ex_host)."""
    import ctypes as C
    assert mode in ("mpc", "gt_mpc") and solver.N == N
    if net_idx is not None and mode != "gt_mpc":
        raise ValueError("net_idx selects value networks: mode 'gt_mpc' only")
    if ca_type not in ("circle", "obca"):
        raise ValueError("ca_type must be 'circle' or 'obca', got %r" % (ca_type,))
    if ca_type == "obca" and solver.params.d_min != 0:
        raise ValueError("ca_type='obca' needs a solver with d_min = 0 (mpc.py:42-43), this one has d_min = %g"
                         % solver.params.d_min)
    gt = mode == "gt_mpc"
    flags = (_lib.EPISODE_GT_MPC if gt else 0) | (_lib.EPISODE_OBCA if ca_type == "obca" else 0)
    E = len(specs)
    B = 2 * E
    rd = np.array([G.route_descriptor(r, exit_coord=G.EXIT_COORD.get(r)) for sp in specs for r in sp.routes], dtype=np.float64)
    curv = np.array([G.curvature_params(r) for sp in specs for r in sp.routes], dtype=np.float64)
    z = np.zeros((B, 7))
    for e, sp in enumerate(specs):
        for i in range(2):
            x, y, th = G.frenet2global(sp.s0[i], sp.routes[i])
            if sp.routes[i] in ('32', '41'):
                th = abs(th)
            z[2 * e + i] = (x, y, sp.s0[i], 0.0, 0.0, 0.0, th)
    u_prev = np.tile([0.0, 0.0] if gt else [0.1, 0.0], (B, 1)).astype(np.float64)
    enc = np.array([G.scenario_encoding(sp.routes) for sp in specs], dtype=np.float64).reshape(B)
    z_cl = np.zeros((E, 2, steps + 1, 7)); u_cl = np.zeros((E, 2, steps, 2)); solved = np.zeros((E, 2, steps), dtype=np.int32)
    ms = np.zeros(steps, dtype=np.float32)
    vp = lambda a: C.c_void_p(a.ctypes.data)
    nets = None
    if net_idx is not None:
        nets = np.ascontiguousarray(net_idx, dtype=np.int32)
        if nets.shape != (E,):
            raise ValueError("net_idx: one bank slot per episode, expected shape (%d,), got %s" % (E, nets.shape))
    rc = solver.lib.igt_episode_run_ex_host(solver._h, E, steps, flags, vp(rd), vp(curv), vp(z), vp(u_prev), vp(enc),
                                            None if nets is None else vp(nets), vp(z_cl), vp(u_cl), vp(solved),
                                            vp(ms) if record_latency else None)
    solver._check(rc, "igt_episode_run_ex_host")
    return _outcome(z_cl, u_cl, solved.astype(bool), d_min, ca_type, [float(v) for v in ms] if record_latency else [])
