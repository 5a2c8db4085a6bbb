"""Host-side mirror of the reference planner interface over the CUDA solver.

* `BatchSolver`  -- the batched API: one call solves B independent MPC problems
  (scenario x vehicle x sampled initial condition) on the GPU.
* `MPC_Planner`  -- drop-in for the reference class of the same name (mpc.py:19-406): same
  constructor keywords, `update_initial_condition`, `update_predictions`, `solve`, and the
  read-after-solve attributes `solve_time`, `NN_query_time`, `x_sol_prev`, `sol.stats()`.

Everything numeric happens behind the C ABI of include/igt_mpc.h (libigtmpc.so); this module
only marshals numbers.  No CPU fallback exists: creating a solver without the CUDA library or
without a GPU raises.
"""
import ctypes as C
import math
import time

import numpy as np

from . import _lib
from . import geometry as G
from . import terminal_set

_vp = C.c_void_p


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None and tuple(a.shape) != tuple(shape):
        raise ValueError("expected shape %s, got %s" % (tuple(shape), tuple(a.shape)))
    return a


def _hp(a):
    return None if a is None else _vp(a.ctypes.data)


def _net_idx(net_idx, B):
    """per-problem bank slots as a contiguous int32 [B] array (None stays None)"""
    if net_idx is None:
        return None
    a = np.ascontiguousarray(net_idx, dtype=np.int32)
    if a.shape != (B,):
        raise ValueError("net_idx: expected shape (%d,), got %s" % (B, a.shape))
    return a


_CINF_CACHE = {}


def _cinf_table(dt, jerk_limit):
    key = (float(dt), float(jerk_limit))
    if key not in _CINF_CACHE:
        _CINF_CACHE[key] = terminal_set.cinf(dt=dt, jerk_limit=jerk_limit)   # mpc.py:88-104
    return _CINF_CACHE[key]


class BatchSolver:
    """Batched MPC solve on the GPU.

    precision: 'f64' (default; parity path) or 'f32'.  `options` override fields of
    `igt_params` (include/igt_mpc.h), e.g. tol=..., max_iter=..., mu0=...
    mlp: optional dict(weights=[(W, b), ...], Wn=6x6, mu_f=[6], sigma_t=float, mu_t=float)
    enabling the gt_mpc terminal cost (mpc.py:105-127, :367-369), or a list of at most 8 such dicts (None: an empty
    slot): a network bank, entry k in slot k.  Calls with `net_idx` pick a slot per problem (the reference's
    network k for scenario k, evaluate.py:123); calls without it use slot 0.
    """

    def __init__(self, N=40, dt=0.1, n_rk=4, precision="f64", mlp=None, jerk_limit=0.9,
                 steering_rate_limit=0.7, d_min=5.6, **options):
        self.lib = _lib.load()
        prec = {"f64": _lib.PREC_F64, "f32": _lib.PREC_F32}[precision]
        p = _lib.default_params(prec)
        p.N, p.dt, p.n_rk = int(N), float(dt), int(n_rk)
        p.da_max, p.ddf_max, p.d_min = dt * jerk_limit, dt * steering_rate_limit, float(d_min)
        A, b = _cinf_table(dt, jerk_limit)
        p.set_cinf(A, b)
        for k, v in options.items():
            if not hasattr(p, k):
                raise KeyError("unknown solver option %r" % k)
            setattr(p, k, v)
        self.params = p
        self.N = int(N)
        self.precision = precision
        h = _vp()
        rc = self.lib.igt_create(C.byref(p), C.byref(h))
        if rc != 0:
            raise _lib.IgtError("igt_create failed (%d): %s" % (rc, self.lib.igt_last_error(None).decode()))
        self._h = h
        self.has_mlp = False
        if isinstance(mlp, (list, tuple)):
            if len(mlp) > _lib.MAX_MLP_NETS:
                raise ValueError("a network bank holds at most %d networks, got %d" % (_lib.MAX_MLP_NETS, len(mlp)))
            for k, net in enumerate(mlp):
                if net is not None:
                    self.set_mlp(**net, net=k)
        elif mlp is not None:
            self.set_mlp(**mlp)

    # -- lifetime --------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self.lib.igt_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise _lib.IgtError("%s failed (%d): %s" % (what, rc, self.lib.igt_last_error(self._h).decode()))

    @property
    def launches(self):
        return int(self.lib.igt_launch_count(self._h))

    def measure_fma_peak(self, precision=None):
        """TFLOP/s of dependent-free FMA chains (the solver kernels' compute roofline)."""
        prec = self.params.precision if precision is None else {"f64": _lib.PREC_F64, "f32": _lib.PREC_F32}[precision]
        out = C.c_double()
        self._check(self.lib.igt_measure_fma_peak(self._h, prec, C.byref(out)), "igt_measure_fma_peak")
        return out.value

    # -- value network ---------------------------------------------------------------------
    def set_mlp(self, weights, Wn, mu_f, sigma_t, mu_t, net=0):
        """load a value network into bank slot `net` (0 = the network of calls without net_idx)"""
        n = len(weights)
        Ws = [_f64(W) for W, _ in weights]
        bs = [_f64(b).ravel() for _, b in weights]
        dims = [Ws[0].shape[1]] + [W.shape[0] for W in Ws]
        dp = C.POINTER(C.c_double)
        Wp = (dp * n)(*[w.ctypes.data_as(dp) for w in Ws])
        bp = (dp * n)(*[b.ctypes.data_as(dp) for b in bs])
        Wn, mu_f = _f64(Wn, (6, 6)), _f64(mu_f, (6,))
        rc = self.lib.igt_set_mlp_at(self._h, int(net), n, (C.c_int * len(dims))(*dims), Wp, bp, Wn.ctypes.data_as(dp),
                                     mu_f.ctypes.data_as(dp), float(sigma_t), float(mu_t))
        self._check(rc, "igt_set_mlp_at")
        self.has_mlp = True

    def set_option(self, name, value):
        self._check(self.lib.igt_set_option(self._h, name.encode(), float(value)), "igt_set_option")

    def mlp_value(self, sN, vN, nn_ctx, tensor_cores=True, net_idx=None):
        """Value term and its (s_N, v_N) derivatives: out[B,6] = (V, Vs, Vv, Vss, Vsv, Vvv).
        tensor_cores: True / 1 tcgen05 kernel, False / 0 per-thread fp64, 2 the solver's cooperative fp64 evaluation.
        net_idx[B]: bank slot of each row (modes 0 and 2 only)."""
        sN = _f64(sN).ravel(); B = sN.shape[0]
        vN = _f64(vN, (B,)); nn_ctx = _f64(nn_ctx, (B, 4))
        out = np.empty((B, 6))
        rc = self.lib.igt_mlp_value_ex_host(self._h, B, _hp(sN), _hp(vN), _hp(nn_ctx), _hp(_net_idx(net_idx, B)), _hp(out),
                                            int(tensor_cores))
        self._check(rc, "igt_mlp_value_ex_host")
        return out

    # -- host-pointer calls (copies inside) ---------------------------------------------------
    def solve_batch(self, x0, u_prev, curv, obs_xy, nn_ctx=None, u_init=None, out=None, obs_psi=None, net_idx=None):
        """numpy in / numpy out.  Returns dict(x[B,N+1,7], u[B,N,2], cost, viol, status, iters).
        obs_psi[B,N+1] (obstacle heading forecast) selects the OBCA collision rows (mpc.py:211-221).
        net_idx[B] (with nn_ctx): the bank slot of each problem's value network; an index that names no loaded
        network raises IgtError before anything runs."""
        N = self.N
        x0 = _f64(x0)
        B = x0.shape[0]
        x0 = _f64(x0, (B, 7)); u_prev = _f64(u_prev, (B, 2)); curv = _f64(curv, (B, 3))
        obs_xy = _f64(obs_xy, (B, N + 1, 2))
        nn_ctx = None if nn_ctx is None else _f64(nn_ctx, (B, 4))
        u_init = None if u_init is None else _f64(u_init, (B, N, 2))
        obs_psi = None if obs_psi is None else _f64(obs_psi, (B, N + 1))
        if out is None:
            out = dict(x=np.empty((B, N + 1, 7)), u=np.empty((B, N, 2)), cost=np.empty(B), viol=np.empty(B),
                       status=np.empty(B, dtype=np.int32), iters=np.empty(B, dtype=np.int32))
        rc = self.lib.igt_solve_ex_host(self._h, B, _hp(x0), _hp(u_prev), _hp(curv), _hp(obs_xy), _hp(obs_psi), _hp(nn_ctx),
                                        _hp(_net_idx(net_idx, B)), _hp(u_init), _hp(out["x"]), _hp(out["u"]),
                                        _hp(out["cost"]), _hp(out["viol"]), _hp(out["status"]), _hp(out["iters"]))
        self._check(rc, "igt_solve_ex_host")
        return out

    def evaluate(self, x0, u_prev, curv, obs_xy, u, nn_ctx=None, obs_psi=None, net_idx=None):
        """Cost (mpc.py:356-373) and max inequality-row value of given controls (net_idx: as in solve_batch)."""
        N = self.N
        x0 = _f64(x0)
        B = x0.shape[0]
        u_prev = _f64(u_prev, (B, 2)); curv = _f64(curv, (B, 3)); obs_xy = _f64(obs_xy, (B, N + 1, 2))
        u = _f64(u, (B, N, 2))
        nn_ctx = None if nn_ctx is None else _f64(nn_ctx, (B, 4))
        obs_psi = None if obs_psi is None else _f64(obs_psi, (B, N + 1))
        cost, viol, z = np.empty(B), np.empty(B), np.empty((B, N + 1, 7))
        rc = self.lib.igt_eval_ex_host(self._h, B, _hp(x0), _hp(u_prev), _hp(curv), _hp(obs_xy), _hp(obs_psi), _hp(nn_ctx),
                                       _hp(_net_idx(net_idx, B)), _hp(u), _hp(cost), _hp(viol), _hp(z))
        self._check(rc, "igt_eval_ex_host")
        return dict(cost=cost, viol=viol, x=z)

    def rollout(self, z0, u, curv=None, jac=False, model=0):
        """fp32 rollout (+ Jacobians).  model 0: Frenet RK4 (z0[B,7]); model 1: Cartesian Euler
        (z0[B,4] = x, y, psi, v)."""
        N = self.N
        nz = 7 if model == 0 else 4
        z0 = np.ascontiguousarray(z0, dtype=np.float32)
        B = z0.shape[0]
        u = np.ascontiguousarray(u, dtype=np.float32)
        if z0.shape != (B, nz) or u.shape != (B, N, 2):
            raise ValueError("bad rollout shapes")
        curv = np.zeros((B, 3), np.float32) if curv is None else np.ascontiguousarray(curv, dtype=np.float32)
        z = np.empty((B, N + 1, nz), np.float32)
        A = np.empty((B, N, nz, nz), np.float32) if jac else None
        Bm = np.empty((B, N, nz, 2), np.float32) if jac else None
        rc = self.lib.igt_rollout_host(self._h, B, _hp(z0), _hp(u), _hp(curv), _hp(z), _hp(A), _hp(Bm), model)
        self._check(rc, "igt_rollout_host")
        return (z, A, Bm) if jac else z

    # -- device-pointer call (torch tensors already in HBM; no copies, no sync) ---------------
    def solve_batch_device(self, x0, u_prev, curv, obs_xy, nn_ctx=None, u_init=None, out=None, stream=None, obs_psi=None,
                           net_idx=None):
        """torch CUDA float64 tensors in / out; enqueues on the current torch stream.
        net_idx: int32 device tensor [B] of bank slots (with nn_ctx); checked in the kernel: a problem whose index
        names no loaded network gets status 7 (STATUS_BAD_NET) and NaN outputs."""
        import torch
        N = self.N
        B = x0.shape[0]
        dev = x0.device

        def check(t, shp, dtype, name):
            if not (t.is_cuda and t.device == dev and t.dtype == dtype and t.is_contiguous() and tuple(t.shape) == shp):
                raise ValueError("%s: expected a contiguous %s tensor of shape %s on %s" % (name, dtype, shp, dev))

        for t, shp, name in ((x0, (B, 7), "x0"), (u_prev, (B, 2), "u_prev"), (curv, (B, 3), "curv"),
                             (obs_xy, (B, N + 1, 2), "obs_xy"), (nn_ctx, (B, 4), "nn_ctx"), (u_init, (B, N, 2), "u_init"),
                             (obs_psi, (B, N + 1), "obs_psi")):
            if t is not None:
                check(t, shp, torch.float64, name)
        if net_idx is not None:
            check(net_idx, (B,), torch.int32, "net_idx")
        if out is None:
            out = dict(x=torch.empty((B, N + 1, 7), dtype=torch.float64, device=dev),
                       u=torch.empty((B, N, 2), dtype=torch.float64, device=dev),
                       cost=torch.empty(B, dtype=torch.float64, device=dev),
                       viol=torch.empty(B, dtype=torch.float64, device=dev),
                       status=torch.empty(B, dtype=torch.int32, device=dev),
                       iters=torch.empty(B, dtype=torch.int32, device=dev))
        else:
            for k, shp, dt in (("x", (B, N + 1, 7), torch.float64), ("u", (B, N, 2), torch.float64), ("cost", (B,), torch.float64),
                               ("viol", (B,), torch.float64), ("status", (B,), torch.int32), ("iters", (B,), torch.int32)):
                check(out[k], shp, dt, "out[%r]" % k)
        st = torch.cuda.current_stream(dev).cuda_stream if stream is None else stream
        p = lambda t: None if t is None else _vp(t.data_ptr())
        rc = self.lib.igt_solve_ex_dev(self._h, B, p(x0), p(u_prev), p(curv), p(obs_xy), p(obs_psi), p(nn_ctx), p(net_idx),
                                       p(u_init), p(out["x"]), p(out["u"]), p(out["cost"]), p(out["viol"]),
                                       p(out["status"]), p(out["iters"]), _vp(st))
        self._check(rc, "igt_solve_ex_dev")
        return out


# ---------------------------------------------------------------------------------------------
class _Sol:
    """Stand-in for the CasADi OptiSol object the reference keeps in `planner.sol`
    (evaluate.py:294-297, :549-552 read `sol.stats()` 't_wall_*' keys)."""

    def __init__(self, t_wall, iters, status):
        self._stats = {"t_wall_total": t_wall, "t_proc_total": t_wall, "iter_count": int(iters),
                       "return_status": _lib.STATUS_NAMES.get(int(status), "unknown"),
                       "success": int(status) in _lib.STATUS_OK}

    def stats(self):
        return dict(self._stats)


class MPC_Planner:
    """Drop-in for reference mpc.py `MPC_Planner` (constructor :21-37; protocol :241-294, :383-406).

    Objects passed in follow the reference's attribute-bag types (common/VehicleState.py,
    VehicleAction.py, VehicleReference.py): `.x .y .heading .v .s .ey .epsi` and `.a .df`.
    `solve` returns `(x[7,N+1], u[2,N], True)` fp64 numpy arrays or `(None, None, False)`;
    like the reference it never raises on solver failure (mpc.py:402-406).
    """

    def __init__(self, N=10, dt=0.1, agents=None, goals=None, ca_radius=2.8, ref=None, road_dim=(10, 50),
                 routes=None, ds_right=None, index=None, num_rk4_steps=7, solver='ipopt', ca_type='circle',
                 nn_config_dir=None, use_NN_cost2go=False, weights=[1, 1, 1], nn_model=None,
                 precision="f64", **options):
        assert index is not None                                        # mpc.py:80
        assert agents is not None, 'Agents are not defined'             # mpc.py:155
        if ca_type not in ('circle', 'obca'):
            raise ValueError("collision_avoidance_type must be 'circle' or 'obca' (mpc.yaml:15-16)")
        self.N, self.dt, self.ca_type = N, dt, ca_type
        self.x_sol_prev = None
        self.d_min = 0 if ca_type == 'obca' else 2 * ca_radius          # mpc.py:42-45
        self.routes, self.ind = routes, index
        self.agents, self.goals, self.ref = agents, goals, ref
        self.initial_agent = agents[index]
        self.M = len(ref) if ref is not None else len(agents)
        self.num_obstacles = self.M - 1
        if self.num_obstacles > 1:
            raise NotImplementedError("the reference scenarios have two vehicles (fourwayint.yaml:10)")
        self.pred_ind = [i for i in range(self.M) if i != index]
        self.road_width, self.road_length = road_dim
        self.ds_right = ds_right
        self.weights = weights
        self.use_NN_cost2go = use_NN_cost2go
        self.nn_config_dir = nn_config_dir
        self.solve_time = 0.0
        self.NN_query_time = -1
        self.sol = None
        self.curv = self._curvature_params()
        self._solver = BatchSolver(N=N, dt=dt, n_rk=num_rk4_steps, d_min=self.d_min, precision=precision,
                                   mlp=nn_model, **options)
        if use_NN_cost2go and nn_model is None:
            raise ValueError("use_NN_cost2go needs nn_model=dict(weights, Wn, mu_f, sigma_t, mu_t); the "
                             "reference unpickles them from a dataset that is not shipped (mpc.py:105-118)")
        self._x0 = np.zeros((1, 7)); self._uprev = np.zeros((1, 2))
        self._obs = np.full((1, N + 1, 2), -20.0); self._ctx = np.zeros((1, 4))
        self._obs_psi = np.zeros((1, N + 1))                            # obstacle heading forecast (OBCA rows only)

    # mpc.py:183-200 -- curvature of this agent's route as (b0, b1, Kval)
    def _curvature_params(self):
        K = None if self.ref is None else np.asarray(self.ref[self.ind]['K'])
        if K is None or np.all(K == 0):
            return np.array([[1e30, 1e30, 0.0]])
        nz = K[np.nonzero(K)]
        r = float(np.max(np.abs(1.0 / nz)))
        half = (self.road_length - self.road_width) / 2
        b0 = half if self.routes[self.ind] in G.LEFT else half - self.ds_right
        return np.array([[b0, b0 + r * math.pi / 2, float(nz[0])]])

    def set_reference(self, ref):
        self.ref = ref

    # mpc.py:280-294
    def update_initial_condition(self, agent, u_prev):
        st = agent['state']
        heading = abs(st.heading) if self.routes[self.ind] in ['32', '41'] else st.heading
        self._x0[0] = (st.x, st.y, st.s, st.ey, st.epsi, st.v, heading)
        self._uprev[0] = (u_prev.a, u_prev.df)
        self.u_prev_raw = u_prev
        self.initial_agent = agent

    # mpc.py:241-278
    def update_predictions(self, preds, raw_preds=None):
        assert len(preds) == self.M, ValueError('Invalid number of predictions')
        self.pred_ind = []
        for i, pred in enumerate(preds):
            if i != self.ind:
                self.pred_ind.append(i)
                assert len(pred) == self.N + 1, ValueError('Invalid prediction length (Horizon)')
                flip = self.routes[i] in ['32', '41']                   # mpc.py:250-253
                for k in range(self.N + 1):
                    self._obs[0, k] = (pred[k].x, pred[k].y)
                    if self.ca_type == 'obca':
                        self._obs_psi[0, k] = abs(pred[k].heading) if flip else pred[k].heading
        if raw_preds is not None:
            j = self.pred_ind[0]
            enc = G.scenario_encoding(self.routes)
            self._ctx[0] = (raw_preds[j][-1].s, raw_preds[j][-1].v, enc[j], enc[self.ind])   # mpc.py:326-337
        self.NN_query_time = -1

    # mpc.py:383-406
    def solve(self, x_sol_prev=None, u_sol_prev=None):
        try:
            u_init = None if u_sol_prev is None else np.ascontiguousarray(np.asarray(u_sol_prev, dtype=np.float64).T)[None]
            t0 = time.time()
            out = self._solver.solve_batch(self._x0, self._uprev, self.curv, self._obs,
                                           nn_ctx=self._ctx if self.use_NN_cost2go else None, u_init=u_init,
                                           obs_psi=self._obs_psi if self.ca_type == 'obca' else None)
            self.solve_time = time.time() - t0
            self.sol = _Sol(self.solve_time, out["iters"][0], out["status"][0])
            if int(out["status"][0]) not in _lib.STATUS_OK:   # IPOPT: Solve_Succeeded covers both (igt_mpc.h)
                raise RuntimeError(_lib.STATUS_NAMES.get(int(out["status"][0]), "failed"))
            x = np.ascontiguousarray(out["x"][0].T)       # [7, N+1]
            u = np.ascontiguousarray(out["u"][0].T)       # [2, N]
            self.x_sol_prev = x
            return (x, u, True)
        except _lib.IgtError:
            raise                                          # API misuse / no GPU is not a solver failure
        except Exception:
            print('NLP SOLVE FAILED'.center(80, '*'))
            return (None, None, False)
