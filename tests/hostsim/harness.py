"""TEST HARNESS ONLY: run the product's per-thread solver code on the CPU (see hostsim.cu)."""
import ctypes as C
import os
import subprocess

import numpy as np

from igt_mpc_int_b200._lib import IgtParams

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libhostsim.so")
_dp = C.POINTER(C.c_double)


def build():
    src = os.path.join(_HERE, "hostsim.cu")
    deps = [src] + [os.path.join(_HERE, "..", "..", "igt_mpc_int_b200", "csrc", f)
                    for f in ("solver_core.cuh", "params_host.hpp", "obca.cuh", "mlp_coop.cuh", "mlp_tc.cuh")]
    if not os.path.exists(_SO) or any(os.path.getmtime(_SO) < os.path.getmtime(d) for d in deps):
        subprocess.check_call(["nvcc", "-O2", "-std=c++17", "--expt-relaxed-constexpr", "-Wno-deprecated-gpu-targets",
                               "-Xcompiler", "-fPIC", "-shared", "-o", _SO, src])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
    return _lib


def default_params(precision):
    p = IgtParams()
    lib().hostsim_default_params(C.byref(p), precision)
    return p


def _c(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return None if a is None else a.ctypes.data_as(_dp)


def solve(p, x0, u_prev, curv, obs, nn_ctx=None, u_init=None, mlp=None, lanes=False):
    """lanes: one solver object per slot reused for problems q, q + 32, ... (persistent lanes) instead of a fresh one
    per problem"""
    x0, u_prev, curv, obs, nn_ctx, u_init = map(_c, (x0, u_prev, curv, obs, nn_ctx, u_init))
    B, N = x0.shape[0], p.N
    Z = np.empty((B, N + 1, 7)); U = np.empty((B, N, 2)); cost = np.empty(B); viol = np.empty(B)
    status = np.empty(B, dtype=np.int32); iters = np.empty(B, dtype=np.int32)
    n_layers, dims, Wp, bp, Wn, mu_f, st, mt, keep = 0, None, None, None, None, None, 0.0, 0.0, []
    if mlp is not None:
        n_layers = len(mlp.weights)
        d = [mlp.weights[0][0].shape[1]] + [W.shape[0] for W, _ in mlp.weights]
        dims = (C.c_int * len(d))(*d)
        Ws = [_c(W) for W, _ in mlp.weights]; bs = [_c(b) for _, b in mlp.weights]
        keep = Ws + bs
        Wp = (_dp * n_layers)(*[_ptr(w) for w in Ws]); bp = (_dp * n_layers)(*[_ptr(b) for b in bs])
        Wn = _c(mlp.Wn); mu_f = _c(mlp.mu_f); st, mt = float(mlp.sigma_t), float(mlp.mu_t)
        keep += [Wn, mu_f]
    rc = lib().hostsim_solve(C.byref(p), B, _ptr(x0), _ptr(u_prev), _ptr(curv), _ptr(obs), _ptr(nn_ctx), _ptr(u_init),
                             _ptr(Z), _ptr(U), _ptr(cost), _ptr(viol), status.ctypes.data_as(C.POINTER(C.c_int)),
                             iters.ctypes.data_as(C.POINTER(C.c_int)), n_layers, dims, Wp, bp, _ptr(Wn), _ptr(mu_f),
                             C.c_double(st), C.c_double(mt), int(bool(lanes)))
    assert rc == 0
    return dict(Z=Z, U=U, cost=cost, viol=viol, status=status, iters=iters)


def rollout(p, prec, z0, U, curv, jac=False):
    z0, U, curv = map(_c, (z0, U, curv))
    B, N = U.shape[0], p.N
    Z = np.empty((B, N + 1, 7))
    A = np.empty((B, N, 7, 7)) if jac else None
    Bm = np.empty((B, N, 7, 2)) if jac else None
    rc = lib().hostsim_rollout(C.byref(p), B, prec, _ptr(z0), _ptr(U), _ptr(curv), _ptr(Z), _ptr(A), _ptr(Bm))
    assert rc == 0, "value-only and sensitivity RK4 steps disagree"
    return (Z, A, Bm) if jac else Z


def solve_obca(p, x0, u_prev, curv, obs, obs_psi, u_init=None, lanes=False):
    """product solver code (OBCA collision rows, fp64) on the CPU; lanes: as in solve"""
    x0, u_prev, curv, obs, obs_psi, u_init = map(_c, (x0, u_prev, curv, obs, obs_psi, u_init))
    B, N = x0.shape[0], p.N
    Z = np.empty((B, N + 1, 7)); U = np.empty((B, N, 2)); cost = np.empty(B); viol = np.empty(B)
    status = np.empty(B, dtype=np.int32); iters = np.empty(B, dtype=np.int32)
    rc = lib().hostsim_solve_obca(C.byref(p), B, _ptr(x0), _ptr(u_prev), _ptr(curv), _ptr(obs), _ptr(obs_psi), _ptr(u_init),
                                  _ptr(Z), _ptr(U), _ptr(cost), _ptr(viol), status.ctypes.data_as(C.POINTER(C.c_int)),
                                  iters.ctypes.data_as(C.POINTER(C.c_int)), int(bool(lanes)))
    assert rc == 0
    return dict(Z=Z, U=U, cost=cost, viol=viol, status=status, iters=iters)


def rect_sdist(ego, obs):
    ego, obs = _c(ego), _c(obs)
    n = ego.shape[0]
    d = np.empty(n); g = np.empty((n, 3))
    lib().hostsim_rect_sdist(n, _ptr(ego), _ptr(obs), _ptr(d), _ptr(g))
    return d, g
