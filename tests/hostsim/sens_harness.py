"""TEST HARNESS ONLY: run the product's dual-exporting solve epilogue and VJP code (csrc/sens.cuh) on the CPU
(see sens_hostsim.cu)."""
import ctypes as C
import os
import subprocess

import numpy as np

from igt_mpc_int_b200._lib import IgtParams

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libsenshost.so")
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


def build():
    src = os.path.join(_HERE, "sens_hostsim.cu")
    deps = [src] + [os.path.join(_HERE, "..", "..", "igt_mpc_int_b200", "csrc", f)
                    for f in ("solver_core.cuh", "sens.cuh", "params_host.hpp", "obca.cuh", "mlp_coop.cuh", "mlp_tc.cuh")]
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
    lib().senshost_default_params(C.byref(p), precision)
    return p


def _c(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return None if a is None else a.ctypes.data_as(_dp)


def _net_args(mlp):
    """(n_layers, dims, W, b, Wn, mu_f, sigma_t, mu_t, keep-alive list) of an nlp.MLPTerm or None"""
    if mlp is None:
        return 0, None, None, None, None, None, C.c_double(0.0), C.c_double(0.0), []
    n = len(mlp.weights)
    d = [mlp.weights[0][0].shape[1]] + [W.shape[0] for W, _ in mlp.weights]
    Ws = [_c(W) for W, _ in mlp.weights]; bs = [_c(b) for _, b in mlp.weights]
    Wn, mu_f = _c(mlp.Wn), _c(mlp.mu_f)
    return (n, (C.c_int * len(d))(*d), (_dp * n)(*[_ptr(w) for w in Ws]), (_dp * n)(*[_ptr(b) for b in bs]), _ptr(Wn),
            _ptr(mu_f), C.c_double(float(mlp.sigma_t)), C.c_double(float(mlp.mu_t)), Ws + bs + [Wn, mu_f])


def solve_duals(p, x0, u_prev, curv, obs, nn_ctx=None, u_init=None, mlp=None):
    """fp64 circle-mode solve of the product code that also returns every row's final slack Y[B,M] and multiplier
    S[B,M] (the epilogue of the dual-exporting kernels)"""
    x0, u_prev, curv, obs, nn_ctx, u_init = map(_c, (x0, u_prev, curv, obs, nn_ctx, u_init))
    B, N = x0.shape[0], p.N
    M = 8 + 13 * (N - 1) + p.n_cinf + 3
    Z = np.empty((B, N + 1, 7)); U = np.empty((B, N, 2)); cost = np.empty(B); viol = np.empty(B)
    status = np.empty(B, dtype=np.int32); iters = np.empty(B, dtype=np.int32)
    Y = np.empty((B, M)); S = np.empty((B, M))
    n, dims, Wp, bp, Wn, mu_f, st, mt, keep = _net_args(mlp)
    rc = lib().senshost_solve_duals(C.byref(p), B, _ptr(x0), _ptr(u_prev), _ptr(curv), _ptr(obs), _ptr(nn_ctx),
                                    _ptr(u_init), _ptr(Z), _ptr(U), _ptr(cost), _ptr(viol), status.ctypes.data_as(_ip),
                                    iters.ctypes.data_as(_ip), _ptr(Y), _ptr(S), n, dims, Wp, bp, Wn, mu_f, st, mt)
    assert rc == 0
    return dict(Z=Z, U=U, cost=cost, viol=viol, status=status, iters=iters, Y=Y, S=S)


def vjp(p, x0, u_prev, curv, obs, U, Y, S, status, gx=None, gu=None, gcost=None, nn_ctx=None, mlp=None):
    """csrc/sens.cuh's VJP on the CPU: (gx0[B,7], gu_prev[B,2], gobs[B,N+1,2], ok[B])"""
    x0, u_prev, curv, obs, U, Y, S, gx, gu, gcost, nn_ctx = map(_c, (x0, u_prev, curv, obs, U, Y, S, gx, gu, gcost, nn_ctx))
    status = np.ascontiguousarray(status, dtype=np.int32)
    B, N = x0.shape[0], p.N
    gx0 = np.empty((B, 7)); gup = np.empty((B, 2)); gobs = np.empty((B, N + 1, 2)); ok = np.empty(B, dtype=np.int32)
    n, dims, Wp, bp, Wn, mu_f, st, mt, keep = _net_args(mlp)
    rc = lib().senshost_vjp(C.byref(p), B, _ptr(x0), _ptr(u_prev), _ptr(curv), _ptr(obs), _ptr(nn_ctx), _ptr(U), _ptr(Y),
                            _ptr(S), status.ctypes.data_as(_ip), _ptr(gx), _ptr(gu), _ptr(gcost), _ptr(gx0), _ptr(gup),
                            _ptr(gobs), ok.ctypes.data_as(_ip), n, dims, Wp, bp, Wn, mu_f, st, mt)
    assert rc == 0
    return gx0, gup, gobs, ok
