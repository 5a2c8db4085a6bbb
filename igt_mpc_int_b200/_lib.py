"""ctypes binding of libigtmpc.so (the C ABI declared in include/igt_mpc.h).

There is no CPU fallback: if the shared library is missing, or no CUDA device is present when a
solver object is created, an exception is raised.  Build the library with
`python -m igt_mpc_int_b200.build` (nvcc, sm_100a) -- `__graft_entry__.build()` does that.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("IGT_LIB", os.path.join(_HERE, "lib", "libigtmpc.so"))   # IGT_LIB: developer override

MAX_CINF, MAX_LAYERS = 128, 5
MAX_MLP_NETS = 8        # value networks per handle (igt_set_mlp_at)
PREC_F32, PREC_F64 = 0, 1
STATUS_BAD_NET = 7      # a bank solve whose net_idx names no loaded network (igt_solve_ex_dev)
STATUS_NAMES = {0: "converged", 1: "max_iter", 2: "x0_infeasible", 3: "reg_limit", 4: "line_search",
                5: "stalled_infeasible", 6: "acceptable", 7: "bad_net"}
EPISODE_GT_MPC, EPISODE_OBCA = 1, 2   # mode bits of igt_episode_run_host
STATUS_OK = (0, 6)      # converged, or stopped within the reference's own IPOPT tolerances (igt_mpc.h: IGT_STATUS_ACCEPTABLE)

_dp = C.POINTER(C.c_double)
_fp = C.POINTER(C.c_float)
_ip = C.POINTER(C.c_int)


class IgtParams(C.Structure):
    """Mirror of `igt_params` (include/igt_mpc.h)."""
    _fields_ = [
        ("N", C.c_int), ("n_rk", C.c_int),
        ("dt", C.c_double), ("l_r", C.c_double), ("l_f", C.c_double),
        ("v_min", C.c_double), ("v_max", C.c_double), ("a_min", C.c_double), ("a_max", C.c_double),
        ("df_max", C.c_double), ("ey_lim", C.c_double),
        ("da_max", C.c_double), ("ddf_max", C.c_double),
        ("d_min", C.c_double), ("w_u", C.c_double),
        ("n_cinf", C.c_int),
        ("cinf_A", C.c_double * 2 * MAX_CINF), ("cinf_b", C.c_double * MAX_CINF),
        ("tol", C.c_double), ("tol_rp", C.c_double), ("tol_comp", C.c_double),
        ("mu0", C.c_double), ("mu_floor", C.c_double), ("kappa_eps", C.c_double), ("kappa_mu", C.c_double),
        ("theta_mu", C.c_double), ("y_init_min", C.c_double), ("tau_min", C.c_double),
        ("mu0_warm", C.c_double), ("y_init_min_warm", C.c_double),
        ("reg_min", C.c_double), ("reg_up", C.c_double), ("reg_down", C.c_double), ("reg_max", C.c_double),
        ("reg_jump", C.c_double),
        ("eps_phi", C.c_double), ("gamma_theta", C.c_double), ("theta_small", C.c_double),
        ("max_iter", C.c_int), ("n_alpha", C.c_int), ("second_order", C.c_int),
        ("stall_iter", C.c_int), ("stall_rp", C.c_double), ("max_trials", C.c_int), ("precision", C.c_int),
        ("acc_tol", C.c_double), ("acc_rp", C.c_double), ("acc_comp", C.c_double), ("x0_tol", C.c_double),
    ]

    def set_cinf(self, A, b):
        A = np.asarray(A, dtype=np.float64)
        b = np.asarray(b, dtype=np.float64)
        if A.shape[0] > MAX_CINF:
            raise ValueError("terminal set has too many rows")
        self.n_cinf = A.shape[0]
        for m in range(A.shape[0]):
            self.cinf_A[m][0], self.cinf_A[m][1] = float(A[m, 0]), float(A[m, 1])
            self.cinf_b[m] = float(b[m])


class IgtError(RuntimeError):
    pass


_lib = None

EXPORTS = ("igt_version", "igt_default_params", "igt_create", "igt_destroy", "igt_last_error",
           "igt_set_mlp", "igt_rollout_dev", "igt_rollout_host", "igt_eval_host", "igt_solve_dev",
           "igt_solve_host", "igt_launch_count", "igt_measure_fma_peak", "igt_mlp_value_host", "igt_set_option",
           "igt_episode_run_host", "igt_set_mlp_at", "igt_solve_ex_dev", "igt_solve_ex_host", "igt_eval_ex_host",
           "igt_mlp_value_ex_host", "igt_episode_run_ex_host", "igt_row_count", "igt_solve_duals_ex_dev",
           "igt_solve_duals_ex_host", "igt_solve_vjp_dev", "igt_solve_vjp_host")


def load():
    """dlopen libigtmpc.so and declare its prototypes.  Raises IgtError if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise IgtError("libigtmpc.so not found at %s -- build it with `python -m igt_mpc_int_b200.build`; "
                       "there is no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    lib.igt_version.restype = C.c_char_p
    lib.igt_default_params.argtypes = [C.POINTER(IgtParams), C.c_int]
    lib.igt_create.argtypes = [C.POINTER(IgtParams), C.POINTER(vp)]
    lib.igt_destroy.argtypes = [vp]
    lib.igt_destroy.restype = None
    lib.igt_last_error.argtypes = [vp]
    lib.igt_last_error.restype = C.c_char_p
    lib.igt_set_mlp.argtypes = [vp, C.c_int, _ip, C.POINTER(_dp), C.POINTER(_dp), _dp, _dp, C.c_double, C.c_double]
    lib.igt_rollout_dev.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp, vp, C.c_int, vp]
    lib.igt_rollout_host.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp, vp, C.c_int]
    lib.igt_eval_host.argtypes = [vp, C.c_int] + [vp] * 10
    lib.igt_solve_dev.argtypes = [vp, C.c_int] + [vp] * 13 + [vp]
    lib.igt_solve_host.argtypes = [vp, C.c_int] + [vp] * 13
    lib.igt_launch_count.argtypes = [vp]
    lib.igt_measure_fma_peak.argtypes = [vp, C.c_int, C.POINTER(C.c_double)]
    lib.igt_measure_fma_peak.restype = C.c_int
    lib.igt_mlp_value_host.argtypes = [vp, C.c_int, vp, vp, vp, vp, C.c_int]
    lib.igt_mlp_value_host.restype = C.c_int
    lib.igt_set_option.argtypes = [vp, C.c_char_p, C.c_double]
    lib.igt_set_option.restype = C.c_int
    lib.igt_launch_count.restype = C.c_longlong
    lib.igt_episode_run_host.argtypes = [vp, C.c_int, C.c_int, C.c_int] + [vp] * 9
    lib.igt_episode_run_host.restype = C.c_int
    lib.igt_set_mlp_at.argtypes = [vp, C.c_int, C.c_int, _ip, C.POINTER(_dp), C.POINTER(_dp), _dp, _dp, C.c_double, C.c_double]
    lib.igt_solve_ex_dev.argtypes = [vp, C.c_int] + [vp] * 14 + [vp]
    lib.igt_solve_ex_host.argtypes = [vp, C.c_int] + [vp] * 14
    lib.igt_eval_ex_host.argtypes = [vp, C.c_int] + [vp] * 11
    lib.igt_mlp_value_ex_host.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp, C.c_int]
    lib.igt_episode_run_ex_host.argtypes = [vp, C.c_int, C.c_int, C.c_int] + [vp] * 10
    lib.igt_row_count.argtypes = [vp]
    lib.igt_solve_duals_ex_dev.argtypes = [vp, C.c_int] + [vp] * 16 + [vp]
    lib.igt_solve_duals_ex_host.argtypes = [vp, C.c_int] + [vp] * 16
    lib.igt_solve_vjp_dev.argtypes = [vp, C.c_int] + [vp] * 17 + [vp]
    lib.igt_solve_vjp_host.argtypes = [vp, C.c_int] + [vp] * 17
    for f in ("igt_set_mlp_at", "igt_solve_ex_dev", "igt_solve_ex_host", "igt_eval_ex_host", "igt_mlp_value_ex_host",
              "igt_episode_run_ex_host", "igt_row_count", "igt_solve_duals_ex_dev", "igt_solve_duals_ex_host",
              "igt_solve_vjp_dev", "igt_solve_vjp_host"):
        getattr(lib, f).restype = C.c_int
    for f in ("igt_default_params", "igt_create", "igt_set_mlp", "igt_rollout_dev", "igt_rollout_host",
              "igt_eval_host", "igt_solve_dev", "igt_solve_host"):
        getattr(lib, f).restype = C.c_int
    _lib = lib
    return lib


def default_params(precision=PREC_F64):
    p = IgtParams()
    rc = load().igt_default_params(C.byref(p), precision)
    if rc != 0:
        raise IgtError("igt_default_params failed (%d)" % rc)
    return p
