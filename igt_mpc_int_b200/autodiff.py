"""torch autograd through the batched solve.

`solve(solver, x0, u_prev, curv, obs_xy, ...)` runs a dual-exporting solve on the GPU (BatchSolver.solve_batch_device
with duals=True) and returns x, u, cost, status and ok as torch tensors; x, u and cost carry a grad_fn.  The backward
pass is one call of the VJP kernel (csrc/sens.cuh, BatchSolver.vjp_device): the implicit function theorem on the
solve's converged KKT system, so gradients flow to x0, u_prev and obs_xy.  Never raises on a solver failure: a problem
that did not converge (status != 0) or whose stage Hessian is not positive definite gets zero gradient, and
`ok` (int32, filled in by the backward pass; all zero until then) marks the problems whose gradient is exact.
Out of scope: gradients w.r.t. nn_ctx, curv, u_init and network weights (DESIGN.md section 10).
"""
import torch


class _SolveFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x0, u_prev, obs_xy, solver, curv, nn_ctx, net_idx, u_init, ok):
        out = solver.solve_batch_device(x0.detach(), u_prev.detach(), curv, obs_xy.detach(), nn_ctx=nn_ctx, u_init=u_init,
                                        net_idx=net_idx, duals=True)
        ctx.solver = solver
        ctx.ok = ok
        ctx.save_for_backward(x0, u_prev, obs_xy, curv, *(t for t in (nn_ctx, net_idx) if t is not None), out["u"],
                              out["slack"], out["mult"], out["status"])
        ctx.has = (nn_ctx is not None, net_idx is not None)
        ctx.mark_non_differentiable(out["status"])
        return out["x"], out["u"], out["cost"], out["status"]

    @staticmethod
    def backward(ctx, gx, gu, gcost, _gstatus):
        saved = list(ctx.saved_tensors)
        x0, u_prev, obs_xy, curv = saved[:4]
        rest = saved[4:]
        nn_ctx = rest.pop(0) if ctx.has[0] else None
        net_idx = rest.pop(0) if ctx.has[1] else None
        u, slack, mult, status = rest
        c = lambda t: None if t is None else t.contiguous()
        g = ctx.solver.vjp_device(x0.detach(), u_prev.detach(), curv, obs_xy.detach(), u, slack, mult, status, gx=c(gx),
                                  gu=c(gu), gcost=c(gcost), nn_ctx=nn_ctx, net_idx=net_idx)
        ctx.ok.copy_(g["ok"])
        return g["gx0"], g["gu_prev"], g["gobs"], None, None, None, None, None, None


def solve(solver, x0, u_prev, curv, obs_xy, nn_ctx=None, net_idx=None, u_init=None):
    """Differentiable batched solve.  solver: a BatchSolver (f64; 'mpc' or gt_mpc with one network or a bank, exact
    value term); tensors as solve_batch_device takes them.  Returns (x, u, cost, status, ok): gradients of a loss of
    x, u, cost flow to x0, u_prev and obs_xy; ok[B] (int32) is written by the backward pass."""
    ok = torch.zeros(x0.shape[0], dtype=torch.int32, device=x0.device)
    x, u, cost, status = _SolveFn.apply(x0, u_prev, obs_xy, solver, curv, nn_ctx, net_idx, u_init, ok)
    return x, u, cost, status, ok
