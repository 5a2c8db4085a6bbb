"""Gradients through the batched solve on the GPU: the dual-exporting solve against the plain one, the VJP kernel
against the oracle VJP (oracle/sensitivity.py) and the CPU run of the same code (tests/hostsim), torch autograd through
igt_mpc_int_b200.autodiff, and the calls that must be refused."""
import numpy as np
import pytest

from igt_mpc_int_b200 import _lib, scenarios as S, terminal_set as TS
from oracle import nlp, sensitivity as SE
from tests.hostsim import sens_harness as H
from tests.test_value_nets import shipped_net

N = 40


def _solver(**kw):
    from igt_mpc_int_b200.planner import BatchSolver
    return BatchSolver(N=N, **kw)


def _nets():
    return [shipped_net(k)[0] for k in range(1, 9)]


def _rp_check(s, pb, r, ctx=None, net_idx=None):
    """|c(u) + y|_inf <= tol_rp for converged problems, s, y > 0"""
    ok = r["status"] == 0
    assert np.all(r["slack"][ok] > 0) and np.all(r["mult"][ok] > 0)
    P = nlp.Params(N=N, cinf_A=TS.cinf()[0], cinf_b=TS.cinf()[1])
    from oracle import solver as SV
    for b in np.where(ok)[0][:64]:
        prob = nlp.Problem(x0=pb.x0[b], u_prev=pb.u_prev[b], curv=tuple(pb.curv[b]), obs=pb.obs[b])
        c = np.concatenate(SV.all_rows_values(P, prob, r["x"][b], r["u"][b]))
        assert np.abs(c + r["slack"][b]).max() <= s.params.tol_rp * 1.0001


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["mpc", "gt", "bank"])
@pytest.mark.parametrize("B", [2, "big"])
def test_dual_solve_is_the_plain_solve(case, B):
    nets = _nets()
    s = _solver(mlp=nets if case == "bank" else (nets[0] if case == "gt" else None))
    if B == "big":                                              # more problems than the resident lanes (one CTA of 256 per SM)
        import torch
        B = torch.cuda.get_device_properties(0).multi_processor_count * 256 + 40
    pb = S.mid_episode(8 * ((B + 7) // 8), N=N, seed=41).slice(0, B)
    ctx = pb.nn_ctx if case != "mpc" else None
    net = (np.arange(B) % 8).astype(np.int32) if case == "bank" else None
    a = s.solve_batch(pb.x0, pb.u_prev, pb.curv, pb.obs, nn_ctx=ctx, net_idx=net)
    d = s.solve_batch(pb.x0, pb.u_prev, pb.curv, pb.obs, nn_ctx=ctx, net_idx=net, duals=True)
    for k in ("x", "u", "cost", "viol", "status", "iters"):
        assert np.array_equal(a[k], d[k], equal_nan=True), k
    assert d["slack"].shape == (B, s.n_rows)
    _rp_check(s, pb, d)


def _vjp_case(case, B, seed, **options):
    nets = _nets()
    s = _solver(mlp=nets if case == "bank" else None, **options)
    pb = S.mid_episode(B, N=N, seed=seed)
    ctx = pb.nn_ctx if case == "bank" else None
    net = (np.arange(B) % 8).astype(np.int32) if case == "bank" else None
    r = s.solve_batch(pb.x0, pb.u_prev, pb.curv, pb.obs, nn_ctx=ctx, net_idx=net, duals=True)
    rng = np.random.default_rng(seed)
    gx, gu, gc = rng.standard_normal((B, N + 1, 7)), rng.standard_normal((B, N, 2)), rng.standard_normal(B)
    g = s.vjp(pb.x0, pb.u_prev, pb.curv, pb.obs, r["u"], r["slack"], r["mult"], r["status"], gx, gu, gc, nn_ctx=ctx, net_idx=net)
    return s, pb, ctx, net, r, (gx, gu, gc), g, nets


@pytest.mark.gpu
@pytest.mark.parametrize("case,B", [("mpc", 1024), ("bank", 256)])
def test_gpu_vjp_matches_oracle_and_hostsim(case, B):
    """the GPU VJP against the dense oracle fed the GPU's (u, y, s) and against the CPU run of the same code, both to
    1e-8 relative, ok exactly.  The solves end at mu_floor = 1e-4: at the default 1e-8, s / y reaches 1e12 on active
    rows and rounding differences (another factorisation, or the device's fused multiply-adds) grow by that
    conditioning, to ~1e-5 relative on a few obstacle gradients (DESIGN.md section 10)"""
    floor = dict(mu_floor=1e-4, tol_comp=1.5e-4)
    s, pb, ctx, net, r, (gx, gu, gc), g, nets = _vjp_case(case, B, 51 if case == "mpc" else 52, **floor)
    cinf = TS.cinf()
    P = nlp.Params(N=N, cinf_A=cinf[0], cinf_b=cinf[1])
    p = H.default_params(1); p.set_cinf(*cinf)
    for k, v in floor.items():
        setattr(p, k, v)
    assert (g["ok"] == 1).sum() >= 0.8 * B
    worst = 0.0
    idx = np.arange(B) if case == "bank" else np.arange(0, B, 8)
    for b in idx:
        mlp = nlp.MLPTerm(**nets[net[b]]) if case == "bank" else None
        prob = nlp.Problem(x0=pb.x0[b], u_prev=pb.u_prev[b], curv=tuple(pb.curv[b]), obs=pb.obs[b],
                           nn_ctx=tuple(ctx[b]) if ctx is not None else None)
        o = SE.vjp(P, prob, mlp, r["u"][b], r["slack"][b], r["mult"][b], r["status"][b], gx[b], gu[b], gc[b])
        assert g["ok"][b] == o[3], b
        hs = H.vjp(p, pb.x0[b:b + 1], pb.u_prev[b:b + 1], pb.curv[b:b + 1], pb.obs[b:b + 1], r["u"][b:b + 1],
                   r["slack"][b:b + 1], r["mult"][b:b + 1], r["status"][b:b + 1], gx[b:b + 1], gu[b:b + 1], gc[b:b + 1],
                   nn_ctx=None if ctx is None else ctx[b:b + 1], mlp=mlp)
        for i, k in enumerate(("gx0", "gu_prev", "gobs")):
            if o[3]:
                rel = np.abs(g[k][b] - o[i]).max() / max(np.abs(o[i]).max(), 1e-300)
                worst = max(worst, rel)
                assert rel <= 1e-8, (b, k, rel)
                assert np.abs(g[k][b] - hs[i][0]).max() <= 1e-8 * max(np.abs(hs[i][0]).max(), 1e-300), (b, k)
            else:
                assert np.all(g[k][b] == 0.0)
    print("%s: worst relative difference to the oracle VJP %.2e" % (case, worst))


@pytest.mark.gpu
def test_vjp_dev_and_host_give_the_same_bits_and_autograd():
    import torch
    from igt_mpc_int_b200 import autodiff
    s, pb, ctx, net, r, (gx, gu, gc), g, nets = _vjp_case("mpc", 512, 61)
    T = lambda a, dt=torch.float64: torch.tensor(np.ascontiguousarray(a), dtype=dt, device="cuda")
    d = s.vjp_device(T(pb.x0), T(pb.u_prev), T(pb.curv), T(pb.obs), T(r["u"]), T(r["slack"]), T(r["mult"]),
                     T(r["status"], torch.int32), T(gx), T(gu), T(gc))
    for k in ("gx0", "gu_prev", "gobs", "ok"):
        assert np.array_equal(d[k].cpu().numpy(), g[k]), k
    # autograd: grad of a scalar loss equals the direct VJP; problems with ok = 0 get exact zeros
    x0, up, ob = T(pb.x0).requires_grad_(), T(pb.u_prev).requires_grad_(), T(pb.obs).requires_grad_()
    x, u, cost, status, ok = autodiff.solve(s, x0, up, T(pb.curv), ob)
    loss = (x * T(gx)).sum() + (u * T(gu)).sum() + (cost * T(gc)).sum()
    g0, g1, g2 = torch.autograd.grad(loss, (x0, up, ob))
    assert np.array_equal(g0.cpu().numpy(), g["gx0"]) and np.array_equal(g1.cpu().numpy(), g["gu_prev"])
    assert np.array_equal(g2.cpu().numpy(), g["gobs"]) and np.array_equal(ok.cpu().numpy(), g["ok"])
    bad = g["ok"] == 0
    assert bad.sum() > 0 and np.all(g0.cpu().numpy()[bad] == 0) and np.all(g2.cpu().numpy()[bad] == 0)


@pytest.mark.gpu
def test_refused_calls_return_einval():
    pb = S.mid_episode(8, N=N, seed=71)
    nets = _nets()
    for kw, solve_kw, opt in ((dict(), dict(obs_psi=pb.obs_psi), None), (dict(precision="f32"), dict(), None),
                              (dict(mlp=nets[0]), dict(nn_ctx=pb.nn_ctx), "tensor_core_mlp")):
        s = _solver(**kw)
        if opt:
            s.set_option(opt, 1)
        with pytest.raises(_lib.IgtError) as e:
            s.solve_batch(pb.x0, pb.u_prev, pb.curv, pb.obs, duals=True, **solve_kw)
        assert "(-1)" in str(e.value) and "igt_solve_duals" in str(e.value)
    s = _solver(precision="f32")
    M = s.n_rows
    with pytest.raises(_lib.IgtError) as e:
        s.vjp(pb.x0, pb.u_prev, pb.curv, pb.obs, np.zeros((8, N, 2)), np.ones((8, M)), np.ones((8, M)), np.zeros(8))
    assert "(-1)" in str(e.value) and "precision f64" in str(e.value)
