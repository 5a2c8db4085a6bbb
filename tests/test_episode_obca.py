"""Closed-loop episodes in the OBCA collision mode (collision_avoidance_type 'obca', mpc.py:42-43, :170-175, :211-221):
the obstacle heading forecast of the host and device glue, the rectangle outcome, and `evaluate --ca_type obca`.
CPU: geometry and host logic with the oracle as the solver.  GPU: outcome parity with the oracle, device glue = host
glue, gt_mpc + OBCA, the latency path, the C ABI's mode bits."""
import math
import os
from types import SimpleNamespace

import numpy as np
import pytest
import yaml

from igt_mpc_int_b200 import episode, evaluate, geometry as G
from oracle import nlp, c_oracle, obca
from tests.oracle_backend import OracleBackend


class ObcaOracleBackend(OracleBackend):
    """The oracle with the reference's OBCA settings: d_min = 0 (mpc.py:42-43) and the obstacle heading forecast
    forwarded to the dual-eliminated rectangle rows."""

    def __init__(self, N=40, mlp=None, **options):
        super().__init__(N=N, mlp=mlp, **options)
        self.P = nlp.Params(N=N, d_min=0.0)
        term = None if mlp is None else nlp.MLPTerm(**mlp)
        self.cold = c_oracle.COracle(self.P, term, **options)
        warm = dict(options); warm.update(mu0=1e-3, y_init_min=1e-2)
        self.warm = c_oracle.COracle(self.P, term, **warm)
        self.plain = c_oracle.COracle(self.P, **options)

    def solve_batch(self, x0, u_prev, curv, obs_xy, nn_ctx=None, u_init=None, obs_psi=None):
        co = self.warm if u_init is not None else self.cold
        r = co.solve(x0, u_prev, curv, obs_xy, nn_ctx=nn_ctx, u_init=u_init, obs_psi=obs_psi)
        return dict(x=r["Z"], u=r["U"], cost=r["cost"], viol=r["viol"], status=r["status"], iters=r["iters"])


def _value_net(hidden=(128, 128), seed=2026):
    import torch
    torch.manual_seed(seed)
    dims = [6] + list(hidden) + [1]
    layers = [torch.nn.Linear(dims[i], dims[i + 1], dtype=torch.double) for i in range(len(dims) - 1)]
    w = [(l.weight.detach().numpy().copy(), l.bias.detach().numpy().copy()) for l in layers]
    return dict(weights=w, Wn=np.eye(6), mu_f=np.zeros(6), sigma_t=1.0, mu_t=0.0)


def _min_rect_gap(z_cl):
    """smallest signed distance between the two rectangles over all episodes and recorded steps"""
    z = z_cl[..., [0, 1, 6]]
    return min(obca.rect_distance(z[e, 0, t], z[e, 1, t])[0] for e in range(z.shape[0]) for t in range(z.shape[2]))


# ---------------------------------------------------------------------------------------------------------- CPU
def test_route_heading_matches_frenet2global():
    """geometry.route_heading and the descriptor's heading (a Python restatement of csrc/episode.cuh route_heading:
    rd[10] = th0, sgn, b0, b1, r) give the heading of frenet2global on all 12 routes; rd[11] marks routes 32 and 41."""
    s = np.linspace(0.0, 74.0, 371)
    for r in G.ROUTES:
        rd = G.route_descriptor(r, exit_coord=G.EXIT_COORD.get(r))
        th0, sgn, b0, b1, rr = rd[10], rd[4], rd[5], rd[6], rd[7]
        vec = G.route_heading(s, r)
        for k, sk in enumerate(s):
            ref = G.frenet2global(sk, r)[2]
            if sgn == 0.0 or sk < b0:
                th = th0
            elif sk <= b1:
                th = th0 + sgn * ((sk - b0) / rr)
            else:
                th = th0 + sgn * (math.pi / 2)
            assert abs(th - ref) < 1e-12 and abs(vec[k] - ref) < 1e-12, (r, sk)
        assert rd[11] == (1.0 if r in ('32', '41') else 0.0), r


def test_rectangles_overlap_matches_rect_distance():
    """The separating-axis test agrees with the sign of the oracle's signed rectangle distance on random pose pairs."""
    rng = np.random.default_rng(7)
    n = 10000
    p = np.column_stack([rng.uniform(-4, 4, n), rng.uniform(-4, 4, n), rng.uniform(-math.pi, math.pi, n)])
    q = np.column_stack([rng.uniform(-4, 4, n), rng.uniform(-4, 4, n), rng.uniform(-math.pi, math.pi, n)])
    ov = G.rectangles_overlap(p, q)
    d = np.array([obca.rect_distance(p[i], q[i])[0] for i in range(n)])
    keep = np.abs(d) >= 1e-9
    assert keep.sum() > 0.99 * n and 0.2 < ov.mean() < 0.8
    assert np.array_equal(ov[keep], d[keep] < 0)


def test_closed_loop_obca_host_logic_with_oracle_backend():
    """Host driver in OBCA mode: the obs_psi handed to every solve follows the convention of episode.py (current
    heading at k = 0, route heading of the constant-acceleration forecast, previous-plan heading in V2V steps, abs() on
    routes 32 / 41, 0 for a filtered obstacle); the rectangles never overlap."""
    N, T = 10, 12
    calls = []

    class Spy(ObcaOracleBackend):
        def solve_batch(self, x0, u_prev, curv, obs_xy, nn_ctx=None, u_init=None, obs_psi=None):
            r = super().solve_batch(x0, u_prev, curv, obs_xy, nn_ctx=nn_ctx, u_init=u_init, obs_psi=obs_psi)
            calls.append((np.array(x0), np.array(curv), np.array(obs_xy), None if obs_psi is None else np.array(obs_psi), r))
            return r

    ref = episode.reference_episode_specs()
    specs = [ref[0], ref[4], ref[24]]                     # (13, 23), (31, 41), (12, 32): routes 41 and 32 are flipped
    assert {'41', '32'} <= {r for sp in specs for r in sp.routes}
    # a fourth episode whose vehicle 0 has passed the intersection: vehicle 1 is behind it (filter_preds)
    specs.append(episode.EpisodeSpec(routes=['13', '23'], s0=(40.0, 0.0)))
    res = episode.run_closed_loop(Spy(N=N, max_iter=60), specs, steps=T, N=N, ca_type="obca")
    E = len(specs)
    assert res.z_cl.shape == (E, 2, T + 1, 7)
    assert np.all(res.solved[:, :, 0])
    assert not res.collision.any() and _min_rect_gap(res.z_cl) > -1e-6
    route_of = [sp.routes[i] for sp in specs for i in range(2)]
    zc = res.z_cl.reshape(2 * E, T + 1, 7)
    uc = res.u_cl.reshape(2 * E, T, 2)
    ok = res.solved.reshape(2 * E, T)
    cv = [np.array(G.curvature_params(r)) for r in route_of]
    # map every solved row back to (step, vehicle) through its initial state and route curvature
    seen, plans = {}, {}
    for x0, curv, ob, psi, r in calls:
        assert psi is not None and psi.shape == (len(x0), N + 1)
        for j in range(len(x0)):
            hit = [(t, b) for b in range(2 * E) for t in range(T)
                   if np.array_equal(zc[b, t], x0[j]) and np.array_equal(cv[b], curv[j])]
            assert len(hit) == 1
            seen[hit[0]] = (ob[j], psi[j])
            plans[hit[0]] = r["x"][j]
    assert len(seen) == 2 * E * T
    n_cold = n_v2v = n_flip = n_filt = 0
    for (t, b), (ob, psi) in seen.items():
        o = b ^ 1
        fl = (lambda a: np.abs(a)) if route_of[o] in ('32', '41') else (lambda a: a)
        if ob[0, 0] == -20.0 and np.all(ob == -20.0):
            assert np.all(psi == 0.0)
            n_filt += 1
            continue
        assert psi[0] == fl(zc[o, t, 6])                                     # k = 0: the current heading
        if t > 0 and ok[o, t - 1]:                                           # V2V: the previous plan's headings
            assert np.array_equal(psi[:N], fl(plans[(t - 1, o)][1:, 6]))
            n_v2v += 1
        else:                                                                # constant-acceleration forecast
            a = uc[o, t - 1, 0] if t > 0 else 0.1
            s, v = zc[o, t, 2], zc[o, t, 5]
            sk = []
            for _ in range(N):
                s, v = s + v * 0.1 + 0.5 * a * 0.1 * 0.1, min(max(v + a * 0.1, -2.0), 20.0)
                sk.append(s)
            assert np.max(np.abs(psi[1:] - fl(G.route_heading(np.array(sk), route_of[o])))) < 1e-12
            n_cold += 1
        if route_of[o] in ('32', '41'):
            assert np.all(psi >= 0.0)
            n_flip += 1
    assert n_cold > 0 and n_v2v > 0 and n_flip > 0 and n_filt > 0


def _args(tmp, **kw):
    d = dict(save_dir=str(tmp), num_samples=1, eval_mode='mpc', sc=1, rotation=0, order=0, all_variants=False,
             nn_weights=None, steps=150)
    d.update(kw)
    return SimpleNamespace(**d)


def test_evaluate_ca_type_obca_writes_policy_config(tmp_path):
    a = evaluate.build_parser().parse_args(['--save_dir', str(tmp_path), '--eval_mode', 'mpc', '--sc', '4',
                                             '--ca_type', 'obca', '--steps', '12'])
    assert a.ca_type == 'obca'
    run_dir, summary = evaluate.main(a, solver=ObcaOracleBackend(N=40, max_iter=60))
    cfg = yaml.safe_load(open(os.path.join(run_dir, 'mpc', 'mpc.yaml')))
    assert cfg['collision_avoidance_type'] == 'obca'
    assert evaluate.POLICY_CONFIG['collision_avoidance_type'] == 'circle'          # the module default is untouched
    assert len(summary) == 1 and not summary[0]['collision']


# ---------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_obca_closed_loop_outcomes_match_oracle_all_scenarios():
    """All 64 reference episodes, 150 steps, N = 40, OBCA rows: same per-episode outcome with the GPU solver and the
    oracle, no overlap, and the trajectory / solve-statistics bars of the circle-mode test."""
    from igt_mpc_int_b200.planner import BatchSolver
    specs = episode.reference_episode_specs()
    gpu = BatchSolver(N=40, d_min=0.0)
    rg = episode.run_closed_loop(gpu, specs, steps=150, N=40, ca_type="obca")
    ro = episode.run_closed_loop(ObcaOracleBackend(N=40, max_iter=gpu.params.max_iter, max_trials=gpu.params.max_trials),
                                 specs, steps=150, N=40, ca_type="obca")
    gpu.close()
    assert np.array_equal(rg.deadlock, ro.deadlock)
    assert np.array_equal(rg.collision, ro.collision)
    assert np.array_equal(rg.goal, ro.goal)
    assert not rg.collision.any()
    assert _min_rect_gap(rg.z_cl) >= -1e-6
    dz = np.abs(rg.z_cl - ro.z_cl).reshape(len(specs), -1).max(axis=1)
    assert np.mean(dz < 1e-3) >= 0.85, dz
    assert abs(int(rg.num_infeasible.sum()) - int(ro.num_infeasible.sum())) <= 0.05 * ro.num_infeasible.sum()
    assert (rg.solved == ro.solved).mean() > 0.99


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["mpc", "gt_mpc"])
def test_obca_device_closed_loop_equals_host_driven_loop(mode):
    """igt_episode_run_host with IGT_EPISODE_OBCA against the host-driven loop, same GPU solver: the bars of the
    circle-mode test, and the first 20 steps the same numbers (the device heading forecast is the host's)."""
    from igt_mpc_int_b200.planner import BatchSolver
    specs = episode.reference_episode_specs()[::4] if mode == "mpc" else episode.reference_episode_specs()[::8]
    kw = dict(mlp=_value_net()) if mode == "gt_mpc" else {}
    gpu = BatchSolver(N=40, d_min=0.0, **kw)
    rh = episode.run_closed_loop(gpu, specs, steps=150, N=40, mode=mode, ca_type="obca")
    rd = episode.run_closed_loop_device(gpu, specs, steps=150, N=40, mode=mode, record_latency=True, ca_type="obca")
    gpu.close()
    assert np.array_equal(rd.collision, rh.collision) and not rd.collision.any()
    assert np.sum(rd.deadlock != rh.deadlock) <= 1 and np.sum(np.any(rd.goal != rh.goal, axis=1)) <= 1
    dz = np.abs(rd.z_cl - rh.z_cl).reshape(len(specs), -1).max(axis=1)
    assert np.mean(dz < 1e-6) >= 0.75, dz
    assert np.mean(rd.solved == rh.solved) > 0.99 and abs(rd.solved.mean() - rh.solved.mean()) < 0.01
    assert np.max(np.abs(rd.z_cl[:, :, :20] - rh.z_cl[:, :, :20])) < 1e-7
    assert len(rd.step_latency_ms) == 150 and min(rd.step_latency_ms) > 0


@pytest.mark.gpu
def test_gt_mpc_obca_matches_oracle():
    """gt_mpc + OBCA (per-thread value term, OBCA rows): at solve level on 1024 mid-episode problems with the bars of
    the 'mpc' OBCA parity test, and in closed loop (variant 0 of the 8 scenarios) with identical outcomes."""
    from igt_mpc_int_b200.planner import BatchSolver
    from igt_mpc_int_b200 import scenarios as S
    from tests.util import relerr
    N, B = 40, 1024
    net = _value_net()
    pb = S.mid_episode(B, N=N, seed=5)
    s = BatchSolver(N=N, d_min=0.0, mlp=net)
    r = s.solve_batch(pb.x0, pb.u_prev, pb.curv, pb.obs, nn_ctx=pb.nn_ctx, obs_psi=pb.obs_psi)
    P = nlp.Params(N=N, d_min=0.0)
    o = c_oracle.COracle(P, nlp.MLPTerm(**net), max_iter=s.params.max_iter).solve(pb.x0, pb.u_prev, pb.curv, pb.obs,
                                                                                 nn_ctx=pb.nn_ctx, obs_psi=pb.obs_psi)
    assert np.mean(r["status"] == o["status"]) > 0.99
    ok = (o["status"] == 0) & (r["status"] == 0)
    assert ok.sum() > 0.85 * B
    assert np.max(relerr(r["cost"][ok], o["cost"][ok])) < 1e-4
    assert np.max(np.abs(r["u"][ok] - o["U"][ok])) < 1e-3
    assert np.max(r["viol"][ok]) <= 1e-6
    specs = episode.reference_episode_specs()[::8]
    rg = episode.run_closed_loop(s, specs, steps=150, N=40, mode="gt_mpc", ca_type="obca")
    s.close()
    ro = episode.run_closed_loop(ObcaOracleBackend(N=40, mlp=net, max_iter=60), specs, steps=150, N=40, mode="gt_mpc",
                                 ca_type="obca")
    assert not rg.collision.any()
    assert np.array_equal(rg.collision, ro.collision)
    assert np.array_equal(rg.deadlock, ro.deadlock)
    assert np.array_equal(rg.goal, ro.goal)


@pytest.mark.gpu
def test_obca_latency_path_is_bit_identical_to_throughput_kernel():
    """OBCA 'mpc' batches of at most one problem per SM (closed-loop episodes with E <= n_sm / 2) run on the latency
    path: identical bits to the throughput kernel, cold and warm-started."""
    import torch
    from igt_mpc_int_b200.planner import BatchSolver
    from igt_mpc_int_b200 import scenarios as S
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    N = 40
    pb = S.mid_episode(n_sm // 8 * 8 + 8, N=N, seed=23)
    s = BatchSolver(N=N, d_min=0.0)
    for B in (1, 2, 33, n_sm):
        a = (pb.x0[:B], pb.u_prev[:B], pb.curv[:B], pb.obs[:B])
        out = {}
        for flag in (0, 1):
            s.set_option("latency_path", flag)
            cold = s.solve_batch(*a, obs_psi=pb.obs_psi[:B])
            warm = s.solve_batch(*a, u_init=np.nan_to_num(cold["u"]), obs_psi=pb.obs_psi[:B])
            out[flag] = (cold, warm)
        for i in (0, 1):
            for k in ("status", "iters", "cost", "viol", "u", "x"):
                assert np.array_equal(out[0][i][k], out[1][i][k], equal_nan=True), (B, i, k)
    s.close()


@pytest.mark.gpu
def test_episode_mode_bits_and_evaluate_obca_device_loop(tmp_path):
    """igt_episode_run_host refuses unknown mode bits; the device driver refuses OBCA with the circle gap; and
    `evaluate --ca_type obca --device_loop --all_variants` writes the reference's files with the oracle's outcomes."""
    import ctypes as C
    import pickle
    from igt_mpc_int_b200.planner import BatchSolver
    s = BatchSolver(N=40)
    sp = episode.reference_episode_specs()[0]
    rd = np.array([G.route_descriptor(r, exit_coord=G.EXIT_COORD.get(r)) for r in sp.routes])
    cv = np.array([G.curvature_params(r) for r in sp.routes])
    z0 = np.zeros((2, 7)); up = np.zeros((2, 2)); enc = np.zeros(2)
    z_cl = np.zeros((1, 2, 2, 7)); u_cl = np.zeros((1, 2, 1, 2)); solved = np.zeros((1, 2, 1), dtype=np.int32)
    vp = lambda a: C.c_void_p(a.ctypes.data)
    rc = s.lib.igt_episode_run_host(s._h, 1, 1, 4, vp(rd), vp(cv), vp(z0), vp(up), vp(enc), vp(z_cl), vp(u_cl), vp(solved), None)
    assert rc == -1 and b"mode" in s.lib.igt_last_error(s._h)
    with pytest.raises(ValueError):
        episode.run_closed_loop_device(s, [sp], steps=2, N=40, ca_type="obca")
    s.close()
    a = _args(tmp_path / "gpu", all_variants=True, ca_type='obca', device_loop=True)
    run_dir, summary = evaluate.main(a)
    sub = os.path.join(run_dir, 'mpc')
    for f in ('cl_traj.pkl', 'u_cl.pkl', 'evaluation_data.pkl', 'eval_stats.csv', 'mpc.yaml'):
        assert os.path.isfile(os.path.join(sub, f)), f
    cl = pickle.load(open(os.path.join(sub, 'cl_traj.pkl'), 'rb'))
    assert cl.shape == (8, 14, 151)
    assert yaml.safe_load(open(os.path.join(sub, 'mpc.yaml')))['collision_avoidance_type'] == 'obca'
    ref_dir, ref_summary = evaluate.main(_args(tmp_path / "cpu", all_variants=True, ca_type='obca'),
                                         solver=ObcaOracleBackend(N=40, max_iter=60))
    for g, o in zip(summary, ref_summary):
        assert g['routes'] == o['routes'] and g['deadlock'] == o['deadlock'] and g['collision'] == o['collision'] and g['goal'] == o['goal']
    assert not any(g['collision'] for g in summary)
