"""Batches larger than the machine's resident solver lanes, and the evaluation kernel against the plain NLP.

The throughput kernels run one CTA of 256 persistent lanes per SM; a lane takes problems from a global counter until
none are left.  A batch of at most that many problems gives every lane one problem at most, so only a larger batch
makes a lane solve a second problem with the same Solver object and workspace slot, next to CTA neighbours that are
in the middle of their own solves.  Each solver instantiation is run here at about twice the lanes and must give, bit
for bit, what the same problems give in slices of at most one problem per lane (the regime the oracle-parity tests
cover) and in reversed order.

The second part checks `evaluate` (eval_kernel) against oracle/nlp.py and a numpy fp64 rollout at controls that make
each row family the largest row on some problems, and at non-finite controls."""
import numpy as np
import pytest

from tests.util import relerr

pytestmark = pytest.mark.gpu

N = 40


def _lanes():
    import torch
    # 256 = SOLVE_BLOCK (csrc/igt_abi.cu): one CTA of 256 persistent lanes per SM
    return torch.cuda.get_device_properties(0).multi_processor_count * 256


@pytest.fixture(scope="module")
def big():
    """B_big = the smallest multiple of 8 >= 2 lanes + 37 mid_episode problems, with infeasible initial states and
    non-finite states at seeded positions spread over the batch"""
    from igt_mpc_int_b200 import scenarios as S
    lanes = _lanes()
    B = -(-(2 * lanes + 37) // 8) * 8
    pb = S.mid_episode(B, N=N, seed=1234)
    x0 = pb.x0.copy()
    pos = np.sort(np.random.default_rng(4321).choice(B, 48, replace=False))
    infeas, nonfin = pos[:40], pos[40:]
    for i, q in enumerate(infeas):                     # v above / below its limits, |ey| above its limit
        col, val = ((5, 5.5), (5, -0.4), (3, 0.3), (3, -0.35))[i % 4]
        x0[q, col] = val
    for i, q in enumerate(nonfin):                     # NaN v: rejected by init; x, s, psi: accepted, the solve fails
        col, val = ((5, np.nan), (0, np.nan), (2, np.inf), (6, -np.inf))[i % 4]
        x0[q, col] = val
    return dict(lanes=lanes, B=B, x0=x0, u_prev=pb.u_prev, curv=pb.curv, obs=pb.obs, obs_psi=pb.obs_psi,
                nn_ctx=pb.nn_ctx, net_idx=(pb.scenario - 1).astype(np.int32), infeas=infeas, nonfin=nonfin,
                good=np.setdiff1d(np.arange(B), pos))


def _net128():
    from tests.test_gpu_mlp import _net, _term, _as_dict
    return _as_dict(_term(_net((128, 128)), False))


def _shipped(k):
    from tests.test_value_nets import shipped_net
    return shipped_net(k)[0]


# case: solver keywords, value term ('coop' / 'tc' / 'bank' / None), OBCA rows
CASES = {
    "f64": (dict(), None, False),                                   # solve_kernel<double, false, false>
    "f32": (dict(precision="f32"), None, False),                    # solve_kernel<float, false, false>
    "obca": (dict(d_min=0.0), None, True),                          # solve_kernel<double, false, true>
    "gt_coop": (dict(), "coop", False),                             # solve_kernel<double, false, false, true> (COOP)
    "gt_tc": (dict(), "tc", False),                                 # solve_kernel<double, true, false> (TC)
    "gt_obca": (dict(d_min=0.0), "coop", True),                     # solve_kernel<double, false, true>, per-thread value term
    "bank": (dict(), "bank", False),                                # BANK + COOP
    "bank_obca": (dict(d_min=0.0), "bank", True),                   # BANK, per-thread value term
    "bank_f32": (dict(precision="f32"), "bank", False),             # BANK f32
}


def _make(case):
    from igt_mpc_int_b200.planner import BatchSolver
    kw, vt, _ = CASES[case]
    if vt == "bank":
        return BatchSolver(N=N, mlp=[_shipped(k) for k in range(1, 9)], **kw)
    s = BatchSolver(N=N, mlp=_net128() if vt else None, **kw)
    if vt:
        s.set_option("tensor_core_mlp", 1 if vt == "tc" else 0)
    return s


def _args(case, b, idx):
    _, vt, obca = CASES[case]
    sel = slice(None) if idx is None else idx
    kw = dict(obs_psi=b["obs_psi"][sel] if obca else None)
    if vt:
        kw["nn_ctx"] = b["nn_ctx"][sel]
    if vt == "bank":
        kw["net_idx"] = b["net_idx"][sel]
    return (b["x0"][sel], b["u_prev"][sel], b["curv"][sel], b["obs"][sel]), kw


def _solve(s, case, b, idx=None, u_init=None):
    a, kw = _args(case, b, idx)
    return s.solve_batch(*a, u_init=u_init, **kw)


def _same(o, r, idx):
    for k in ("status", "iters", "cost", "u", "x"):
        assert np.array_equal(o[k], r[k][idx], equal_nan=True), k


def _slices(B, lanes):
    return [np.arange(lo, min(lo + lanes, B)) for lo in range(0, B, lanes)]


@pytest.mark.parametrize("case", list(CASES))
def test_beyond_lanes_equals_slices_reversed_and_evaluation(big, case, oracle_params):
    b = big
    B, lanes = b["B"], b["lanes"]
    assert B > lanes                        # n_slots = lanes here, so some lanes solve several problems
    s = _make(case)
    r = _solve(s, case, b)
    st = r["status"]
    print("%s B=%d statuses %s" % (case, B, dict(zip(*[v.tolist() for v in np.unique(st, return_counts=True)]))))
    for idx in _slices(B, lanes):
        _same(_solve(s, case, b, idx), r, idx)
    rev = np.arange(B)[::-1].copy()
    _same(_solve(s, case, b, rev), r, rev)
    assert np.all(st[b["infeas"]] == 2) and np.all(st[b["nonfin"]] != 0)
    assert np.all(np.isnan(r["cost"][b["infeas"]]))
    ok = st == 0
    f32 = CASES[case][0].get("precision") == "f32"
    assert ok[b["good"]].mean() > (0.5 if f32 else 0.6 if CASES[case][1] else 0.85)
    # the evaluation kernel reproduces the solver's cost; fp32 solves and the tensor-core value term (fp32-accurate,
    # not the parity path) are held to their own precision
    loose = f32 or CASES[case][1] == "tc"
    assert np.max(r["viol"][ok]) <= (1e-3 if f32 else 1e-6)
    idx = np.where(ok)[0][::16]
    (x0, up, cv, ob), kw = _args(case, b, idx)
    ev = s.evaluate(x0, up, cv, ob, r["u"][idx], **kw)
    assert np.max(relerr(ev["cost"], r["cost"][idx])) < (1e-4 if loose else 1e-9)
    assert np.max(ev["viol"]) <= (1e-3 if f32 else 1e-6)
    if case == "f64":
        # one lane takes a second problem while the rest of the machine is idle
        e = np.arange(lanes + 1)
        _same(_solve(s, case, b, e), r, e)
        # warm start from the cold solution, against warm slices
        u0 = np.nan_to_num(r["u"])
        w = _solve(s, case, b, u_init=u0)
        for idx in _slices(B, lanes):
            _same(_solve(s, case, b, idx, u_init=u0[idx]), w, idx)
        assert np.mean(w["status"][ok] == 0) > 0.99
    s.close()
    if case in ("f64", "bank"):
        _oracle_sample(r, b, case, oracle_params)


def _oracle_sample(r, b, case, oracle_params):
    """512 problems spread over the batch against the C oracle (each with its own network for the bank): the
    north-star tolerances of test_gpu_solve._vs_oracle"""
    from oracle import c_oracle, nlp
    good = b["good"]
    smp = good[np.linspace(0, len(good) - 1, 512).astype(int)]
    o_st = np.empty(512, dtype=np.int64); o_cost = np.empty(512); o_U = np.empty((512, N, 2))
    groups = [(np.arange(512), None)] if case == "f64" else \
        [(np.where(b["net_idx"][smp] == k)[0], nlp.MLPTerm(**_shipped(k + 1))) for k in range(8)]
    for m, term in groups:
        q = smp[m]
        o = c_oracle.COracle(oracle_params[N], term, max_iter=60).solve(
            b["x0"][q], b["u_prev"][q], b["curv"][q], b["obs"][q], nn_ctx=None if term is None else b["nn_ctx"][q])
        o_st[m], o_cost[m], o_U[m] = o["status"], o["cost"], o["U"]
    st = r["status"][smp]
    both = (o_st == 0) & (st == 0)
    assert np.mean((o_st == 0) == (st == 0)) >= 0.99
    assert both.mean() >= (0.9 if case == "f64" else 0.6)
    assert np.max(relerr(r["cost"][smp][both], o_cost[both])) < 1e-4
    assert np.max(np.abs(r["u"][smp][both] - o_U[both])) < 1e-3
    assert np.max(r["viol"][smp][both]) <= 1e-6


def test_bank_device_entry_bad_indices_beyond_lanes(big):
    """solve_batch_device checks the index in the kernel: a problem whose index is outside the bank or names an empty
    slot gets STATUS_BAD_NET and NaN outputs, and its lane fetches again; every other problem equals the host path"""
    import torch
    from igt_mpc_int_b200 import _lib
    from igt_mpc_int_b200.planner import BatchSolver
    b = big
    B, lanes = b["B"], b["lanes"]
    assert B > lanes
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    bad = np.sort(np.random.default_rng(11).choice(b["good"], 24, replace=False))
    rest = np.setdiff1d(np.arange(B), bad)
    for nets, good_idx, bad_vals in (([_shipped(k) for k in range(1, 9)], b["net_idx"], (-1, 8)),
                                     ([_shipped(k) for k in range(1, 8)] + [None], b["net_idx"] % 7, (7,))):
        s = BatchSolver(N=N, mlp=nets)
        ni = good_idx.astype(np.int32).copy()
        ni[bad] = np.resize(np.array(bad_vals, dtype=np.int32), len(bad))
        out = s.solve_batch_device(d(b["x0"]), d(b["u_prev"]), d(b["curv"]), d(b["obs"]), nn_ctx=d(b["nn_ctx"]), net_idx=d(ni))
        torch.cuda.synchronize()
        o = {k: v.cpu().numpy() for k, v in out.items()}
        assert np.all(o["status"][bad] == _lib.STATUS_BAD_NET) and np.all(o["iters"][bad] == 0)
        assert np.all(np.isnan(o["x"][bad])) and np.all(np.isnan(o["u"][bad])) and np.all(np.isnan(o["cost"][bad]))
        ref = s.solve_batch(b["x0"][rest], b["u_prev"][rest], b["curv"][rest], b["obs"][rest], nn_ctx=b["nn_ctx"][rest],
                            net_idx=ni[rest])
        s.close()
        for k in ("status", "iters", "cost", "u", "x"):
            assert np.array_equal(o[k][rest], ref[k], equal_nan=True), k


@pytest.mark.parametrize("mode", ["mpc", "gt_mpc"])
def test_closed_loop_beyond_lanes_equals_two_loops(mode):
    """lanes / 2 + 64 episodes (2 vehicles each: more solves per step than lanes, with the per-problem warm / cold
    mask) for 8 steps, against the same episodes run as two loops of at most lanes / 2 episodes"""
    from igt_mpc_int_b200 import episode
    from igt_mpc_int_b200.planner import BatchSolver
    lanes = _lanes()
    E = lanes // 2 + 64
    specs = []
    d = 0
    while len(specs) < E:
        specs += episode.reference_episode_specs(sample=d)
        d += 1
    specs = specs[:E]
    assert 2 * E > lanes
    if mode == "gt_mpc":
        s = BatchSolver(N=N, mlp=[_shipped(k) for k in range(1, 9)])
        net_idx = np.array([sp.scenario - 1 for sp in specs], dtype=np.int32)
    else:
        s = BatchSolver(N=N)
        net_idx = None
    run = lambda lo, hi: episode.run_closed_loop_device(s, specs[lo:hi], steps=8, N=N, mode=mode,
                                                        net_idx=None if net_idx is None else net_idx[lo:hi])
    full = run(0, E)
    h = lanes // 2
    parts = [run(0, h), run(h, E)]
    s.close()
    for key in ("z_cl", "u_cl", "solved"):
        assert np.array_equal(getattr(full, key), np.concatenate([getattr(p, key) for p in parts]), equal_nan=True), key
    assert full.solved.mean() > 0.9


# ------------------------------------------------------------------------------------ evaluation kernel vs the NLP
KINDS = ("feasible", "far", "a_hi", "a_lo", "df_hi", "df_lo", "rate0_a", "rate0_df", "rate_a", "rate_df", "v_hi", "v_lo",
         "ey", "cinf", "collision")
FAMILIES = ("v", "v", "a", "a", "df", "df", "rate_a", "rate_a", "rate_df", "rate_df", "ey", "ey", "cinf", "collision")


def _row_labels(P):
    """family name and node index of every entry of oracle.nlp.inequality_rows"""
    sizes = [P.N] * 10 + [P.N + 1, P.N + 1, len(P.cinf_b), P.N]
    lab = np.concatenate([[f] * n for f, n in zip(FAMILIES, sizes)])
    node = np.concatenate([np.arange(n) if f != "collision" else np.arange(1, n + 1) for f, n in zip(FAMILIES, sizes)])
    return lab, node


def _nlp_params(s):
    """oracle.nlp.Params with the handle's limits and terminal-set table"""
    from oracle import nlp
    p = s.params
    return nlp.Params(N=N, d_min=p.d_min, jerk_limit=round(p.da_max / p.dt, 12), steer_rate=round(p.ddf_max / p.dt, 12),
                      cinf_A=np.array([[p.cinf_A[m][0], p.cinf_A[m][1]] for m in range(p.n_cinf)]),
                      cinf_b=np.array([p.cinf_b[m] for m in range(p.n_cinf)]))


def _controls(pb, P, obca, seed):
    """per problem (x0, u_prev, obs, U): the tracking controller's plan, perturbed so that one row family is violated
    (kinds cycle through KINDS; the loose-rate handle lets the bound rows of a and df dominate their rate rows)"""
    from oracle import nlp, dynamics as D
    rng = np.random.default_rng(seed)
    x0s, ups, obss, Us = [], [], [], []
    for i in range(len(pb)):
        kind = KINDS[i % len(KINDS)]
        x0, up, obs = pb.x0[i].copy(), pb.u_prev[i].copy(), pb.obs[i].copy()
        if kind == "v_hi":
            x0[D.IV] = 5.0 + rng.uniform(0.05, 0.3)
        elif kind == "v_lo":
            x0[D.IV] = -rng.uniform(0.05, 0.3)
        elif kind == "ey":
            x0[D.IEY] = rng.choice([-1, 1]) * rng.uniform(0.3, 0.5)
        elif kind == "cinf":
            x0[D.IV] = 4.9
        prob = nlp.Problem(x0=x0, u_prev=up, curv=tuple(pb.curv[i]), obs=obs)
        U, Z = nlp.tracking_rollout(P, prob, 5.0 if kind == "cinf" else float(np.clip(x0[D.IV], 0.5, 4.5)))
        k, dv = int(rng.integers(2, N - 2)), rng.uniform(0.05, 0.4)
        if kind == "a_hi":
            U[N - 2, 0] = P.a_max + dv
        elif kind == "a_lo":
            U[N - 2, 0] = P.a_min - dv
        elif kind == "df_hi":
            U[N - 2, 1] = P.df_max + dv
        elif kind == "df_lo":
            U[N - 2, 1] = -P.df_max - dv
        elif kind == "rate0_a":
            up[0] = U[0, 0] + rng.choice([-1, 1]) * (P.da_max + dv)
        elif kind == "rate0_df":
            up[1] = U[0, 1] + rng.choice([-1, 1]) * (P.ddf_max + dv)
        elif kind == "rate_a":
            U[k, 0] += rng.choice([-1, 1]) * (P.da_max + dv)
        elif kind == "rate_df":
            U[k, 1] += rng.choice([-1, 1]) * (P.ddf_max + dv)
        elif kind == "cinf":                                   # accelerate into the end of the horizon at 4.9 m/s
            for j in range(6):
                U[N - 6 + j, 0] = U[N - 7, 0] + 0.085 * (j + 1)
        elif kind == "collision":                              # an obstacle forecast on the rolled-out path
            Z = D.frenet_rollout(x0, U, prob.curv)
            obs[k] = Z[k, :2] + (rng.uniform(-1, 1, 2) if not obca else rng.uniform(-0.5, 0.5, 2))
        elif kind == "far":
            obs[1:] = Z[1:, :2] + 60.0
        x0s.append(x0); ups.append(up); obss.append(obs); Us.append(U)
    return np.array(x0s), np.array(ups), np.array(obss), np.array(Us)


def _reference(P, x0, up, curv, obs, U, obs_psi=None, ctx=None, terms=None):
    """numpy fp64 rollout, cost and rows of oracle/nlp.py, per problem"""
    from oracle import nlp, dynamics as D
    Zs, cost, rows = [], [], []
    for i in range(len(x0)):
        prob = nlp.Problem(x0=x0[i], u_prev=up[i], curv=tuple(curv[i]), obs=obs[i],
                           nn_ctx=None if ctx is None else tuple(ctx[i]), obs_psi=None if obs_psi is None else obs_psi[i])
        Z = D.frenet_rollout(x0[i], U[i], prob.curv)
        Zs.append(Z)
        cost.append(nlp.cost(P, prob, Z, U[i], None if terms is None else terms[i]))
        rows.append(nlp.inequality_rows(P, prob, Z, U[i]))
    return np.array(Zs), np.array(cost), np.array(rows)


@pytest.mark.parametrize("mode", ["circle", "loose_rates", "obca", "gt_mpc", "bank"])
def test_evaluation_kernel_matches_plain_nlp(mode):
    from igt_mpc_int_b200 import scenarios as S
    from igt_mpc_int_b200.planner import BatchSolver
    from oracle import nlp
    pb = S.mid_episode(240, N=N, seed=71)
    kw = dict(d_min=0.0) if mode == "obca" else dict(jerk_limit=100.0, steering_rate_limit=100.0) if mode == "loose_rates" else {}
    if mode == "bank":
        s = BatchSolver(N=N, mlp=[_shipped(k) for k in range(1, 9)])
    elif mode == "gt_mpc":
        s = BatchSolver(N=N, mlp=_shipped(3))
    else:
        s = BatchSolver(N=N, **kw)
    P = _nlp_params(s)
    obca = mode == "obca"
    x0, up, obs, U = _controls(pb, P, obca, seed=5)
    obs_psi = pb.obs_psi if obca else None
    ctx = pb.nn_ctx if mode in ("gt_mpc", "bank") else None
    net_idx = (pb.scenario - 1).astype(np.int32) if mode == "bank" else None
    terms = None
    if mode == "gt_mpc":
        terms = [nlp.MLPTerm(**_shipped(3))] * len(pb)
    elif mode == "bank":
        bank = [nlp.MLPTerm(**_shipped(k)) for k in range(1, 9)]
        terms = [bank[k] for k in net_idx]
    Z, cost, rows = _reference(P, x0, up, pb.curv, obs, U, obs_psi, ctx, terms)
    ev = s.evaluate(x0, up, pb.curv, obs, U, nn_ctx=ctx, obs_psi=obs_psi, net_idx=net_idx)
    assert np.max(relerr(ev["x"], Z)) < 1e-10
    assert np.max(relerr(ev["cost"], cost)) < 1e-11
    assert np.max(np.abs(ev["viol"] - np.maximum(0.0, rows.max(axis=1)))) < 1e-10
    # every family the controls aim at is the largest row (by 1e-3) on some problems, and some controls are feasible
    lab, node = _row_labels(P)
    if obca:
        lab = np.where(lab == "collision", "obca", lab)
    top = rows.argmax(axis=1)
    won = set()
    for i, j in enumerate(top):
        if rows[i, j] > 0 and rows[i, j] - rows[i, lab != lab[j]].max() > 1e-3:
            won.add(lab[j])
            if lab[j] in ("rate_a", "rate_df") and node[j] == 0:
                won.add(lab[j] + "@0")
    assert (rows.max(axis=1) <= 0).sum() >= 3
    want = {"a", "df"} if mode == "loose_rates" else {"v", "ey", "cinf", "rate_a", "rate_df", "rate_a@0", "rate_df@0"}
    want.add("obca" if obca else "collision")
    assert want <= won, want - won
    # row 0 of the obstacle forecast is not a row: NaN there changes nothing
    obs_nan = obs.copy(); obs_nan[:, 0] = np.nan
    ev0 = s.evaluate(x0, up, pb.curv, obs_nan, U, nn_ctx=ctx, obs_psi=obs_psi, net_idx=net_idx)
    for k in ("x", "cost", "viol"):
        assert np.array_equal(ev0[k], ev[k]), k
    s.close()


@pytest.mark.parametrize("mode", ["circle", "obca", "gt_mpc"])
def test_evaluation_kernel_non_finite_controls_are_not_feasible(mode):
    """A control sequence with a NaN, or one that drives the state non-finite, gives a non-finite cost and a violation
    that is not <= 1e-6 (the rows before the NaN are feasible: NaN rows must not be dropped from the maximum)"""
    from igt_mpc_int_b200 import scenarios as S
    from igt_mpc_int_b200.planner import BatchSolver
    from oracle import nlp
    pb = S.mid_episode(16, N=N, seed=71)
    s = BatchSolver(N=N, mlp=_shipped(1) if mode == "gt_mpc" else None, **(dict(d_min=0.0) if mode == "obca" else {}))
    P = _nlp_params(s)
    obs = pb.obs.copy()
    U = np.empty((16, N, 2))
    for i in range(16):
        prob = nlp.Problem(x0=pb.x0[i], u_prev=pb.u_prev[i], curv=tuple(pb.curv[i]), obs=obs[i])
        U[i], Z = nlp.tracking_rollout(P, prob, float(np.clip(pb.x0[i, 5], 0.5, 4.5)))
        obs[i, 1:] = Z[1:, :2] + 60.0                       # far away: the controls are feasible
    kw = dict(nn_ctx=pb.nn_ctx if mode == "gt_mpc" else None, obs_psi=pb.obs_psi if mode == "obca" else None)
    ev = s.evaluate(pb.x0, pb.u_prev, pb.curv, obs, U, **kw)
    feas = ev["viol"] <= 1e-6
    assert feas.sum() >= 8
    Ub = U.copy()
    Ub[0, N - 1, 0] = np.nan                                # last acceleration
    Ub[1, N - 1, 1] = np.nan                                # last steering angle
    Ub[2, 0, 1] = np.nan                                    # first steering angle
    Ub[3, 20, 0] = np.inf
    Ub[4, 10:, 0] = 1e308                                   # finite, the state overflows
    Ub[5, 30, 0] = -np.inf
    bad = np.arange(6)
    evb = s.evaluate(pb.x0, pb.u_prev, pb.curv, obs, Ub, **kw)
    for i in bad:
        assert not np.isfinite(evb["cost"][i]), i
        assert not (evb["viol"][i] <= 1e-6), (i, evb["viol"][i])
    assert not np.all(np.isfinite(evb["x"][4]))
    rest = np.arange(6, 16)
    for k in ("cost", "viol", "x"):
        assert np.array_equal(evb[k][rest], ev[k][rest]), k
    s.close()
