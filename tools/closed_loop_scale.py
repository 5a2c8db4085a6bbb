"""2048 closed-loop episodes (32 draws of the start offsets x the 64 (scenario, rotation, order) variants) x 150 steps:
host-driven numpy glue vs the device-side loop (igt_episode_run_host).
usage: closed_loop_scale.py [draws=32] [device|host|both] [circle|obca] [mpc|gt_mpc]
obca: collision_avoidance_type 'obca' (d_min = 0); also reports the smallest signed rectangle gap over all episodes and
steps (oracle.obca.rect_distance).
gt_mpc: every episode plans with its scenario's shipped value network (tests/golden/value_nets.npz): all episodes in one
device loop with the network bank (net_idx = scenario - 1, "device"), then the same episodes as eight per-scenario device
loops with single-network handles ("device_per_scenario"); the host-driven loop is not run in this mode."""
import json, os, sys, time
import numpy as np
sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
from igt_mpc_int_b200 import episode
from igt_mpc_int_b200.planner import BatchSolver

draws = int(sys.argv[1]) if len(sys.argv) > 1 else 32
which = sys.argv[2] if len(sys.argv) > 2 else "both"
ca_type = sys.argv[3] if len(sys.argv) > 3 else "circle"
mode = sys.argv[4] if len(sys.argv) > 4 else "mpc"
assert ca_type in ("circle", "obca") and mode in ("mpc", "gt_mpc"), (ca_type, mode)
specs = [sp for d in range(draws) for sp in episode.reference_episode_specs(sample=d)]
d_min = 0.0 if ca_type == "obca" else 5.6
out = {"episodes": len(specs), "steps": 150, "ca_type": ca_type, "mode": mode}


def shipped(k):
    g = np.load(os.path.join(os.path.dirname(__file__), "..", "tests", "golden", "value_nets.npz"))
    n = int(g["sc%d_n_layers" % k])
    return dict(weights=[(g["sc%d_W%d" % (k, i)], g["sc%d_b%d" % (k, i)]) for i in range(n)], Wn=np.eye(6), mu_f=np.zeros(6),
                sigma_t=1.0, mu_t=0.0)


if mode == "gt_mpc":
    s = BatchSolver(N=40, d_min=d_min, mlp=[shipped(k) for k in range(1, 9)])
    net_idx = np.array([sp.scenario - 1 for sp in specs])
    # (the warm-up runs the first draw, a prefix of specs)
    bank_loop = lambda sv, sp, **kw: episode.run_closed_loop_device(sv, sp, mode="gt_mpc", net_idx=net_idx[:len(sp)], **kw)
    singles = [BatchSolver(N=40, d_min=d_min, mlp=shipped(k)) for k in range(1, 9)]

    def per_scenario(sv, sp, **kw):   # eight loops, one per scenario, each with its own single-network handle
        parts = [episode.run_closed_loop_device(singles[k], [x for x in sp if x.scenario == k + 1], mode="gt_mpc", **kw)
                 for k in range(8)]
        order = np.argsort(np.concatenate([[i for i, x in enumerate(sp) if x.scenario == k + 1] for k in range(8)]), kind="stable")
        cat = lambda f: np.concatenate([getattr(p, f) for p in parts])[order]
        return episode.EpisodeResult(z_cl=cat("z_cl"), u_cl=cat("u_cl"), solved=cat("solved"), deadlock=cat("deadlock"),
                                     collision=cat("collision"), goal=cat("goal"), num_infeasible=cat("num_infeasible"),
                                     min_distance=cat("min_distance"),
                                     step_latency_ms=list(np.sum([p.step_latency_ms for p in parts], axis=0)) if kw.get("record_latency") else [])
    loops = (("device", bank_loop), ("device_per_scenario", per_scenario))
else:
    s = BatchSolver(N=40, d_min=d_min)
    loops = (("device", lambda sv, sp, **kw: episode.run_closed_loop_device(sv, sp, **kw)),
             ("host", lambda sv, sp, **kw: episode.run_closed_loop(sv, sp, **kw)))
for name, fn in loops:
    if which not in (name, "both") and not (mode == "gt_mpc" and which == "device"):
        continue
    fn(s, specs[:64], steps=5, N=40, ca_type=ca_type)      # warm-up
    t0 = time.perf_counter()
    r = fn(s, specs, steps=150, N=40, record_latency=True, ca_type=ca_type)
    dt = time.perf_counter() - t0
    n_solves = 2 * len(specs) * 150
    out[name] = {"wall_s": dt, "solves_per_s_incl_glue": n_solves / dt, "failed_solve_fraction": float(1 - r.solved.mean()),
                 "deadlocks": int(r.deadlock.sum()), "collisions": int(r.collision.sum()), "goals_both": int(r.goal.all(axis=1).sum()),
                 "min_distance": float(r.min_distance.min()), "p50_step_ms": float(np.percentile(r.step_latency_ms, 50))}
    if ca_type == "obca":
        from oracle import obca
        z = r.z_cl[..., [0, 1, 6]]
        dc = np.hypot(z[:, 0, :, 0] - z[:, 1, :, 0], z[:, 0, :, 1] - z[:, 1, :, 1])
        # gap >= centre distance - 2 circumradii (2 x 2.449 m) and gap <= centre distance - width (2 m): only pairs
        # within 2.9 m of the closest centre distance can hold the smallest gap
        cand = np.argwhere(dc <= dc.min() + 2.9)
        out[name]["min_rect_gap"] = float(min(obca.rect_distance(z[e, 0, t], z[e, 1, t])[0] for e, t in cand))
s.close()
if mode == "gt_mpc":
    for sv in singles:
        sv.close()
print(json.dumps(out))
