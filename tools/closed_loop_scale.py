"""2048 closed-loop episodes (32 draws of the start offsets x the 64 (scenario, rotation, order) variants) x 150 steps:
host-driven numpy glue vs the device-side loop (igt_episode_run_host).
usage: closed_loop_scale.py [draws=32] [device|host|both] [circle|obca]
obca: collision_avoidance_type 'obca' (d_min = 0); also reports the smallest signed rectangle gap over all episodes and
steps (oracle.obca.rect_distance)."""
import json, os, sys, time
import numpy as np
sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
from igt_mpc_int_b200 import episode
from igt_mpc_int_b200.planner import BatchSolver

draws = int(sys.argv[1]) if len(sys.argv) > 1 else 32
which = sys.argv[2] if len(sys.argv) > 2 else "both"
ca_type = sys.argv[3] if len(sys.argv) > 3 else "circle"
assert ca_type in ("circle", "obca"), ca_type
specs = [sp for d in range(draws) for sp in episode.reference_episode_specs(sample=d)]
s = BatchSolver(N=40, d_min=0.0 if ca_type == "obca" else 5.6)
out = {"episodes": len(specs), "steps": 150, "ca_type": ca_type}
for name, fn in (("device", episode.run_closed_loop_device), ("host", episode.run_closed_loop)):
    if which not in (name, "both"):
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
print(json.dumps(out))
