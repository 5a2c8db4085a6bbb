"""Time the plain solve, the dual-exporting solve and the VJP call on the device (CUDA events, torch tensors, median of
--reps after warm-ups), at B = 32768 'mpc' (bench.py's config-2 generator) and B = 16384 gt_mpc with a bank of the
eight shipped networks (problem b plans with network b % 8).  Records the card name and power limit.

    python tools/vjp_probe.py [--out profiles/r6_vjp_probe.json] [--reps 20] [--warmup 3]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
from igt_mpc_int_b200 import scenarios as S              # noqa: E402
from igt_mpc_int_b200.planner import BatchSolver         # noqa: E402
from tools.latency_probe_gt import gpu_info, shipped     # noqa: E402


def time_ms(fn, reps, warmup):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); e1.synchronize()
        out.append(e0.elapsed_time(e1))
    return float(np.median(out)), float(np.min(out)), float(np.max(out))


def case(name, B, gt, reps, warmup):
    import torch
    pb = S.mid_episode(B, N=40, seed=2026)
    s = BatchSolver(N=40, mlp=[shipped(k) for k in range(1, 9)] if gt else None)
    T = lambda a, dt=torch.float64: torch.tensor(np.ascontiguousarray(a), dtype=dt, device="cuda")
    x0, up, cv, ob = T(pb.x0), T(pb.u_prev), T(pb.curv), T(pb.obs)
    ctx = T(pb.nn_ctx) if gt else None
    net = T(np.arange(B) % 8, torch.int32) if gt else None
    plain = lambda: s.solve_batch_device(x0, up, cv, ob, nn_ctx=ctx, net_idx=net)
    dual = lambda: s.solve_batch_device(x0, up, cv, ob, nn_ctx=ctx, net_idx=net, duals=True)
    r = dual()
    rng = np.random.default_rng(0)
    gx, gu, gc = T(rng.standard_normal((B, 41, 7))), T(rng.standard_normal((B, 40, 2))), T(rng.standard_normal(B))
    vjp = lambda: s.vjp_device(x0, up, cv, ob, r["u"], r["slack"], r["mult"], r["status"], gx, gu, gc, nn_ctx=ctx, net_idx=net)
    res = {"workload": name, "B": B, "mode": "gt_mpc bank (8 shipped networks)" if gt else "mpc"}
    for k, fn in (("plain_solve", plain), ("dual_solve", dual), ("vjp", vjp)):
        med, lo, hi = time_ms(fn, reps, warmup)
        res[k + "_ms"] = {"median": med, "min": lo, "max": hi}
    p = plain()
    res["dual_equals_plain"] = bool(all(torch.equal(torch.nan_to_num(p[k]), torch.nan_to_num(r[k]))
                                        for k in ("x", "u", "cost", "status", "iters")))
    g = vjp()
    st = r["status"].cpu().numpy()
    res["converged"] = int((st == 0).sum())
    res["vjp_ok"] = int(g["ok"].sum().item())
    print(json.dumps(res))
    s.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_vjp_probe.json"))
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    info = gpu_info()
    print(json.dumps(info))
    rows = [case("cfg2_mpc_32768", 32768, False, a.reps, a.warmup), case("gt_mpc_bank_16384", 16384, True, a.reps, a.warmup)]
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump({"device": info, "reps": a.reps, "warmup": a.warmup, "results": rows}, f, indent=1)


if __name__ == "__main__":
    main()
