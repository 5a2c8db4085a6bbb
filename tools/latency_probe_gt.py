"""Small-batch gt_mpc latency: throughput kernel vs the shared-memory latency path (igt_set_option "latency_path"),
host to host, in every value-term mode the latency path covers, plus the per-step latency of a host-driven gt_mpc
episode.  Both settings alternate in one process; the outputs of the two are compared bit for bit.

    python tools/latency_probe_gt.py [--out FILE.json] [--reps 15] [--episode-reps 2]

Modes: the shipped sc1 (2 hidden layers) and sc3 (3 hidden layers) networks with the exact cooperative value term,
a bank holding both (net_idx alternating in the batch), gt_mpc + OBCA (d_min = 0, per-thread value term) and fp32
gt_mpc (per-thread).  B = 1, 2, 8, 64 and the SM count, cold and warm-started from the cold solution."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
from igt_mpc_int_b200 import episode                     # noqa: E402
from igt_mpc_int_b200 import scenarios as S              # noqa: E402
from igt_mpc_int_b200.planner import BatchSolver         # noqa: E402

KEYS = ("status", "iters", "cost", "viol", "u", "x")
NETS = np.load(os.path.join(ROOT, "tests", "golden", "value_nets.npz"))   # the shipped V_GT_sc{1..8} weights


def shipped(k):
    n = int(NETS["sc%d_n_layers" % k])
    return dict(weights=[(NETS["sc%d_W%d" % (k, i)], NETS["sc%d_b%d" % (k, i)]) for i in range(n)], Wn=np.eye(6),
                mu_f=np.zeros(6), sigma_t=1.0, mu_t=0.0)


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0), "n_sm": torch.cuda.get_device_properties(0).multi_processor_count}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = q
    except Exception as e:                                  # the name from torch is still recorded
        info["nvidia_smi"] = "unavailable: %s" % e
    return info


def modes():
    n1, n3 = shipped(1), shipped(3)
    return {
        "gt_mpc_sc1_coop": (lambda: BatchSolver(N=40, mlp=n1), dict()),
        "gt_mpc_sc3_coop": (lambda: BatchSolver(N=40, mlp=n3), dict()),
        "gt_mpc_bank_sc1_sc3_coop": (lambda: BatchSolver(N=40, mlp=[n1, n3]), dict(bank=True)),
        "gt_mpc_obca_sc1_per_thread": (lambda: BatchSolver(N=40, mlp=n1, d_min=0.0), dict(obca=True)),
        "gt_mpc_f32_sc1_per_thread": (lambda: BatchSolver(N=40, mlp=n1, precision="f32"), dict()),
    }


def solve_latency(reps, n_sm):
    pb = S.mid_episode(152, N=40, seed=11)
    out = []
    for name, (make, how) in modes().items():
        s = make()
        for B in (1, 2, 8, 64, n_sm):
            a = dict(nn_ctx=pb.nn_ctx[:B])
            if how.get("obca"):
                a["obs_psi"] = pb.obs_psi[:B]
            if how.get("bank"):
                a["net_idx"] = (np.arange(B) % 2).astype(np.int32)
            args = (pb.x0[:B], pb.u_prev[:B], pb.curv[:B], pb.obs[:B])
            s.set_option("latency_path", 0)
            ui = np.nan_to_num(s.solve_batch(*args, **a)["u"])
            t = {(f, w): [] for f in (0, 1) for w in ("cold", "warm")}
            res = {}
            for _ in range(reps):
                for f in (0, 1):                               # alternating in the same process
                    s.set_option("latency_path", f)
                    t0 = time.perf_counter(); c = s.solve_batch(*args, **a); t[(f, "cold")].append(time.perf_counter() - t0)
                    t0 = time.perf_counter(); w = s.solve_batch(*args, u_init=ui, **a); t[(f, "warm")].append(time.perf_counter() - t0)
                    res[f] = (c, w)
            same = all(np.array_equal(res[0][i][k], res[1][i][k], equal_nan=True) for i in (0, 1) for k in KEYS)
            med = {"%s_ms_%s" % (w, "latency" if f else "throughput"): 1e3 * float(np.median(v)) for (f, w), v in t.items()}
            row = dict(mode=name, B=B, identical=bool(same), iters_cold_max=int(res[1][0]["iters"].max()),
                       iters_warm_max=int(res[1][1]["iters"].max()), **med)
            out.append(row)
            print("%-28s B=%3d cold %.2f -> %.2f ms, warm %.2f -> %.2f ms (throughput kernel -> latency path), identical: %s"
                  % (name, B, med["cold_ms_throughput"], med["cold_ms_latency"], med["warm_ms_throughput"], med["warm_ms_latency"],
                     same), flush=True)
        s.close()
    return out


def episode_latency(reps, steps=150):
    """host-driven scenario-1 gt_mpc episode with the shipped sc1 network: per-step latency (both vehicles' solves and
    the host glue), flag 0 and 1 alternating"""
    spec = episode.reference_episode_specs(scenarios=(1,))[:1]
    s = BatchSolver(N=40, mlp=shipped(1))
    s.set_option("latency_path", 1)
    episode.run_closed_loop(s, spec, steps=5, N=40, mode="gt_mpc")     # warm-up
    lat = {0: [], 1: []}
    runs = {}
    for _ in range(reps):
        for f in (0, 1):
            s.set_option("latency_path", f)
            r = episode.run_closed_loop(s, spec, steps=steps, N=40, mode="gt_mpc", record_latency=True)
            lat[f] += r.step_latency_ms
            runs[f] = r
    s.close()
    same = (np.array_equal(runs[0].z_cl, runs[1].z_cl) and np.array_equal(runs[0].u_cl, runs[1].u_cl)
            and np.array_equal(runs[0].solved, runs[1].solved))
    out = dict(steps=steps, reps=reps, identical=bool(same), solved_fraction=float(runs[1].solved.mean()))
    for f, name in ((0, "throughput"), (1, "latency")):
        v = np.array(lat[f])
        out["p50_ms_%s" % name] = float(np.percentile(v, 50))
        out["p90_ms_%s" % name] = float(np.percentile(v, 90))
    print("scenario-1 gt_mpc episode, %d steps x %d: p50 %.2f -> %.2f ms, p90 %.2f -> %.2f ms (throughput kernel -> latency "
          "path), identical: %s" % (steps, reps, out["p50_ms_throughput"], out["p50_ms_latency"], out["p90_ms_throughput"],
                                    out["p90_ms_latency"], same), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--episode-reps", type=int, default=2)
    a = ap.parse_args()
    info = gpu_info()
    print(info, flush=True)
    res = dict(info, solves=solve_latency(a.reps, info["n_sm"]), episode=episode_latency(a.episode_reps))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
