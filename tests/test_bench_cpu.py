"""bench.py's CPU legs (cpu_baseline, --impl reference) run without a GPU, in both cost modes (ADVICE r1: the gt_mpc
baseline used to crash for want of nn_ctx)."""
import json
import subprocess
import sys
import os

import numpy as np

import bench
from igt_mpc_int_b200 import scenarios as S

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def test_cpu_baseline_mpc_and_gt_mpc():
    pb = S.mid_episode(64, N=40, seed=2026)
    c, dt = bench.cpu_baseline(pb.x0, pb.u_prev, pb.curv, pb.obs, 40, "mpc", None, 64, 60)
    assert 40 <= c <= 64 and dt > 0
    for hidden in ((128, 128), (128, 128, 128)):
        c, dt = bench.cpu_baseline(pb.x0, pb.u_prev, pb.curv, pb.obs, 40, "gt_mpc", bench.random_mlp(hidden), 64, 60, ctx=pb.nn_ctx)
        assert 30 <= c <= 64 and dt > 0


def test_workload_table_and_sharded_problem_sets():
    for name, (gen, B, N, mode, scaling, hidden) in bench.WORKLOADS.items():
        assert scaling in ("weak", "strong") and mode in ("mpc", "gt_mpc") and (hidden is None) == (mode == "mpc")
    assert bench.WORKLOADS["cfg4_frenet_65536"][4] == "strong" and bench.WORKLOADS[bench.DEFAULT_WORKLOAD][1] == 32768


def test_dump_outputs_full_and_sampled(tmp_path, monkeypatch):
    import torch
    B, N = 50, 10
    g = torch.Generator().manual_seed(1)
    out = dict(x=torch.randn(B, N + 1, 7, generator=g, dtype=torch.float64), u=torch.randn(B, N, 2, generator=g, dtype=torch.float64),
               cost=torch.randn(B, generator=g, dtype=torch.float64), viol=torch.rand(B, generator=g, dtype=torch.float64),
               status=torch.arange(B, dtype=torch.int32) % 7, iters=torch.arange(B, dtype=torch.int32) + 5)
    names = ["x", "u", "cost", "viol", "status", "iters", "problem_index"]
    bench.dump_outputs(out, str(tmp_path / "full"))
    for k in names[:-1]:
        a = np.load(tmp_path / "full" / (k + ".npy"))
        assert a.dtype == np.float64 and np.array_equal(a, out[k].numpy().astype(np.float64))
    assert np.array_equal(np.load(tmp_path / "full" / "problem_index.npy"), np.arange(B))
    row_bytes = 8 * ((N + 1) * 7 + N * 2 + 5)
    monkeypatch.setattr(bench, "DUMP_BYTES", 20 * row_bytes + 128 * len(names))
    for d in ("a", "b"):
        bench.dump_outputs(out, str(tmp_path / d))
    idx = np.load(tmp_path / "a" / "problem_index.npy")
    assert len(idx) == 20 and np.all(np.diff(idx) > 0)
    assert sum(os.path.getsize(tmp_path / "a" / (k + ".npy")) for k in names) <= bench.DUMP_BYTES
    for k in names:
        a, b = np.load(tmp_path / "a" / (k + ".npy")), np.load(tmp_path / "b" / (k + ".npy"))
        assert np.array_equal(a, b)                                       # the same seeded sample every time
        if k != "problem_index":
            assert np.array_equal(a, out[k].numpy()[idx.astype(int)])


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-500:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port"
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["config"]["workload"] == bench.DEFAULT_WORKLOAD
