"""gt_mpc over all eight scenarios, each problem with its own scenario's value network (the shipped V_GT_sc{1..8} weights,
tests/golden/value_nets.npz): one network-bank solve against eight single-network solves.
16 384 mid_episode problems (sc1-8), device-resident inputs, CUDA events around every step, the L2 overwritten
(256 MiB memset) before every timed step as bench.py does.  Variants:
  a  one bank call, problems in scenario-major order (net_idx = scenario - 1)
  b  the same call with the problems shuffled, so that every CTA mixes networks
  c  eight single-network handles, one call each on its scenario's problems, one after another on one stream
  d  the existing single-network cfg3 run (bench.py's random 6-128-128-1 network for every problem) on the same problems
usage: mlp_bank_probe.py [B=16384] [steps=5] [warmup=2] -> one JSON line"""
import json, os, subprocess, sys
import numpy as np
import torch
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
import bench
from igt_mpc_int_b200 import scenarios as S
from igt_mpc_int_b200.planner import BatchSolver

B = int(sys.argv[1]) if len(sys.argv) > 1 else 16384
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
warmup = int(sys.argv[3]) if len(sys.argv) > 3 else 2
assert torch.cuda.is_available(), "needs a CUDA device"
dev = torch.device("cuda:0")
g = np.load(os.path.join(ROOT, "tests", "golden", "value_nets.npz"))


def shipped(k):
    n = int(g["sc%d_n_layers" % k])
    return dict(weights=[(g["sc%d_W%d" % (k, i)], g["sc%d_b%d" % (k, i)]) for i in range(n)], Wn=np.eye(6), mu_f=np.zeros(6),
                sigma_t=1.0, mu_t=0.0)


pb = S.mid_episode(B, N=40, seed=2026)
perm = np.random.default_rng(11).permutation(B)
T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def inputs(order):
    return dict(x0=T(pb.x0[order]), u_prev=T(pb.u_prev[order]), curv=T(pb.curv[order]), obs_xy=T(pb.obs[order]),
                nn_ctx=T(pb.nn_ctx[order]))


major, shuffled = np.arange(B), perm
bank = BatchSolver(N=40, mlp=[shipped(k) for k in range(1, 9)])
singles = [BatchSolver(N=40, mlp=shipped(k)) for k in range(1, 9)]
cfg3 = BatchSolver(N=40, mlp=bench.random_mlp((128, 128)))
for s in singles + [cfg3]:
    s.set_option("tensor_core_mlp", 0)
inp_major, inp_shuf = inputs(major), inputs(shuffled)
idx_major = T((pb.scenario[major] - 1).astype(np.int32))
idx_shuf = T((pb.scenario[shuffled] - 1).astype(np.int32))
blocks = [np.where(pb.scenario == k)[0] for k in range(1, 9)]
inp_blocks = [inputs(bl) for bl in blocks]
outs = {}


def run_a():
    return [bank.solve_batch_device(**inp_major, net_idx=idx_major)]


def run_b():
    return [bank.solve_batch_device(**inp_shuf, net_idx=idx_shuf)]


def run_c():
    return [s.solve_batch_device(**inp) for s, inp in zip(singles, inp_blocks)]


def run_d():
    return [cfg3.solve_batch_device(**inp_major)]


flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
res = {}
for name, fn in (("a_bank_scenario_major", run_a), ("b_bank_shuffled", run_b), ("c_eight_single_handles", run_c),
                 ("d_cfg3_single_network", run_d)):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms, conv = [], 0
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
        conv = sum(int((o["status"] == 0).sum().item()) for o in out)
    outs[name] = out
    res[name] = {"ms_per_step_median": float(np.median(ms)), "ms_per_step_all": [float(v) for v in ms],
                 "converged_per_step": conv, "converged_solves_per_s": conv / (np.median(ms) * 1e-3)}
# the bank results are the single-network handles' results, bit for bit (a vs c, b vs c)
st_c = np.empty(B, dtype=np.int32); cost_c = np.empty(B)
for bl, o in zip(blocks, outs["c_eight_single_handles"]):
    st_c[bl] = o["status"].cpu().numpy(); cost_c[bl] = o["cost"].cpu().numpy()
a = outs["a_bank_scenario_major"][0]; b = outs["b_bank_shuffled"][0]
st_b = np.empty(B, dtype=np.int32); st_b[shuffled] = b["status"].cpu().numpy()
cost_b = np.empty(B); cost_b[shuffled] = b["cost"].cpu().numpy()
res["a_equals_c_bitwise"] = bool(np.array_equal(a["status"].cpu().numpy(), st_c) and np.array_equal(a["cost"].cpu().numpy(), cost_c, equal_nan=True))
res["b_equals_c_bitwise"] = bool(np.array_equal(st_b, st_c) and np.array_equal(cost_b, cost_c, equal_nan=True))
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
res.update({"B": B, "steps": steps, "warmup": warmup, "device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip(),
            "l2": "flushed (256 MiB memset) before every timed step",
            "ratio_c_over_a": res["c_eight_single_handles"]["ms_per_step_median"] / res["a_bank_scenario_major"]["ms_per_step_median"],
            "ratio_a_over_d": res["a_bank_scenario_major"]["ms_per_step_median"] / res["d_cfg3_single_network"]["ms_per_step_median"]})
for s in singles + [bank, cfg3]:
    s.close()
print(json.dumps(res))
