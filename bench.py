#!/usr/bin/env python
"""bench.py -- converged MPC solves/sec of the batched solver (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path (cold-start guess kernel + persistent solver kernel) over
one batch of synthetic problems.  Default workload = BASELINE.json configs[1]: 'mpc' mode,
scenarios 1-8, 4096 synthetic initial conditions per scenario (32768 problems), horizon N=40,
on ONE B200; with --gpus N every rank solves its own batch of that size (weak scaling; no
data-path collective -- NCCL only gathers the counters).

value   = converged solves/s, inputs resident in HBM, CUDA events around the kernels
e2e     = same metric through the host-pointer C ABI call (igt_solve_host): pinned host buffers,
          H2D of the inputs and D2H of x, u, cost, viol, status, iters inside the timed region
--impl reference: the reference's own solver (CasADi/IPOPT) cannot run offline, so this arm times
          the oracle's fp64 C restatement of the same NLP/algorithm on all host cores.
--dump-outputs DIR: after the timed steps, rank 0 writes what the last timed step returned (x, u, cost,
          viol, status, iters) as DIR/<name>.npy in float64, so that two builds can be compared output
          for output on the same seeded inputs (see dump_outputs).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "converged MPC solves/sec"
UNIT = "solves/s"

WORKLOADS = {
    # name: (generator, problems [per GPU if weak, in total if strong], horizon, mode, scaling, value-network hidden layers)
    "cfg2_mpc_sc1-8_4096ic": ("mid_episode", 32768, 40, "mpc", "weak", None),
    "cfg2_episode_start": ("episode_start", 32768, 40, "mpc", "weak", None),
    # BASELINE config 4: 65536 sampled states in TOTAL, sharded over the GPUs (strong scaling)
    "cfg4_frenet_65536": ("mid_episode", 65536, 40, "mpc", "strong", None),
    # BASELINE config 5: 2^20 problems over 8 GPUs = 131072 per GPU, horizon sweep (weak: per-GPU share fixed)
    "cfg5_131072_N40": ("mid_episode", 131072, 40, "mpc", "weak", None),
    "cfg5_131072_N20": ("mid_episode", 131072, 20, "mpc", "weak", None),
    "cfg5_131072_N10": ("mid_episode", 131072, 10, "mpc", "weak", None),
    # BASELINE config 3: gt_mpc, random-init value network, both shapes the reference ships (sc*_config.yaml num_layers 2 / 3)
    "cfg3_gt_mpc_16384": ("mid_episode", 16384, 40, "gt_mpc", "weak", (128, 128)),
    "cfg3_gt_mpc_16384_3hidden": ("mid_episode", 16384, 40, "gt_mpc", "weak", (128, 128, 128)),
}
DEFAULT_WORKLOAD = "cfg2_mpc_sc1-8_4096ic"
MAX_ITER_DEFAULT = 60        # the library's default iteration cap (igt_default_params); the CPU arm uses the same


def make_problems(name, rank, world=1, scaling=None):
    """This rank's problems.  weak: every rank draws its own batch (seed + 1000 rank); strong: every rank draws the
    SAME full batch and keeps its contiguous block (sharding.shard_range)."""
    from igt_mpc_int_b200 import scenarios as S, sharding
    gen, B, N, mode, default_scaling, _ = WORKLOADS[name]
    scaling = scaling or default_scaling
    strong = scaling == "strong"
    seed = {"cfg4_frenet_65536": 4}.get(name, 2026) + (0 if strong else 1000 * rank)      # SURVEY 8(d): seeds 2026+sc / 4
    cache = os.path.join(tempfile.gettempdir(), "igt_bench_%s_s%d.npz" % (name, seed))
    if os.path.exists(cache):
        d = np.load(cache)
        arrs = [d["x0"], d["up"], d["cv"], d["ob"], d["ctx"]]
    else:
        pb = getattr(S, gen)(B, N=N, seed=seed)
        arrs = [pb.x0, pb.u_prev, pb.curv, pb.obs, pb.nn_ctx]
        try:
            tmp = cache + ".%d.tmp.npz" % os.getpid()
            np.savez(tmp, x0=pb.x0, up=pb.u_prev, cv=pb.curv, ob=pb.obs, ctx=pb.nn_ctx)
            os.replace(tmp, cache)
        except OSError:
            pass
    if strong:
        lo, hi = sharding.shard_range(B, rank, world)
        arrs = [a[lo:hi] for a in arrs]
    return arrs[0], arrs[1], arrs[2], arrs[3], arrs[4], N, mode


def random_mlp(hidden=(128, 128), seed=2026):
    """Random-init value network, torch.nn.Linear default init in fp64 (SURVEY 8(d) config 3)."""
    import torch
    torch.manual_seed(seed)
    dims = [6] + list(hidden) + [1]
    layers = [torch.nn.Linear(dims[i], dims[i + 1], dtype=torch.double) for i in range(len(dims) - 1)]
    weights = [(l.weight.detach().numpy().copy(), l.bias.detach().numpy().copy()) for l in layers]
    return dict(weights=weights, Wn=np.eye(6), mu_f=np.zeros(6), sigma_t=1.0, mu_t=0.0)


DUMP_BYTES = 64 * 10**6     # --dump-outputs writes at most this much, .npy headers included


def dump_outputs(out, directory):
    """Write the solver's outputs (x[B,N+1,7], u[B,N,2], cost, viol, status, iters) as <directory>/<name>.npy in
    float64.  When all B problems do not fit in DUMP_BYTES, the same fixed, seeded sample of problems is kept in every
    array, and problem_index.npy says which ones they are."""
    arrs = {k: v.cpu().numpy() for k, v in out.items()}
    B = len(arrs["cost"])
    row_bytes = 8 * (sum(a[0].size for a in arrs.values()) + 1)               # + 1: the problem's index
    keep = min(B, (DUMP_BYTES - 128 * (len(arrs) + 1)) // row_bytes)
    idx = np.arange(B) if keep == B else np.sort(np.random.default_rng(0).choice(B, keep, replace=False))
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "problem_index.npy"), idx.astype(np.float64))
    for name, a in arrs.items():
        np.save(os.path.join(directory, name + ".npy"), a[idx].astype(np.float64))


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples = index, threading.Event(), []

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = sorted(float(s[0]) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons}


def cpu_baseline(x0, up, cv, ob, N, mode, mlp, n_sample, max_iter, threads=0, max_trials=0, ctx=None):
    """The oracle's C restatement timed on the host cores on the first n_sample problems."""
    from oracle import nlp, c_oracle
    P = nlp.Params(N=N)
    term = None
    if mode == "gt_mpc":
        term = nlp.MLPTerm(weights=mlp["weights"], Wn=mlp["Wn"], mu_f=mlp["mu_f"], sigma_t=mlp["sigma_t"], mu_t=mlp["mu_t"])
    co = c_oracle.COracle(P, term, max_iter=max_iter, max_trials=max_trials)
    c_of = lambda n: None if term is None else ctx[:n]
    co.solve(x0[:64], up[:64], cv[:64], ob[:64], nn_ctx=c_of(64), n_threads=threads)           # warm the library / page in
    t0 = time.perf_counter()
    r = co.solve(x0[:n_sample], up[:n_sample], cv[:n_sample], ob[:n_sample], nn_ctx=c_of(n_sample), n_threads=threads)
    dt = time.perf_counter() - t0
    return int((r["status"] == 0).sum()), dt


def run_reference(args, rank, world):
    """--impl reference: CPU arm (rank 0 only)."""
    if rank != 0:
        return
    x0, up, cv, ob, ctx, N, mode = make_problems(args.workload, 0)
    hidden = WORKLOADS[args.workload][5]
    mlp = random_mlp(hidden) if mode == "gt_mpc" else None
    cores = os.cpu_count() or 1
    n_sample = min(len(x0), max(256, 64 * cores))
    for _ in range(args.warmup):
        cpu_baseline(x0, up, cv, ob, N, mode, mlp, min(256, n_sample), MAX_ITER_DEFAULT, ctx=ctx)
    conv, tsum = 0, 0.0
    for _ in range(args.steps):
        c, dt = cpu_baseline(x0, up, cv, ob, N, mode, mlp, n_sample, MAX_ITER_DEFAULT, ctx=ctx)
        conv += c
        tsum += dt
    val = conv / tsum
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tsum / args.steps, "higher_is_better": True,
        "scaling": args.scaling or WORKLOADS[args.workload][4],
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "horizon": N, "mode": mode, "problems_per_step": n_sample},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "first %d problems of the workload per step, all host threads; the reference's "
                                   "CasADi/IPOPT solver is not installable offline, so the oracle's fp64 C restatement "
                                   "of the same NLP is timed (per-solve throughput is comparable with the GPU arm's: "
                                   "same problems, same algorithm and tolerances, same iteration cap)" % n_sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


_REAL_STDOUT = None


def emit(line):
    """Print the one JSON line on the real stdout (fd 1 is pointed at stderr while the bench runs, so that
    library chatter such as NCCL's version banner cannot end up next to it)."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="f64", choices=["f64", "f32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-closed-loop", action="store_true")
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"],
                    help="default: the workload's own (cfg4 = strong: 65536 states in total, sharded)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the solver has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from igt_mpc_int_b200.planner import BatchSolver
    from igt_mpc_int_b200 import sharding
    scaling = args.scaling or WORKLOADS[args.workload][4]
    x0, up, cv, ob, ctx, N, mode = make_problems(args.workload, rank, world, scaling)
    B = len(x0)
    hidden = WORKLOADS[args.workload][5]
    mlp = random_mlp(hidden) if mode == "gt_mpc" else None
    solver = BatchSolver(N=N, precision=args.precision, mlp=mlp)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    dx0, dup, dcv, dob = t(x0), t(up), t(cv), t(ob)
    dctx = t(ctx) if mode == "gt_mpc" else None
    # All outputs of a rank live in ONE flat buffer (x | u | cost | viol | status, iters), so that with several GPUs the
    # solutions are gathered by one all_gather_into_tensor over NVLink (north star: "NCCL ... only to gather solutions
    # and metrics").  Strong-scaling blocks may differ by one problem: the buffer is sized for the largest block.
    Bmax = B
    if world > 1:
        bm = torch.tensor([B], device=dev)
        dist.all_reduce(bm, op=dist.ReduceOp.MAX)
        Bmax = int(bm.item())
    n64 = Bmax * ((N + 1) * 7 + N * 2 + 2)
    flat = torch.zeros(n64 + Bmax, dtype=torch.float64, device=dev)        # + Bmax doubles = 2 Bmax int32
    o = 0
    def view(n, shape):
        nonlocal o
        v = flat[o:o + n].view(shape); o += n
        return v
    out = dict(x=view(B * (N + 1) * 7, (B, N + 1, 7)), u=view(B * N * 2, (B, N, 2)), cost=view(B, (B,)), viol=view(B, (B,)))
    ints = flat[n64:].view(torch.int32)
    out["status"], out["iters"] = ints[:B], ints[Bmax:Bmax + B]
    gathered = torch.empty((world, flat.numel()), dtype=torch.float64, device=dev) if world > 1 else None
    solver.solve_batch_device(dx0, dup, dcv, dob, nn_ctx=dctx, out=out)
    torch.cuda.synchronize()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        solver.solve_batch_device(dx0, dup, dcv, dob, nn_ctx=dctx, out=out)
        if world > 1:
            dist.all_gather_into_tensor(gathered.view(-1), flat)            # every rank ends up with every solution

    for _ in range(args.warmup):
        step()
    barrier()

    # ---- device-resident timing: CUDA events around every step, L2 flushed between steps ----
    l0 = solver.launches
    sampler = ClockSampler(local_rank)
    sampler.start()
    evs = [tuple(torch.cuda.Event(enable_timing=True) for _ in range(3)) for _ in range(args.steps)]
    barrier()
    wall0 = time.perf_counter()
    for e0, em, e1 in evs:
        flush.zero_()
        e0.record()
        solver.solve_batch_device(dx0, dup, dcv, dob, nn_ctx=dctx, out=out)
        em.record()
        if world > 1:
            dist.all_gather_into_tensor(gathered.view(-1), flat)
        e1.record()
    barrier()
    wall = time.perf_counter() - wall0
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    launches = solver.launches - l0
    step_ms = [e0.elapsed_time(e1) for e0, em, e1 in evs]
    solve_ms = float(sum(e0.elapsed_time(em) for e0, em, e1 in evs))
    coll_ms = float(sum(em.elapsed_time(e1) for e0, em, e1 in evs))
    dev_ms = float(sum(step_ms))
    status = out["status"].cpu().numpy()
    iters = out["iters"].cpu().numpy()
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)
    conv_per_step = int((status == 0).sum())
    acc_per_step = int((status == 6).sum())
    dev_ms_max, conv_all, iters_all, B_all = sharding.reduce_counters(dev_ms, conv_per_step, iters.sum(), B, device=dev)
    coll_ms_max, acc_all, _, _ = sharding.reduce_counters(coll_ms, acc_per_step, 0, 0, device=dev)
    value = conv_all * args.steps / (dev_ms_max * 1e-3)
    if world > 1:      # the gathered buffer really holds every rank's statuses (checked once, outside the timed region)
        st_all = torch.cat([gathered[r, n64:].view(torch.int32)[:B] for r in range(world)]) if scaling != "strong" else None
        if st_all is not None:
            assert int((st_all == 0).sum().item()) == int(conv_all), "gathered solutions do not match the reduced counters"

    # ---- end-to-end: host-pointer C ABI call with pinned host buffers ----
    hin = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in (x0, up, cv, ob)]
    hctx = torch.from_numpy(np.ascontiguousarray(ctx)).pin_memory() if mode == "gt_mpc" else None
    hout = dict(x=torch.empty((B, N + 1, 7), dtype=torch.float64).pin_memory(),
                u=torch.empty((B, N, 2), dtype=torch.float64).pin_memory(),
                cost=torch.empty(B, dtype=torch.float64).pin_memory(), viol=torch.empty(B, dtype=torch.float64).pin_memory(),
                status=torch.empty(B, dtype=torch.int32).pin_memory(), iters=torch.empty(B, dtype=torch.int32).pin_memory())
    hout_np = {k: v.numpy() for k, v in hout.items()}
    hin_np = [a.numpy() for a in hin]
    h2d = sum(a.nbytes for a in hin_np) + (hctx.numpy().nbytes if hctx is not None else 0)
    d2h = sum(v.nbytes for v in hout_np.values())
    e2e_steps = args.steps
    solver.solve_batch(*hin_np, nn_ctx=None if hctx is None else hctx.numpy(), out=hout_np)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        solver.solve_batch(*hin_np, nn_ctx=None if hctx is None else hctx.numpy(), out=hout_np)
    torch.cuda.synchronize()
    e2e_t = time.perf_counter() - t0
    e2e_conv = int((hout_np["status"] == 0).sum())
    e2e_t, e2e_conv_all, _, _ = sharding.reduce_counters(e2e_t, e2e_conv, 0, 0, device=dev)
    e2e_value = e2e_conv_all * e2e_steps / e2e_t

    # ---- p50 per-step solve latency of a closed-loop episode (second half of BASELINE.json's metric):
    #      scenario 1, both vehicles per step (B = 2), 150 steps, host to host through solve_batch ----
    cl_p50 = cl_p90 = cl_cpu_p50 = cl_cpu_p90 = None
    if rank == 0 and mode == "mpc" and not args.no_closed_loop:
        from igt_mpc_int_b200 import episode
        spec = episode.reference_episode_specs(scenarios=[1])[:1]
        cl_solver = solver if N == 40 else BatchSolver(N=40, precision=args.precision)
        res = episode.run_closed_loop(cl_solver, spec, steps=150, N=40, record_latency=True)
        cl_p50, cl_p90 = float(np.percentile(res.step_latency_ms, 50)), float(np.percentile(res.step_latency_ms, 90))
        if cl_solver is not solver:
            cl_solver.close()
        if not args.no_cpu_baseline:        # the same episode with the oracle's C port as the solver (2 host threads: one per vehicle)
            from tests.oracle_backend import OracleBackend
            ro = episode.run_closed_loop(OracleBackend(N=40, max_iter=MAX_ITER_DEFAULT), spec, steps=150, N=40, record_latency=True)
            cl_cpu_p50, cl_cpu_p90 = float(np.percentile(ro.step_latency_ms, 50)), float(np.percentile(ro.step_latency_ms, 90))

    if rank == 0:
        # ---- rooflines ----
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        traffic = traffic_gbs = None                          # dram bytes per launch from the committed ncu capture
        tr = {}
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if tr.get("workload") == args.workload and tr.get("precision") == args.precision:
                traffic = tr["dram_bytes_per_launch"]
                traffic_gbs = traffic / (tr["launch_ms_under_ncu"] * 1e-3) / 1e9
        except Exception:
            pass
        kernel_ms = solve_ms / args.steps                     # solver + guess kernels of one step on this rank
        alg_bytes = 8.0 * (11 * N + 24) * B                   # SURVEY 8(d): 4(11N+24) B/solve for fp32 I/O; ours is fp64
        achieved_gbs = alg_bytes / (kernel_ms * 1e-3) / 1e9
        stage_iters = float(iters.sum()) * N
        alg_flops = stage_iters * 1.4e4                       # SURVEY 8(d): 1.4e4 FLOP per stage-iteration
        fma_peak = solver.measure_fma_peak()
        # measured fp64 work: thread-level DFMA / DADD / DMUL of the solver kernel counted by ncu in the committed
        # capture (profiles/traffic.json), scaled by this run's stage-iterations
        meas_flops = None
        try:
            if tr.get("workload") == args.workload and tr.get("precision") == args.precision and "fp64_flop_per_stage_iter" in tr:
                meas_flops = stage_iters * float(tr["fp64_flop_per_stage_iter"])
        except Exception:
            pass
        roof_flops = meas_flops if meas_flops is not None else alg_flops
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": args.precision, "data": "synthetic",
            "config": {"workload": args.workload, "horizon": N, "mode": mode,
                       "problems_per_gpu_per_step": B, "problems_per_step_all_gpus": int(B_all),
                       "l2": "flushed (256 MiB memset) between timed steps", "warm_start": False,
                       "value_network": None if hidden is None else "6-" + "-".join(str(h) for h in hidden) + "-1 random init, exact fp64 value term",
                       "parallelism": "dp%d: independent problems, contiguous block per rank; %s" % (
                           world, "one all_gather_into_tensor of every rank's solutions per step inside the timed region"
                           if world > 1 else "single GPU")},
            "converged_fraction": conv_all / B_all, "mean_iterations": iters_all / B_all,
            "ipopt_band": {"acceptable_per_step": int(acc_all), "fraction": acc_all / B_all,
                           "what": "solves that failed the tight tolerances (1e-6 / 1e-8 / 1e-7) but stopped at a point inside the "
                                   "reference's own IPOPT tolerances (mpc.py:133-135, tol 1e-3; status 6): NOT counted in value"},
            "p50_step_latency_ms": float(np.median(step_ms)), "wall_ms_per_step_incl_flush": 1e3 * wall / args.steps,
            "solve_ms_per_step": solve_ms / args.steps,
            "collective_ms_per_step": coll_ms_max / args.steps if world > 1 else 0.0,
            "gathered_bytes_per_step": int(flat.numel() * 8 * world) if world > 1 else 0,
            "closed_loop_step_latency_ms": {"p50": cl_p50, "p90": cl_p90, "cpu_p50": cl_cpu_p50, "cpu_p90": cl_cpu_p90,
                                            "what": "scenario 1 episode, 150 steps, one B=2 solve per step (both vehicles), "
                                                    "host to host incl. H2D/D2H, warm-started after step 0; cpu_* = the same "
                                                    "episode with the oracle's fp64 C port as the solver on the host"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(launches),
            # the binding roofline of this path is the FP64 CUDA-core pipe (SURVEY 8(d)), not HBM bytes
            "roofline": {"bound": "fp64-fma", "achieved": roof_flops / (kernel_ms * 1e-3) / 1e12, "peak": fma_peak, "unit": "TFLOP/s",
                         "frac": roof_flops / (kernel_ms * 1e-3) / 1e12 / fma_peak, "traffic": traffic,
                         "flops_source": "ncu-counted DFMA x2 + DADD + DMUL thread instructions per stage-iteration (profiles/traffic.json) x "
                                         "this run's stage-iterations" if meas_flops is not None else
                                         "SURVEY 8(d) estimate 1.4e4 FLOP per stage-iteration x this run's stage-iterations",
                         "peak_source": "dependent-free fp64 FMA chains measured on this GPU in this run (MEASURED_PEAKS.json has no fp64 figure)",
                         "algorithmic_frac": alg_flops / (kernel_ms * 1e-3) / 1e12 / fma_peak},
            "hbm_traffic": {"bound": "hbm", "algorithmic_gbs": achieved_gbs, "peak": hbm_peak, "unit": "GB/s",
                            "algorithmic_frac": achieved_gbs / hbm_peak, "peak_source": hbm_src,
                            "dram_bytes_per_launch": traffic, "drawn_gbs": traffic_gbs,
                            "drawn_frac": None if traffic_gbs is None else traffic_gbs / hbm_peak,
                            "wasted_ratio": None if traffic is None else traffic / alg_bytes,
                            "note": "algorithmic = 8*(11N+24) bytes per solve; dram_bytes = dram__bytes_read + write of the solver "
                                    "kernel (ncu, committed capture): the per-problem workspace streams through HBM in every phase"},
            "clocks": sampler.summary(),
        }
        if not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            n_sample = min(B, max(512, 128 * cores))
            c, dt = cpu_baseline(x0, up, cv, ob, N, mode, mlp, n_sample, solver.params.max_iter,
                                 max_trials=solver.params.max_trials, ctx=ctx)
            n1 = min(B, 192)
            c1, dt1 = cpu_baseline(x0, up, cv, ob, N, mode, mlp, n1, solver.params.max_iter, threads=1,
                                   max_trials=solver.params.max_trials, ctx=ctx)
            line["cpu_baseline"] = {"value": c / dt, "unit": UNIT, "cores": cores, "kind": "port",
                                    "single_core_value": c1 / dt1, "single_core_sample": "first %d problems, 1 thread" % n1,
                                    "sample": "first %d problems of the same batch, oracle fp64 C restatement on all "
                                              "host threads (the reference's CasADi/IPOPT solver is not installable "
                                              "offline)" % n_sample}
        emit(line)
    solver.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
