"""Closed-loop evaluation with the reference's command line and result files (BASELINE config 1):

    python -m igt_mpc_int_b200.evaluate --save_dir runs/ --eval_mode mpc --sc 1 [--num_samples 1]

mirrors `python evaluate.py --save_dir ... --eval_mode mpc --sc 1` (evaluate.py:26-650): the same
scenario sampling (default_rng(2026) start offsets in region order, evaluate.py:56,:91-94), reference
tracks, closed loop (igt_mpc_int_b200.episode), deadlock flag and result files
(igt_mpc_int_b200.results), with the GPU solver in place of CasADi/IPOPT.  The reference picks the
rotation of the scenario and the order of the two vehicles with an unseeded `random.choice`
(utils.py:177-179); here they are arguments (--rotation, --order; --all_variants runs the eight of them).
No video is rendered (evaluate.py:589 needs matplotlib/ffmpeg: out of scope).

`--ca_type obca` runs the reference's other collision-avoidance mode (mpc.yaml collision_avoidance_type, mpc.py:42-43):
rectangle rows with d_min = 0 instead of the 5.6 m circle gap; an episode's collision flag then means that the two
4.47 x 2.0 rectangles overlapped at a recorded step (min_distance stays the centre distance).

`--eval_mode gt_mpc` needs the value network: --nn_weights FILE.npz with arrays W0, b0, W1, b1, ...
(model.py:14-51 layer order) and optionally Wn, mu_f, sigma_t, mu_t (mpc.py:109-118; the reference's
processed_sc*.pkl statistics are not shipped, identity / zero are used when absent).

`--sc all` runs the episodes of all eight scenarios through ONE closed loop (one batched solve per step for every
vehicle of every scenario) and writes one run directory per scenario, laid out as for `--sc k`.  In gt_mpc mode the
reference plans scenario k with its own network V_GT_sc{k} (evaluate.py:123): a --nn_weights path containing `{sc}`
is filled in per scenario, and with `--sc all` the eight networks form the solver's network bank (episode of
scenario k -> slot k - 1).  A plain path is one network for every scenario.
"""
import argparse
import datetime
import os

import numpy as np

from . import episode, geometry as G, reference_track as RT, results

POLICY_CONFIG = {   # the reference's mpc.yaml (note v_min: -1.0 there; MPC_Planner's own row uses 0, mpc.py:56)
    'type': 'MPC', 'NN_type': 't+N', 'input_sequence_length': 5, 'N': 40, 'dt': 0.1, 'a_min': -4, 'a_max': 3,
    'v_min': -1.0, 'v_max': 5, 'prediction_type': 'constant_acceleration', 'collision_avoidance_type': 'circle',
}


def load_mlp(path):
    d = np.load(path)
    n = len([k for k in d.files if k.startswith('W') and k[1:].isdigit()])
    weights = [(d['W%d' % i], d['b%d' % i]) for i in range(n)]
    return dict(weights=weights, Wn=d['Wn'] if 'Wn' in d.files else np.eye(6),
                mu_f=d['mu_f'] if 'mu_f' in d.files else np.zeros(6),
                sigma_t=float(d['sigma_t']) if 'sigma_t' in d.files else 1.0,
                mu_t=float(d['mu_t']) if 'mu_t' in d.files else 0.0)


def networks(path, scenarios):
    """--nn_weights for the given scenarios: a plain path or one scenario -> one network dict; a path with `{sc}` and
    several scenarios -> the network bank, a list with entry k - 1 = scenario k's network (None for the others)."""
    if '{sc}' not in path:
        return load_mlp(path)
    if len(scenarios) == 1:
        return load_mlp(path.format(sc=scenarios[0]))
    return [load_mlp(path.format(sc=k)) if k in scenarios else None for k in range(1, max(scenarios) + 1)]


def scenario_arg(v):
    """--sc: a scenario number 1..8 or 'all'"""
    if v == 'all':
        return v
    k = int(v)
    if not 1 <= k <= 8:
        raise argparse.ArgumentTypeError("--sc must be 1..8 or 'all', got %r" % (v,))
    return k


def main(args, solver=None):
    """`solver`: any object with the BatchSolver methods (default: a BatchSolver made here, d_min = 0 for OBCA); with
    `--sc all` and a `{sc}` weights path it gets a per-problem `net_idx` keyword (its network bank).
    Returns (run directory, summary) -- with `--sc all`, a list of run directories, one per scenario."""
    seed = 2026
    ca_type = getattr(args, 'ca_type', 'circle')
    if ca_type not in ('circle', 'obca'):
        raise ValueError("ca_type must be 'circle' or 'obca', got %r" % (ca_type,))
    policy_config = dict(POLICY_CONFIG, collision_avoidance_type=ca_type)
    N, dt = POLICY_CONFIG['N'], POLICY_CONFIG['dt']
    T = getattr(args, 'steps', None) or 150                                                # T_sim / dt, evaluate.py:84-85
    timenow = datetime.datetime.now().strftime("%Y%m%d_%H%M%S")
    scenarios = list(range(1, 9)) if args.sc == 'all' else [args.sc]
    run_dirs = {k: os.path.join(args.save_dir, '%s_sc%d_seed%d_%s' % (args.eval_mode, k, seed, timenow)) for k in scenarios}
    gt = args.eval_mode == 'gt_mpc'
    bank = gt and len(scenarios) > 1 and '{sc}' in (args.nn_weights or '')    # network k - 1 for scenario k
    own = solver is None
    if own:
        from .planner import BatchSolver
        mlp = networks(args.nn_weights, scenarios) if gt else None
        solver = BatchSolver(N=N, dt=dt, mlp=mlp, **(dict(d_min=0.0) if ca_type == 'obca' else {}))
    variants = [(r, o) for r in range(4) for o in range(2)] if args.all_variants else [(args.rotation, args.order)]
    summary = []
    for it in range(args.num_samples):
        all_specs = episode.reference_episode_specs(scenarios=scenarios, sample=it, seed=seed)
        specs = [all_specs[8 * j + r * 2 + o] for j in range(len(scenarios)) for r, o in variants]
        loop = episode.run_closed_loop_device if getattr(args, 'device_loop', False) else episode.run_closed_loop
        kw = dict(net_idx=np.array([sp.scenario - 1 for sp in specs])) if bank else {}
        res = loop(solver, specs, steps=T, N=N, record_latency=True, mode=args.eval_mode, ca_type=ca_type, **kw)
        for e, sp in enumerate(specs):
            run_dir = run_dirs[scenarios[e // len(variants)]]
            starts = [G.frenet2global(sp.s0[i], sp.routes[i]) for i in range(2)]
            refs = [RT.reference_dict(sp.routes[i], starts[i][0], starts[i][1], n=T) for i in range(2)]
            goals = np.array([[G.goal_pose(r[1])[0] for r in sp.routes], [G.goal_pose(r[1])[1] for r in sp.routes]])
            agents = [{'type': 'CAV', 'state': dict(x=starts[i][0], y=starts[i][1], heading=starts[i][2], v=0.0)} for i in range(2)]
            default = [{'type': 'CAV', 'state': dict(zip(('x', 'y', 'heading'), G.start_pose(r[0])), v=0.0)} for r in sp.routes]
            times = [[1e-3 * ms for ms in res.step_latency_ms]] * 2          # both vehicles are solved in one batched call
            sub = results.write_episode(run_dir, args.eval_mode, res.z_cl[e], res.u_cl[e], res.solved[e], res.deadlock[e],
                                        times, N=N, refs=refs, initial_agents=agents, initial_default=default,
                                        routes=sp.routes, goals=goals, policy_config=policy_config)
            summary.append(dict(sample=it, **(dict(scenario=sp.scenario) if args.sc == 'all' else {}), routes=sp.routes, deadlock=bool(res.deadlock[e]), collision=bool(res.collision[e]),
                                goal=[bool(g) for g in res.goal[e]], infeasible=[int(n) for n in res.num_infeasible[e]],
                                min_distance=float(res.min_distance[e])))
            print("sample %d routes %s: deadlock %s, goals %s, failed solves %s, min distance %.2f m -> %s"
                  % (it, sp.routes, res.deadlock[e], list(res.goal[e]), list(res.num_infeasible[e]), res.min_distance[e], sub))
    if own:
        solver.close()
    return (list(run_dirs.values()) if args.sc == 'all' else run_dirs[args.sc]), summary


def build_parser():
    p = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    p.add_argument('--save_dir', type=str, required=True)
    p.add_argument('--num_samples', type=int, default=1)
    p.add_argument('--eval_mode', type=str, required=True, choices=['mpc', 'gt_mpc'])
    p.add_argument('--sc', type=scenario_arg, default=1, help="scenario 1..8, or 'all': every scenario in one loop")
    p.add_argument('--rotation', type=int, default=0, choices=range(4))
    p.add_argument('--order', type=int, default=0, choices=range(2))
    p.add_argument('--all_variants', action='store_true')
    p.add_argument('--nn_weights', type=str, default=None,
                   help="gt_mpc value network(s), .npz; '{sc}' in the path is replaced by the scenario number")
    p.add_argument('--steps', type=int, default=150, help='closed-loop steps (the reference simulates 15 s = 150)')
    p.add_argument('--device_loop', action='store_true', help='run the per-timestep glue on the GPU as well (igt_episode_run_host)')
    p.add_argument('--ca_type', type=str, default='circle', choices=['circle', 'obca'],
                   help="collision avoidance (mpc.yaml collision_avoidance_type): 5.6 m circles or OBCA rectangles with d_min = 0")
    return p


if __name__ == '__main__':
    a = build_parser().parse_args()
    if a.eval_mode == 'gt_mpc' and not a.nn_weights:
        raise SystemExit("--eval_mode gt_mpc needs --nn_weights FILE.npz")
    main(a)
