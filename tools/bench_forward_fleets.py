#!/usr/bin/env python
"""Timing of the CEM-GMM and random-action fleets (cps_cem_gmm_fleet_step / fleet.CemGmmFleet at the shipped
optimizer_cem_gmm_tf size, 200 plans x 35 steps, 3 outer iterations, best_k 40; cps_random_action_fleet_step /
fleet.RandomActionFleet at 640 plans x 35 steps, the random-action size bench.py times), E in {1024, 8192} closed-loop
experiments, targets from make_experiments, Philox draws, records on.  Beside each, in the same process: one
cps_cem_gmm_step / cps_plan_random_action of the same size in-stream (device time per solve, many solves between two CUDA
events), and optimizer_cem_gmm_b200.step / optimizer_random_action_b200.step host -> host, one experiment after another --
what driving the reference's controller one experiment at a time costs here.

    python tools/bench_forward_fleets.py [--experiments 1024 8192] [--periods 50] [--out FILE]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

from cartpolesimulation_b200 import _lib as L                                          # noqa: E402
from cartpolesimulation_b200.core import Engine                                        # noqa: E402
from cartpolesimulation_b200.fleet import CemGmmFleet, DataGenConfig, RandomActionFleet, make_experiments   # noqa: E402
from cartpolesimulation_b200.optimizer_forward_b200 import (optimizer_cem_gmm_b200,                          # noqa: E402
                                                             optimizer_random_action_b200)

COST, T, ITS, BEST_K = "quadratic_boundary_grad_minimal", 35, 3, 40
KINDS = {   # name: (K, fleet class and keywords, optimizer class and keywords)
    "CEM-GMM": (200, CemGmmFleet, dict(cem_outer_it=ITS, cem_best_k=BEST_K), optimizer_cem_gmm_b200,
                dict(cem_outer_it=ITS, cem_best_k=BEST_K)),
    "random action": (640, RandomActionFleet, {}, optimizer_random_action_b200, {}),
}


def fleet_time(kind, E, P, R, W, lines):
    K, cls, kw = KINDS[kind][:3]
    total = W + R * P
    cfg = DataGenConfig(length_of_experiment=total * 0.02)   # target traces over the simulated span
    t0 = time.perf_counter()
    s0, tp, te = make_experiments(E, total, cfg, seed=0)
    t_tables = time.perf_counter() - t0
    fl = cls(E, num_rollouts=K, mpc_horizon=T, cost=COST, noise="philox", seed=0, device=0, **kw)
    fl.reset(s0)
    d_tp, d_te = torch.from_numpy(tp).cuda(), torch.from_numpy(te).cuda()
    rec = torch.zeros((P, E, 16), device="cuda")
    fl.run(W, d_tp[:W].contiguous(), d_te[:W].contiguous(), record=torch.zeros((W, E, 16), device="cuda"))
    torch.cuda.synchronize()
    n0 = fl.engine.launch_count()
    ms = []
    for r in range(R):
        a, b = W + r * P, W + (r + 1) * P
        tpr, ter = d_tp[a:b].contiguous(), d_te[a:b].contiguous()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fl.run(P, tpr, ter, record=rec)
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1) / P)
    launches = (fl.engine.launch_count() - n0) / (R * P)
    r_np = rec.cpu().numpy()
    assert np.all(np.isfinite(r_np)), "non-finite record entries"
    per = float(np.median(ms))
    lines.append(f"{kind} fleet E = {E}: {per:.3f} ms per period (min {min(ms):.3f}, max {max(ms):.3f}); {per / E * 1e3:.3f} us per "
                 f"experiment-period; {E / per * 1e3:.4g} experiment-periods/s; {E * cfg.dt_control / (per * 1e-3):.4g} "
                 f"simulated seconds per wall second; {launches:.1f} launches per period (host-side target tables: "
                 f"{t_tables:.1f} s, not timed)")
    states = fl.states()
    fl.close()
    return per, states


def single_time(kind, states, n, lines):
    """One solve in-stream: device time per solve, n solves between two CUDA events, median of 5."""
    K = KINDS[kind][0]
    eng = Engine(K, T, cost=COST, device=0)
    s_dev = torch.from_numpy(states[0]).cuda()
    if kind == "CEM-GMM":
        eng.cem_gmm_configure(BEST_K, 0.5, 0.01)
        eps, u01 = torch.randn((ITS, 2, T, K), device="cuda"), torch.rand((ITS, T, K), device="cuda")
        name = "cps_cem_gmm_step"
        solve = lambda: eng.cem_gmm_step(s_dev, eps, u01, L.TIME_MAJOR)   # noqa: E731
    else:
        Q = torch.rand((T, K), device="cuda") * 2.0 - 1.0
        name = "cps_plan_random_action"
        solve = lambda: eng.plan_random_action(s_dev, Q, L.TIME_MAJOR)   # noqa: E731
    for _ in range(20):
        solve()
    torch.cuda.synchronize()
    single = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            solve()
        e1.record()
        e1.synchronize()
        single.append(e0.elapsed_time(e1) / n)
    one = float(np.median(single))
    lines.append(f"{name} in-stream ({n} solves between two CUDA events, median of 5): {one:.4f} ms per solve")
    return one


def host_time(kind, states, sample, lines):
    """optimizer_*_b200.step, one experiment after another (host -> host; each step synchronises)."""
    K, opt_cls, kw = KINDS[kind][0], KINDS[kind][3], KINDS[kind][4]
    lim = (np.array([-1.0], np.float32), np.array([1.0], np.float32))
    opt = opt_cls(predictor="ODE", cost_function=COST, control_limits=lim, seed=1, mpc_horizon=T, num_rollouts=K, device=0, **kw)
    opt.configure(num_states=6, num_control_inputs=1, dt=0.02, predictor_specification="ODE")
    E = len(states)
    for i in range(20):   # warm-up
        opt.step(states[i % E])
    torch.cuda.synchronize()
    idx = np.linspace(0, E - 1, sample).astype(int)
    ts = []
    for rep in range(5):
        for i in idx:
            t = time.perf_counter()
            opt.step(states[i])
            ts.append(time.perf_counter() - t)
    solve = float(np.median(ts)) * 1e3
    lines.append(f"{opt_cls.__name__}.step, one experiment after another ({sample} experiments x 5, host -> host): "
                 f"median {solve:.3f} ms per solve, p99 {np.percentile(ts, 99) * 1e3:.3f} ms")
    return solve


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--experiments", type=int, nargs="+", default=[1024, 8192])
    ap.add_argument("--periods", type=int, default=50, help="periods per timed round")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=5, help="periods run before timing")
    ap.add_argument("--sample", type=int, default=32, help="experiments solved one by one with the optimizer")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_forward_fleets.py measures on a CUDA device; none found")
    lines = [subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                            text=True).stdout.strip()]
    lines.append(f"# tools/bench_forward_fleets.py: T = {T}, {COST}, CEM-GMM K = {KINDS['CEM-GMM'][0]} with cem_outer_it = "
                 f"{ITS}, cem_best_k = {BEST_K}; random action K = {KINDS['random action'][0]}; Philox draws, records on; "
                 f"device time per period = CUDA events around {args.periods} periods (one _step call), median of "
                 f"{args.rounds} rounds after {args.warmup} warm-up periods")
    for kind in KINDS:
        per, states = {}, None
        for E in args.experiments:
            per[E], states = fleet_time(kind, E, args.periods, args.rounds, args.warmup, lines)
        one = single_time(kind, states, 400, lines)
        for E, p in per.items():
            lines.append(f"  E = {E}: the fleet's device time per experiment-period is {one / (p / E):.0f}x below one "
                         f"in-stream solve")
        solve = host_time(kind, states, args.sample, lines)
        for E, p in per.items():
            lines.append(f"  E = {E}: sequential solves would need {solve * E:.1f} ms per period, {solve * E / p:.0f}x the "
                         f"fleet's device time per period")
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
