#!/usr/bin/env python
"""Timing of the CEM fleet (cps_cem_fleet_step, fleet.CemFleet) at the shipped optimizer_cem_tf size (200 plans x 35 steps,
3 outer iterations, best_k 40), E in {1024, 8192} closed-loop experiments, targets from make_experiments, Philox draws,
records on.  Beside it, in the same process: one cps_cem_step of the same size in-stream (device time per solve, many
solves between two CUDA events), and optimizer_cem_b200.step host -> host, one experiment after another -- what driving
the reference's CEM controller one experiment at a time costs here.

    python tools/bench_cem_fleet.py [--experiments 1024 8192] [--periods 50] [--out FILE]
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
from cartpolesimulation_b200.fleet import CemFleet, DataGenConfig, make_experiments    # noqa: E402
from cartpolesimulation_b200.optimizer_forward_b200 import optimizer_cem_b200          # noqa: E402

COST, K, T, ITS, BEST_K = "quadratic_boundary_grad_minimal", 200, 35, 3, 40


def fleet_time(E, P, R, W, lines):
    total = W + R * P
    cfg = DataGenConfig(length_of_experiment=total * 0.02)   # target traces over the simulated span
    t0 = time.perf_counter()
    s0, tp, te = make_experiments(E, total, cfg, seed=0)
    t_tables = time.perf_counter() - t0
    fl = CemFleet(E, num_rollouts=K, mpc_horizon=T, cem_outer_it=ITS, cem_best_k=BEST_K, cost=COST, noise="philox", seed=0,
                  device=0)
    fl.reset(s0)
    d_tp, d_te = torch.from_numpy(tp).cuda(), torch.from_numpy(te).cuda()
    rec = torch.zeros((P, E, 16), device="cuda")
    fl.run(W, d_tp[:W].contiguous(), d_te[:W].contiguous(), None, torch.zeros((W, E, 16), device="cuda"))
    torch.cuda.synchronize()
    n0 = fl.engine.launch_count()
    ms = []
    for r in range(R):
        a, b = W + r * P, W + (r + 1) * P
        tpr, ter = d_tp[a:b].contiguous(), d_te[a:b].contiguous()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fl.run(P, tpr, ter, None, rec)
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1) / P)
    launches = (fl.engine.launch_count() - n0) / (R * P)
    r_np = rec.cpu().numpy()
    assert np.all(np.isfinite(r_np)), "non-finite record entries"
    per = float(np.median(ms))
    lines.append(f"CEM fleet E = {E}: {per:.3f} ms per period (min {min(ms):.3f}, max {max(ms):.3f}); {per / E * 1e3:.3f} us per "
                 f"experiment-period; {E / per * 1e3:.4g} experiment-periods/s; {E * cfg.dt_control / (per * 1e-3):.4g} "
                 f"simulated seconds per wall second; {launches:.1f} launches per period (host-side target tables: "
                 f"{t_tables:.1f} s, not timed)")
    states = fl.states()
    fl.close()
    return per, states


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--experiments", type=int, nargs="+", default=[1024, 8192])
    ap.add_argument("--periods", type=int, default=50, help="periods per timed round")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=5, help="periods run before timing")
    ap.add_argument("--sample", type=int, default=32, help="experiments solved one by one with optimizer_cem_b200")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_cem_fleet.py measures on a CUDA device; none found")
    lines = [subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                            text=True).stdout.strip()]
    lines.append(f"# tools/bench_cem_fleet.py: K = {K}, T = {T}, cem_outer_it = {ITS}, cem_best_k = {BEST_K}, {COST}, "
                 f"Philox draws, records on; device time per period = CUDA events around {args.periods} periods (one "
                 f"cps_cem_fleet_step call), median of {args.rounds} rounds after {args.warmup} warm-up periods")
    per, states = {}, None
    for E in args.experiments:
        per[E], states = fleet_time(E, args.periods, args.rounds, args.warmup, lines)

    # one cps_cem_step in-stream: device time per solve (the fleet's per-experiment-period time should be below it)
    eng = Engine(K, T, cost=COST, device=0)
    eng.cem_configure(BEST_K, 0.5, 0.01)
    n = 400
    eps = torch.randn((ITS, T, K), device="cuda")
    s_dev = torch.from_numpy(states[0]).cuda()
    for _ in range(20):
        eng.cem_step(s_dev, eps, L.TIME_MAJOR)
    torch.cuda.synchronize()
    single = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            eng.cem_step(s_dev, eps, L.TIME_MAJOR)
        e1.record()
        e1.synchronize()
        single.append(e0.elapsed_time(e1) / n)
    one = float(np.median(single))
    lines.append(f"cps_cem_step in-stream ({n} solves between two CUDA events, median of 5): {one:.4f} ms per solve")
    for E, p in per.items():
        lines.append(f"  E = {E}: the fleet's device time per experiment-period is {one / (p / E):.0f}x below one in-stream solve")

    # baseline: optimizer_cem_b200.step, one experiment after another (host -> host; each step synchronises)
    lim = (np.array([-1.0], np.float32), np.array([1.0], np.float32))
    opt = optimizer_cem_b200(predictor="ODE", cost_function=COST, control_limits=lim, seed=1, mpc_horizon=T, num_rollouts=K,
                             cem_outer_it=ITS, cem_best_k=BEST_K, device=0)
    opt.configure(num_states=6, num_control_inputs=1, dt=0.02, predictor_specification="ODE")
    E = len(states)
    for i in range(20):   # warm-up
        opt.step(states[i % E])
    torch.cuda.synchronize()
    idx = np.linspace(0, E - 1, args.sample).astype(int)
    ts = []
    for rep in range(5):
        for i in idx:
            t = time.perf_counter()
            opt.step(states[i])
            ts.append(time.perf_counter() - t)
    solve = float(np.median(ts)) * 1e3
    lines.append(f"optimizer_cem_b200.step, one experiment after another ({args.sample} experiments x 5, host -> host): "
                 f"median {solve:.3f} ms per solve, p99 {np.percentile(ts, 99) * 1e3:.3f} ms")
    for E, p in per.items():
        lines.append(f"  E = {E}: sequential solves would need {solve * E:.1f} ms per period, {solve * E / p:.0f}x the fleet's "
                     f"device time per period")
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
