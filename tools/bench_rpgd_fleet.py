#!/usr/bin/env python
"""Timing of the RPGD fleet (cps_rpgd_fleet_step, fleet.RpgdFleet) at BASELINE configs[4]'s count: E = 8192 closed-loop
experiments at the shipped RPGD size (16 plans x 35 steps, 4 Adam steps per solve, resampling every 10 solves), targets
from make_experiments, Philox draws, records on.  Beside it, in the same process, optimizer_rpgd_b200.step (host -> host,
one experiment after another) on a sample of the same experiments: what driving the reference's default controller one
experiment at a time costs here.  --network runs both on the neural predictor instead of predictor "ODE": a seeded network
of the shipped architecture (neural.synthetic_net_spec; GRU 2 x 32 is the reference's default predictor), and reports the
adjoint's workspace beside the times.

    python tools/bench_rpgd_fleet.py [--experiments 8192] [--periods 50] [--network {gru32,gru64,dense32}] [--out FILE]
"""
import argparse
import os
import subprocess
import sys
import time
from types import SimpleNamespace

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

from cartpolesimulation_b200.fleet import DataGenConfig, RpgdFleet, make_experiments   # noqa: E402
from cartpolesimulation_b200.neural import synthetic_net_spec                         # noqa: E402
from cartpolesimulation_b200.optimizer_forward_b200 import optimizer_rpgd_b200         # noqa: E402

COST = "quadratic_boundary_grad_minimal"
NETWORKS = {"gru32": ("GRU", (32, 32)), "gru64": ("GRU", (64, 64)), "dense32": ("Dense", (32, 32))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--experiments", type=int, default=8192)
    ap.add_argument("--periods", type=int, default=50, help="periods per timed round")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=12, help="periods run before timing (covers a resampling solve)")
    ap.add_argument("--sample", type=int, default=32, help="experiments solved one by one with optimizer_rpgd_b200")
    ap.add_argument("--network", choices=list(NETWORKS), default=None,
                    help="the neural predictor with a seeded network of this shape (default: predictor ODE)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_rpgd_fleet.py measures on a CUDA device; none found")
    lines = [subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                            text=True).stdout.strip()]
    E, P, R, W = args.experiments, args.periods, args.rounds, args.warmup
    total = W + R * P
    cfg = DataGenConfig(length_of_experiment=total * 0.02)   # target traces over the simulated span
    t0 = time.perf_counter()
    s0, tp, te = make_experiments(E, total, cfg, seed=0)
    t_tables = time.perf_counter() - t0
    spec = None
    if args.network:
        ntype, hsz = NETWORKS[args.network]
        spec = synthetic_net_spec(hsz, ntype, seed=0)
        torch.cuda.init()
        free0 = torch.cuda.mem_get_info(0)[0]
        fl = RpgdFleet(E, noise="philox", seed=0, device=0, integrator="neural", network=spec)
        torch.cuda.synchronize()
        held = free0 - torch.cuda.mem_get_info(0)[0]
    else:
        fl = RpgdFleet(E, noise="philox", seed=0, device=0)
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
    dt_control = cfg.dt_control
    net = f", neural predictor {args.network} (seeded synthetic weights)" if args.network else ""
    lines.append(f"# tools/bench_rpgd_fleet.py: E = {E}, K = 16, T = 35, outer_its = 4, resamp_per = 10, {COST}{net}, Philox draws, "
                 f"records on; device time per period = CUDA events around {P} periods (one cps_rpgd_fleet_step call), "
                 f"median of {R} rounds after {W} warm-up periods")
    lines.append(f"RPGD fleet: {per:.3f} ms per period (min {min(ms):.3f}, max {max(ms):.3f}); {per / E * 1e3:.3f} us per "
                 f"experiment-period; {E / per * 1e3:.4g} experiment-periods/s; {E * dt_control / (per * 1e-3):.4g} simulated "
                 f"seconds per wall second; {launches:.1f} launches per period")
    if spec is not None:
        # the adjoint's forward records: (T + 1) htot R + 16 T R floats per CTA of R = 16 plans; at K = 16 one CTA per experiment
        ws = 4 * ((35 + 1) * sum(spec["hsz"]) * 16 + 16 * 35 * 16) * E
        lines.append(f"workspace of the network adjoint: {ws} bytes ({ws / 1e9:.3f} GB; E CTAs x ((T + 1) htot + 16 T) x 16 "
                     f"floats); device memory taken by creating the fleet (engine, network, plans, workspace; "
                     f"cudaMemGetInfo before / after): {held / 1e9:.3f} GB")

    # baseline: optimizer_rpgd_b200.step, one experiment after another (host -> host; each step synchronises)
    lim = (np.array([-1.0], np.float32), np.array([1.0], np.float32))
    pred = SimpleNamespace(predictor_type="neural", net_spec=spec) if spec is not None else "ODE"
    opt = optimizer_rpgd_b200(predictor=pred, cost_function=COST, control_limits=lim, seed=1, mpc_horizon=35,
                              num_rollouts=16, device=0)
    opt.configure(num_states=6, num_control_inputs=1, dt=0.02, predictor_specification="neural" if spec is not None else "ODE")
    states = fl.states()
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
    lines.append(f"optimizer_rpgd_b200.step, one experiment after another ({args.sample} experiments x 5, host -> host): "
                 f"median {solve:.3f} ms per solve, p99 {np.percentile(ts, 99) * 1e3:.3f} ms; {E} experiments would need "
                 f"{solve * E:.1f} ms per period, {solve * E / per:.0f}x the fleet's device time per period")
    lines.append(f"(host-side target tables for {E} experiments x {total} periods: {t_tables:.1f} s, not timed above)")
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
