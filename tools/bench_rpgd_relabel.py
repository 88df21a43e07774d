#!/usr/bin/env python
"""Timing of offline relabelling under RPGD (cps_rpgd_fleet_relabel, RpgdFleet.relabel) at the size of the MPPI relabel
entry (mppi_solve.relabel_256_files): 256 files x 50 rows, at the shipped RPGD configuration (16 plans x 35 steps, 4 Adam
steps per solve, resampling every 10 solves), Philox draws, the row's L fed per row and file (as add_control_along_trajectories
feeds the L column; predictor "ODE" then folds each file's model on the device).  The recordings are 50 closed-loop periods
of an RpgdFleet over the same files, whose device time per period is reported beside the row's.  Then, in the same
process, optimizer_rpgd_b200.step (host -> host) over the rows of one file after another: what relabelling with the
drop-in optimizer costs.  --network gru32 runs everything on a seeded GRU 2 x 32 (neural.synthetic_net_spec; the
reference's default predictor architecture) instead of predictor "ODE".

    python tools/bench_rpgd_relabel.py [--files 256] [--rows 50] [--network gru32] [--out FILE]
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
NETWORKS = {"gru32": ("GRU", (32, 32))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=256)
    ap.add_argument("--rows", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--sample", type=int, default=8, help="files relabelled one by one with optimizer_rpgd_b200")
    ap.add_argument("--network", choices=list(NETWORKS), default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_rpgd_relabel.py measures on a CUDA device; none found")
    lines = [subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                            text=True).stdout.strip()]
    E, R, N = args.files, args.rows, args.rounds
    spec, kw = None, {}
    if args.network:
        ntype, hsz = NETWORKS[args.network]
        spec = synthetic_net_spec(hsz, ntype, seed=0)
        kw = dict(integrator="neural", network=spec)
    cfg = DataGenConfig(length_of_experiment=R * 0.02)
    s0, tp, te = make_experiments(E, R, cfg, seed=0)
    d_tp, d_te = torch.from_numpy(tp).cuda(), torch.from_numpy(te).cuda()
    L = torch.from_numpy(np.random.default_rng(0).uniform(0.25, 0.55, (R, E)).astype(np.float32)).cuda()

    # the recordings: R closed-loop periods, timed as the reference point
    loop = RpgdFleet(E, noise="philox", seed=0, device=0, **kw)
    rec = torch.zeros((R, E, 16), device="cuda")
    loop_ms = []
    for r in range(N + 1):
        loop.reset(s0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loop.run(R, d_tp, d_te, None, rec)
        e1.record()
        e1.synchronize()
        if r:   # the first round warms up
            loop_ms.append(e0.elapsed_time(e1) / R)
    states = rec[:, :, [1, 2, 4, 5, 6, 7]].contiguous()

    rl = RpgdFleet(E, noise="philox", seed=0, device=0, **kw)
    Q = torch.empty((R, E), device="cuda")
    ms = []
    for r in range(N + 1):
        rl.reset(np.zeros((E, 6), np.float32))
        n0 = rl.engine.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rl.relabel(states, d_tp, d_te, L, None, None, Q)
        e1.record()
        e1.synchronize()
        launches = (rl.engine.launch_count() - n0) / R
        if r:
            ms.append(e0.elapsed_time(e1) / R)
    assert torch.isfinite(Q).all(), "non-finite labels"
    per, per_loop = float(np.median(ms)), float(np.median(loop_ms))
    pred = f"neural predictor {args.network} (seeded synthetic weights)" if spec is not None else 'predictor "ODE"'
    lines.append(f"# tools/bench_rpgd_relabel.py: {E} files x {R} rows, K = 16, T = 35, outer_its = 4, resamp_per = 10, {COST}, "
                 f"{pred}, Philox draws, per-row L; device time = CUDA events around {R} rows (one cps_rpgd_fleet_relabel "
                 f"call) / {R} periods (one cps_rpgd_fleet_step call), median of {N} rounds after one warm-up round")
    lines.append(f"RPGD relabelling: {per:.3f} ms per row of all files (min {min(ms):.3f}, max {max(ms):.3f}); "
                 f"{E / per * 1e3:.4g} labels/s; {launches:.1f} launches per row")
    lines.append(f"RPGD fleet, closed loop over the same files: {per_loop:.3f} ms per period (min {min(loop_ms):.3f}, "
                 f"max {max(loop_ms):.3f}); a row costs {per / per_loop:.2f} periods")

    # baseline: optimizer_rpgd_b200.step over the rows of one file after another (host -> host; each step synchronises)
    lim = (np.array([-1.0], np.float32), np.array([1.0], np.float32))
    predictor = SimpleNamespace(predictor_type="neural", net_spec=spec) if spec is not None else "ODE"
    opt = optimizer_rpgd_b200(predictor=predictor, cost_function=COST, control_limits=lim, seed=1, mpc_horizon=35,
                              num_rollouts=16, device=0)
    opt.configure(num_states=6, num_control_inputs=1, dt=0.02, predictor_specification="neural" if spec is not None else "ODE")
    s_host = states.cpu().numpy()
    for r in range(10):   # warm-up
        opt.step(s_host[r, 0])
    torch.cuda.synchronize()
    files = np.linspace(0, E - 1, args.sample).astype(int)
    t = time.perf_counter()
    for f in files:
        opt.optimizer_reset()
        for r in range(R):
            opt.step(s_host[r, f])
    per_file = (time.perf_counter() - t) / len(files) * 1e3
    lines.append(f"optimizer_rpgd_b200.step, the {R} rows of one file after another ({len(files)} files, host -> host): "
                 f"{per_file:.1f} ms per file, {per_file / R:.3f} ms per label; {E} files would take {per_file * E / 1e3:.2f} s, "
                 f"{per_file * E / (per * R):.0f}x the relabelling's device time")
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
