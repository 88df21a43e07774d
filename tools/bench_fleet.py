#!/usr/bin/env python
"""Timing of the closed-loop fleet (cps_fleet_run: E experiments x (MPPI solve + plant period) per launch) -- the ncu
target for fleet_kernel (BASELINE.json configs[4]).

--network runs the fleet on the neural predictor instead: a seeded network of the given shape (neural.synthetic_net_spec;
GRU 2 x 32 is the reference's shipped predictor) at E = 1024 and 8192, K = 2000, T = 50, Philox draws, records on.  It
reports the device time per period and per experiment-period, launches per period, the kernel and its rollouts per CTA,
and the device memory the fleet's creation took; beside them, in the same process and on the same network, one experiment
after another: Engine.mppi_step in-stream (device events around consecutive solves) and optimizer_mppi_b200.step
(host -> host).

    python tools/bench_fleet.py [--E 1024 --K 2000 --T 50 --periods 10]
    python tools/bench_fleet.py --network {gru32,gru64,dense32} [--experiments 1024 8192] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from types import SimpleNamespace

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

COST = "quadratic_boundary_grad_minimal"
NETWORKS = {"gru32": ("GRU", (32, 32)), "gru64": ("GRU", (64, 64)), "dense32": ("Dense", (32, 32))}


def neural(args):
    import numpy as np
    import torch
    from cartpolesimulation_b200 import _lib as L
    from cartpolesimulation_b200.core import Engine
    from cartpolesimulation_b200.fleet import DataGenConfig, Fleet, make_experiments
    from cartpolesimulation_b200.neural import synthetic_net_spec
    from cartpolesimulation_b200.optimizer_mppi_b200 import optimizer_mppi_b200
    if not torch.cuda.is_available():
        raise SystemExit("bench_fleet.py --network measures on a CUDA device; none found")
    lines = [subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                            text=True).stdout.strip()]
    K, T, P, R, W = args.K, args.T, args.periods, args.rounds, args.warmup
    ntype, hsz = NETWORKS[args.network]
    spec = synthetic_net_spec(hsz, ntype, seed=0)
    torch.cuda.init()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    lines.append(f"# tools/bench_fleet.py --network {args.network}: {ntype} {' x '.join(map(str, hsz))} (seeded synthetic "
                 f"weights), K = {K}, T = {T}, {COST}, Philox draws, records on; device time per period = CUDA events around "
                 f"{P} periods (one cps_fleet_step call), median of {R} rounds after {W} warm-up periods")
    per_exp = {}
    total = W + R * P
    cfg = DataGenConfig(length_of_experiment=total * 0.02)
    for E in args.experiments:
        s0, tp, te = make_experiments(E, total, cfg, seed=0)
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info(0)[0]
        fl = Fleet(E, K, T, cost=COST, noise="philox", seed=0, device=0, integrator="neural", network=spec)
        torch.cuda.synchronize()
        held = free0 - torch.cuda.mem_get_info(0)[0]
        fl.reset(s0)
        d_tp, d_te = torch.from_numpy(tp).cuda(), torch.from_numpy(te).cuda()
        rec = torch.zeros((max(P, W), E, 16), device="cuda")
        fl.run(W, d_tp[:W].contiguous(), d_te[:W].contiguous(), None, rec[:W])
        torch.cuda.synchronize()
        n0 = fl.engine.launch_count()
        ms = []
        for r in range(R):
            a, b = W + r * P, W + (r + 1) * P
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fl.run(P, d_tp[a:b].contiguous(), d_te[a:b].contiguous(), None, rec[:P])
            e1.record()
            e1.synchronize()
            ms.append(e0.elapsed_time(e1) / P)
        launches = (fl.engine.launch_count() - n0) / (R * P)
        assert np.all(np.isfinite(rec.cpu().numpy())), "non-finite record entries"
        kernel = fl.engine.net_last_kernel()
        if kernel == "tensor":
            rows = int(os.environ.get("CPS_TC_ROWS", 0)) or (32 if E * K <= 32 * sms else 64 if E * K <= 64 * sms else 128)
            tiling = f"net_tc_kernel, {rows} live rollouts per CTA, grid {(K + rows - 1) // rows} x {E}"
        else:
            rows = 32 if K > 148 * 16 else 16
            tiling = f"net_kernel (FP32), R = {rows} rollouts per CTA, grid {(K + rows - 1) // rows} x {E}"
        per = float(np.median(ms))
        per_exp[E] = per / E * 1e3
        lines.append(f"fleet E = {E}: {per:.3f} ms per period (min {min(ms):.3f}, max {max(ms):.3f}); {per_exp[E]:.3f} us per "
                     f"experiment-period; {launches:.1f} launches per period; {tiling}; device memory taken by creating the "
                     f"fleet (cudaMemGetInfo before / after, engine and network included): {held / 1e6:.1f} MB")
        fl.close()
        del fl, rec
        torch.cuda.empty_cache()

    # one experiment after another on the same network: Engine.mppi_step in-stream
    eng = Engine(K, T, integrator="neural", cost=COST, device=0)
    eng.net_load(spec)
    noise = torch.randn((eng.n_ind, K), device="cuda")
    s = torch.from_numpy(s0[0]).cuda()
    for _ in range(20):
        eng.mppi_step(s, noise, L.TIME_MAJOR, 0.0)
    torch.cuda.synchronize()
    n = 200
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        eng.mppi_step(s, noise, L.TIME_MAJOR, 0.0)
    e1.record()
    e1.synchronize()
    step_us = e0.elapsed_time(e1) / n * 1e3
    lines.append(f"Engine.mppi_step in-stream ({n} consecutive solves, {eng.net_last_kernel()} kernel): {step_us:.1f} us per "
                 f"solve; fleet per experiment-period: " +
                 ", ".join(f"E = {E} {v:.2f} us ({step_us / v:.1f}x fewer)" for E, v in per_exp.items()))
    # optimizer_mppi_b200.step, host -> host
    lim = (np.array([-1.0], np.float32), np.array([1.0], np.float32))
    opt = optimizer_mppi_b200(predictor=SimpleNamespace(predictor_type="neural", net_spec=spec), cost_function=COST,
                              control_limits=lim, seed=1, mpc_horizon=T, num_rollouts=K, device=0)
    opt.configure(num_states=6, num_control_inputs=1, dt=0.02, predictor_specification="neural")
    for i in range(20):
        opt.step(s0[i % len(s0)])
    ts = []
    for i in range(200):
        t = time.perf_counter()
        opt.step(s0[i % len(s0)])
        ts.append(time.perf_counter() - t)
    solve = float(np.median(ts)) * 1e3
    lines.append(f"optimizer_mppi_b200.step, host -> host (200 solves): median {solve * 1e3:.1f} us per solve, p99 "
                 f"{np.percentile(ts, 99) * 1e6:.1f} us")
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write(text + "\n\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--E", type=int, default=1024)
    ap.add_argument("--K", type=int, default=2000)
    ap.add_argument("--T", type=int, default=50)
    ap.add_argument("--periods", type=int, default=10)
    ap.add_argument("--network", choices=list(NETWORKS), default=None,
                    help="the neural predictor with a seeded network of this shape (default: predictor ODE)")
    ap.add_argument("--experiments", type=int, nargs="+", default=[1024, 8192], help="--network: fleet sizes")
    ap.add_argument("--rounds", type=int, default=5, help="--network: timed rounds")
    ap.add_argument("--warmup", type=int, default=3, help="--network: periods run before timing")
    ap.add_argument("--out", default=None, help="--network: append the report to this file")
    args = ap.parse_args()
    if args.network:
        if args.periods == 10:
            args.periods = 5
        neural(args)
        return
    import bench
    print(json.dumps(bench.fleet_bench(0, E_total=args.E, periods=args.periods, K=args.K, T=args.T)))


if __name__ == "__main__":
    main()
