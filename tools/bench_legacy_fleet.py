#!/usr/bin/env python
"""Timing of the legacy controller fleet (cps_legacy_fleet_step / fleet.LegacyFleet) at the shipped `mppi-cartpole` size,
3500 rollouts x 35 steps, interpolated sampler, predictor ODE and ODE_v0, E in {1024, 8192} closed-loop experiments,
targets from make_experiments, Philox draws, records on: device time per period and per experiment-period between two
CUDA events.  Beside it, in the same process, controller_mppi_cartpole_b200.step host -> host (its own SFC64 draws and
one legacy_mppi_kernel launch per call), what driving the controller one experiment at a time costs here.  The card name
and power limit are read in the same run.

    python tools/bench_legacy_fleet.py [--experiments 1024 8192] [--periods 20] [--out FILE]
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

from cartpolesimulation_b200.controller_mppi_cartpole_b200 import controller_mppi_cartpole_b200   # noqa: E402
from cartpolesimulation_b200.fleet import DataGenConfig, LegacyFleet, make_experiments               # noqa: E402

K, T = 3500, 35


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as ex:   # noqa: BLE001
        return f"unknown ({ex})"


def fleet_time(predictor, E, P, R, W):
    total = W + R * P
    s0, tp, te = make_experiments(E, total, DataGenConfig(length_of_experiment=total * 0.02), seed=0)
    fl = LegacyFleet(E, dict(predictor_specification=predictor), noise="philox", seed=0, device=0)
    fl.reset(s0)
    d_tp, d_te = torch.from_numpy(tp).cuda(), torch.from_numpy(te).cuda()
    rec = torch.zeros((P, E, 16), device="cuda")
    fl.run(W, d_tp[:W].contiguous(), d_te[:W].contiguous(), record=torch.zeros((W, E, 16), device="cuda"))
    torch.cuda.synchronize()
    n0 = fl.engine.launch_count()
    ms = []
    for r in range(R):
        a, b = W + r * P, W + (r + 1) * P
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fl.run(P, d_tp[a:b].contiguous(), d_te[a:b].contiguous(), record=rec)
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1) / P)
    launches = (fl.engine.launch_count() - n0) / (R * P)
    finite = bool(torch.isfinite(rec).all())
    fl.close()
    return float(np.median(ms)), float(np.min(ms)), launches, finite


def controller_time(predictor, n):
    ctl = controller_mppi_cartpole_b200(dict(predictor_specification=predictor, seed=0), device=0)
    s = np.array([0.1, 0.0, np.cos(0.1), np.sin(0.1), 0.0, 0.0], np.float32)
    for _ in range(5):
        ctl.step(s)
    t0 = time.perf_counter()
    for _ in range(n):
        ctl.step(s)
    return (time.perf_counter() - t0) / n * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--experiments", type=int, nargs="+", default=[1024, 8192])
    ap.add_argument("--periods", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    lines = [f"card (name, power limit, max SM clock): {card()}",
             f"legacy fleet, K = {K}, T = {T}, SAMPLING_TYPE interpolated, Philox draws, records on, "
             f"{a.periods} periods x {a.repeats} repeats after 5 warm-up periods; device time between CUDA events"]
    for predictor in ("ODE", "ODE_v0"):
        host = controller_time(predictor, 50)
        lines.append(f"{predictor}: controller_mppi_cartpole_b200.step host to host {host:.3f} ms per call")
        for E in a.experiments:
            med, best, launches, finite = fleet_time(predictor, E, a.periods, a.repeats, 5)
            per = med / E * 1e3
            rate = E * K * T * 10 / (med * 1e-3)
            lines.append(f"{predictor}: E = {E:5d}  {med:8.3f} ms / period (min {best:.3f})  {per:7.3f} us / experiment-period"
                         f"  {rate:.3e} substeps/s  launches/period {launches:.0f}  records finite {finite}"
                         f"  vs host step x E: {host * E / med:.0f}x")
    text = "\n".join(lines)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
