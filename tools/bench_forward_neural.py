#!/usr/bin/env python
"""Timing of random action, CEM and CEM-GMM on the neural predictor (GRU 2 x 32, the shipped network, and GRU 2 x 64 from
tests/golden): single solves host -> host (Engine.*_host: state in, u out, median and p99 over many solves) at the
drop-ins' shipped sizes -- CEM and CEM-GMM 200 plans x 35 steps x 3 iterations (best_k 40), random action 640 x 35 --
and the fleets per period and per experiment-period at E in {1024, 8192} (Philox draws, records on).  Baseline, same
process: the same CEM solve restated in float32 torch (oracle/net_grad.predict + stage_costs for the costs, torch.sort
for the elites; weights uploaded once), what a user would run without these kernels.  Prints the GPU's name, power
limit and max SM clock.

    python tools/bench_forward_neural.py [--solves 400] [--periods 20] [--out FILE]
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

from cartpolesimulation_b200 import _lib as L                                     # noqa: E402
from cartpolesimulation_b200.core import Engine                                   # noqa: E402
from cartpolesimulation_b200.fleet import CemFleet, CemGmmFleet, RandomActionFleet, make_experiments   # noqa: E402
from oracle import net_grad as NG                                                 # noqa: E402
from oracle import oracle as O                                                    # noqa: E402
from tests.netutil import net_spec_from_golden                                   # noqa: E402
from tests.parity import load_golden                                              # noqa: E402

COST, T, ITS, BEST_K = "quadratic_boundary_grad_minimal", 35, 3, 40
NETS = {"GRU 2x32": "net_GRU_6IN_32H1_32H2_5OUT_0", "GRU 2x64": "net_GRU_6IN_64H1_64H2_5OUT_0"}


def spec(name):
    sp = net_spec_from_golden(load_golden(NETS[name])[0])
    d = dict(sp)
    d["weights"] = O.pack_net_weights(sp["net_type"], sp["layers"], sp["out_layer"])
    return sp, d


def pct(x):
    x = np.sort(np.asarray(x) * 1e3)
    return f"median {np.median(x):8.3f} ms  p99 {x[int(0.99 * (len(x) - 1))]:8.3f} ms"


def solves(name, n, lines):
    sp, d = spec(name)
    s = np.array([np.pi - 0.1, 0.0, np.cos(np.pi - 0.1), np.sin(np.pi - 0.1), 0.0, 0.0], np.float32)
    g = torch.Generator(device="cuda").manual_seed(0)
    for kind, K in (("CEM", 200), ("CEM-GMM", 200), ("random action", 640)):
        eng = Engine(K, T, integrator="neural", cost=COST, device=0)
        eng.net_load(d)
        eng.set_mppi_params(lo=-1.0, hi=1.0)
        if kind == "CEM":
            eng.cem_configure(BEST_K, 0.5, 0.01)
            eps = torch.randn((ITS, T, K), device="cuda", generator=g)
            call = lambda: eng.cem_step_host(s, eps, L.TIME_MAJOR, 0.0)
        elif kind == "CEM-GMM":
            eng.cem_gmm_configure(BEST_K, 0.5, 0.01)
            eps = torch.randn((ITS, 2, T, K), device="cuda", generator=g)
            u01 = torch.rand((ITS, T, K), device="cuda", generator=g)
            call = lambda: eng.cem_gmm_step_host(s, eps, u01, L.TIME_MAJOR, 0.0)
        else:
            Q = torch.rand((T, K), device="cuda", generator=g) * 2 - 1
            call = lambda: eng.plan_random_action_host(s, Q, L.TIME_MAJOR, 0.0)
        for _ in range(20):
            call()
        n0 = eng.launch_count()
        call()
        per = eng.launch_count() - n0
        ts = []
        for _ in range(n):
            t0 = time.perf_counter()
            call()
            ts.append(time.perf_counter() - t0)
        lines.append(f"{name:9s} {kind:14s} K={K:4d} T={T}  host->host {pct(ts)}  ({per} launches per solve)")
    # float32 torch restatement of the CEM solve, the baseline
    def dev(a):   # the weights go to the device once, so the timed loop holds the solve only
        return torch.as_tensor(np.asarray(a), dtype=torch.float32, device="cuda")
    sp32 = dict(sp, layers=[tuple(dev(a) for a in lay) for lay in sp["layers"]], out_layer=tuple(dev(a) for a in sp["out_layer"]),
                **{k: dev(sp[k]) for k in ("norm_a", "norm_b", "denorm_A", "denorm_B")})
    K = 200
    s_t = torch.from_numpy(s).cuda()
    h0 = torch.zeros(sum(sp["hsz"]), device="cuda", dtype=torch.float32)

    def torch_cem():
        mu, sd = torch.zeros(T, device="cuda"), torch.full((T,), 0.5, device="cuda")
        for _ in range(ITS):
            Q = (mu + torch.randn((K, T), device="cuda", generator=g) * sd).clamp(-1, 1)
            traj = NG.predict(sp32, s_t, Q, h0, dtype=torch.float32)
            J = NG.stage_costs(COST, traj, Q, 0.0).sum(dim=1) / (T + 1)
            el = Q[torch.sort(J, stable=True).indices[:BEST_K]]
            mu, sd = el.mean(0), el.std(0, unbiased=False)
        return float(el[0, 0])
    for _ in range(5):
        torch_cem()
    ts = []
    for _ in range(max(20, n // 10)):
        t0 = time.perf_counter()
        torch_cem()
        ts.append(time.perf_counter() - t0)
    lines.append(f"{name:9s} {'CEM (torch fp32)':14s} K={K:4d} T={T}  host->host {pct(ts)}  (baseline)")


def fleets(E, P, lines):
    _, d = spec("GRU 2x32")
    for kind, cls, K, kw in (("CEM", CemFleet, 200, dict(cem_outer_it=ITS, cem_best_k=BEST_K)),
                             ("CEM-GMM", CemGmmFleet, 200, dict(cem_outer_it=ITS, cem_best_k=BEST_K)),
                             ("random action", RandomActionFleet, 640, {})):
        fl = cls(E, num_rollouts=K, mpc_horizon=T, cost=COST, integrator="neural", network=d, noise="philox", seed=0,
                 device=0, **kw)
        s0, tp, te = make_experiments(E, 2 * P + 2, seed=0)
        fl.reset(s0)
        d_tp, d_te = torch.from_numpy(tp).cuda(), torch.from_numpy(te).cuda()
        rec = torch.zeros((P, E, 16), device="cuda")
        fl.run(2, d_tp[:2].contiguous(), d_te[:2].contiguous(), record=torch.zeros((2, E, 16), device="cuda"))
        torch.cuda.synchronize()
        n0 = fl.engine.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fl.run(P, d_tp[2:2 + P].contiguous(), d_te[2:2 + P].contiguous(), record=rec)
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1) / P
        lines.append(f"fleet GRU 2x32 {kind:14s} K={K:4d} E={E:5d}  {ms:8.3f} ms per period  "
                     f"{ms * 1e3 / E:7.3f} us per experiment-period  ({(fl.engine.launch_count() - n0) // P} launches per period)")
        fl.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--solves", type=int, default=400)
    ap.add_argument("--periods", type=int, default=20)
    ap.add_argument("--experiments", type=int, nargs="+", default=[1024, 8192])
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    lines = [f"GPU: {q}"]
    for name in NETS:
        solves(name, a.solves, lines)
    for E in a.experiments:
        fleets(E, a.periods, lines)
    out = "\n".join(lines)
    print(out)
    if a.out:
        with open(a.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
