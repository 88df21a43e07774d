#!/usr/bin/env python
"""Timing of predict_and_cost with the neural predictor: the gradient (cps_plan_cost_grad, net_grad_kernel), the forward-only
cost (cps_plan_cost) and optimizer_rpgd_b200.step host -> host, beside the same gradient taken by torch autograd on the same
GPU through the float32 torch restatement (oracle/net_grad.py) -- what a user without the CUDA adjoint would run.
Configurations: the shipped RPGD size (16 plans x 35 steps, 4 Adam steps per solve) with the reference's shipped network size
(GRU 2 x 32) and with GRU 2 x 64; 2000 x 50 with GRU 2 x 64 and Dense 2 x 32.  Weights and normalisation: tests/golden."""
import os
import subprocess
import sys
import time
from types import SimpleNamespace

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

from cartpolesimulation_b200 import _lib as L                              # noqa: E402
from cartpolesimulation_b200.optimizer_forward_b200 import optimizer_rpgd_b200   # noqa: E402
from oracle import net_grad as NG                                           # noqa: E402
from oracle import oracle as O                                              # noqa: E402
from tests.netutil import net_spec_from_golden                              # noqa: E402
from tests.parity import load_golden                                        # noqa: E402

NETS = {"GRU 2x32": "net_GRU_6IN_32H1_32H2_5OUT_0", "GRU 2x64": "net_GRU_6IN_64H1_64H2_5OUT_0",
        "Dense 2x32": "net_Dense_6IN_32H1_32H2_5OUT_0"}
CONFIGS = [("GRU 2x32", 16, 35), ("GRU 2x64", 16, 35), ("GRU 2x64", 2000, 50), ("Dense 2x32", 2000, 50)]
COST = "quadratic_boundary_grad_minimal"


def stream_time(fn, reps=20, rounds=15):
    """Median over `rounds` of the device time per call, CUDA events around `reps` back-to-back calls."""
    ts = []
    for _ in range(rounds):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) / reps)
    return float(np.median(ts))


def main():
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                         text=True).stdout.strip())
    a = np.pi - 0.3
    s = np.array([a, 0.2, np.cos(a), np.sin(a), 0.02, 0.0], np.float32)
    lim = (np.array([-1.0], np.float32), np.array([1.0], np.float32))
    for net, K, T in CONFIGS:
        z, _ = load_golden(NETS[net])
        sp = net_spec_from_golden(z)
        spec = dict(sp, weights=O.pack_net_weights(sp["net_type"], sp["layers"], sp["out_layer"]))
        opt = optimizer_rpgd_b200(predictor=SimpleNamespace(predictor_type="neural", net_spec=spec), cost_function=COST,
                                  control_limits=lim, seed=1, mpc_horizon=T, num_rollouts=K, device=0, outer_its=4)
        opt.configure(num_states=6, num_control_inputs=1, dt=0.02, predictor_specification="neural")
        for _ in range(20):
            opt.step(s)
        lat = []
        for _ in range(200):
            t0 = time.perf_counter()
            opt.step(s)
            lat.append((time.perf_counter() - t0) * 1e3)
        eng = opt.engine
        Q = torch.zeros((K, T), device=opt.device).uniform_(-0.5, 0.5)
        s_dev = torch.from_numpy(s).to(opt.device)
        g = stream_time(lambda: eng.plan_cost_grad(s_dev, Q))
        f = stream_time(lambda: eng.plan_cost(s_dev, Q, L.ROLLOUT_MAJOR, 0.0))

        def autograd():
            Qt = Q.clone().requires_grad_(True)
            J = NG.plan_cost(tsp, COST, s_t, Qt, dtype=torch.float32)
            return torch.autograd.grad(J.sum(), Qt)[0]
        # the restatement on the GPU: weights / normalisation as float32 CUDA tensors
        dev = opt.device
        cu = lambda v: torch.as_tensor(np.asarray(v, np.float32), device=dev)   # noqa: E731
        tsp = dict(sp, layers=[tuple(cu(w) for w in lay) for lay in sp["layers"]],
                   out_layer=tuple(cu(w) for w in sp["out_layer"]), norm_a=cu(sp["norm_a"]), norm_b=cu(sp["norm_b"]),
                   denorm_A=cu(sp["denorm_A"]), denorm_B=cu(sp["denorm_B"]))
        s_t = s_dev
        Ga = autograd()
        Gk = eng.plan_cost_grad(s_dev, Q)[1]
        agree = float((Ga - Gk).abs().max() / Gk.abs().max())
        ag = stream_time(autograd, reps=3, rounds=7)
        print(f"{net} K={K} T={T}: gradient {g * 1e3:.1f} us, forward-only plan_cost {f * 1e3:.1f} us (ratio {g / f:.2f}); "
              f"torch autograd (float32, same GPU) {ag * 1e3:.1f} us ({ag / g:.1f}x the kernel; max |G diff| / max |G| "
              f"{agree:.1e}); optimizer_rpgd_b200.step (4 Adam steps) median {np.median(lat):.3f} ms p99 "
              f"{np.percentile(lat, 99):.3f} ms")
        eng.close()


if __name__ == "__main__":
    main()
