#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native CartPole MPPI rollout path.

Workload (BASELINE.json configs[1]): open-loop batched cartpole_ode explicit-Euler rollouts, 1M cartpoles x 500
integrator substeps (T = 50 control steps x n = 10 substeps of 2 ms, the predictor_ODE_v0 operating point), random
controls, full trajectory materialised as predictor.predict_core returns it.  One "step" = one pass over the batch
= B*T*n state-steps.  N > 1: every rank runs its own batch (weak scaling, no data-path collective).

  python bench.py --gpus N --steps K --warmup W            # ours (CUDA through the C ABI)
  python bench.py --impl reference --gpus N ...            # the reference algorithm's CPU port on the host cores
  python bench.py ... --dump-outputs DIR                   # also write what the last timed pass computed (DIR/*.npy)

Prints ONE JSON line on rank 0.  Also measured inside the same run and attached to the line:
  e2e           same pass through cps_rollout_host with pinned HOST buffers (H2D of s0+Q, D2H of the trajectory)
  roofline      algorithmic FLOPs (32 per state-step, SURVEY.md 8d) / CUDA-event kernel time vs the FP32 peak
                measured in place by cps_measure_peaks; MUFU and HBM views beside it
  cpu_baseline  the oracle (C restatement of the reference, OpenMP over rollouts) on a bounded sample, host cores
  mppi_solve    MPPI solve latency at K=2000, T=50 (BASELINE.json configs[0]/metric second half)
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

FLOP_PER_STATE_STEP = 32.0   # SURVEY.md 8(d) / Appendix A.2: 24 (ODE rhs) + 8 (integrator), FMA = 2
# FMA-pipe lane operations the pair kernel executes per state-step (ncu instruction mix, DESIGN.md 4.5): 29 packed in the
# substep + ~2.7 amortised per-control-step work (packed angle resync: 25 packed + 4 scalar per pair and control step)
FP32_LANE_OPS_PER_STATE_STEP = 31.7
MUFU_PER_STATE_STEP = 3.0    # rcp + sin + cos when the MUFU path is used; 1 (rcp) otherwise
B_DEFAULT, T_DEFAULT, N_SUB, DT = 1 << 20, 50, 10, 0.02
METRIC = "rollout_state_steps_per_sec"
UNIT = "state-steps/s"


def workload_name(B, T):
    return (f"open-loop cartpole_ode explicit-Euler rollouts (predictor_ODE_v0), {B} cartpoles x {T * N_SUB} substeps "
            f"(T={T} x n={N_SUB}, dt={DT}), random controls, trajectory [T+1,6,B] materialised")


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index=0, period=0.05):
        super().__init__(daemon=True)
        self.period, self.stop_flag, self.samples, self.reasons = period, False, [], set()
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def make_inputs(B, T, seed):
    """Synthetic inputs of SURVEY.md 8(d) C2: per-cartpole random state, Q ~ U(-1, 1)."""
    rng = np.random.default_rng(seed)
    ang = rng.uniform(-np.pi, np.pi, B).astype(np.float32)
    s0 = np.stack([ang, rng.uniform(-5, 5, B), np.cos(ang), np.sin(ang), rng.uniform(-0.8 * 0.198, 0.8 * 0.198, B),
                   rng.uniform(-0.5 * 0.198, 0.5 * 0.198, B)], 1).astype(np.float32)
    Q = rng.uniform(-1, 1, (T, B)).astype(np.float32)  # time-major
    return s0, Q


DUMP_TRAJ_BYTES = 48 << 20   # --dump-outputs: trajectories of at most this many bytes (64 MB for everything written)


def dump_index(B, T, seed=0):
    """The cartpoles --dump-outputs writes: a fixed, seeded sample of n of the B (every one when their trajectories fit
    in DUMP_TRAJ_BYTES), sorted."""
    n = int(min(B, max(1, DUMP_TRAJ_BYTES // ((T + 1) * 6 * 4))))
    return np.arange(B) if n == B else np.sort(np.random.default_rng(seed).choice(B, n, replace=False))


def write_dump(out_dir, traj_sample, idx):
    """trajectory.npy = the sampled cartpoles' trajectories ([T+1, 6, n] float32, time-major like the full result);
    cartpole_index.npy = their indices in the batch (float64)."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "trajectory.npy"), np.ascontiguousarray(traj_sample, dtype=np.float32))
    np.save(os.path.join(out_dir, "cartpole_index.npy"), idx.astype(np.float64))


def dump_outputs(out_dir, traj):
    """--dump-outputs: what the timed rollouts returned in their last pass (traj [T+1, 6, B] on the device), so that two
    builds can be compared output for output."""
    import torch
    T1, _, B = traj.shape
    idx = dump_index(B, T1 - 1)
    write_dump(out_dir, traj.index_select(2, torch.from_numpy(idx).to(traj.device)).cpu().numpy(), idx)


def cpu_port_rate(B_sample, T, threads=None, repeats=1, seed=0):
    """state-steps/s of the oracle port (cps_oracle_rollout_v0, OpenMP) on this host."""
    from oracle import oracle as O
    # all host cores unless told otherwise (torchrun exports OMP_NUM_THREADS=1, which is not what a CPU baseline wants)
    O.lib().cps_oracle_set_num_threads(int(threads) if threads else (os.cpu_count() or 1))
    s0, Q = make_inputs(B_sample, T, seed)
    Qr = np.ascontiguousarray(Q.T)
    O.rollout("ODE_v0", s0[:64], Qr[:64], n=N_SUB, dt=DT)  # warm up (thread pool, page faults)
    total = 0.0
    for _ in range(repeats):
        t0 = time.perf_counter()
        O.rollout("ODE_v0", s0, Qr, n=N_SUB, dt=DT)
        total += time.perf_counter() - t0
    return B_sample * T * N_SUB * repeats / total, total, O.lib().cps_oracle_num_threads()


def run_reference(args):
    """--impl reference: the reference's algorithm on the host cores.  The reference is pure Python (numba + numpy)
    and cannot travel to the GPU box, so this is the oracle port (kind "port"), OpenMP over all host threads; each
    step is a bounded sample of the workload (B_sample cartpoles of the 1M)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    T = args.horizon
    cores = os.cpu_count() or 1
    # size the sample for ~2 s per step
    rate, _, threads = cpu_port_rate(4096, T)
    B_sample = int(min(args.batch, max(4096, rate * 2.0 / (T * N_SUB))))
    from oracle import oracle as O
    s0, Q = make_inputs(B_sample, T, 0)
    Qr = np.ascontiguousarray(Q.T)
    for _ in range(args.warmup):
        O.rollout("ODE_v0", s0, Qr, n=N_SUB, dt=DT)
    times = []
    for _ in range(args.steps):
        t1 = time.perf_counter()
        O.rollout("ODE_v0", s0, Qr, n=N_SUB, dt=DT)
        times.append(time.perf_counter() - t1)
    if args.dump_outputs:
        # the timed sample's size depends on the host, so the port rolls out the cartpoles --impl ours dumps, from the
        # inputs --impl ours uses (rank 0): the two arms can be compared output for output
        s0_all, Q_all = make_inputs(args.batch, T, seed=1234)
        idx = dump_index(args.batch, T)
        traj = O.rollout("ODE_v0", s0_all[idx], np.ascontiguousarray(Q_all[:, idx].T), n=N_SUB, dt=DT)   # [n, T+1, 6]
        write_dump(args.dump_outputs, traj.transpose(1, 2, 0), idx)
    total = float(np.sum(times))
    value = B_sample * T * N_SUB * args.steps / total
    sample = f"{B_sample} of {args.batch} cartpoles x {T * N_SUB} substeps per step"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (f64 inside a control step)",
            "data": "synthetic", "config": {"workload": workload_name(args.batch, T), "sample": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                             "host_cores": cores},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def mppi_latency(device, n_calls=1000):
    """MPPI solve latency at K=2000, T=50 through the reference-facing optimizer.step(s): numpy state in, numpy
    control out (the reference's Q_update_time analogue, CartPole/__init__.py:494,521)."""
    import torch
    import cartpolesimulation_b200 as cps
    from cartpolesimulation_b200.optimizer_mppi_b200 import optimizer_mppi_b200
    K, T = 2000, 50
    vp = cps.VariableParameters(target_position=0.0, target_equilibrium=1.0, L=0.395, m_pole=0.087)
    out = {}
    for pred in ("ODE_v0", "ODE"):
        opt = optimizer_mppi_b200(predictor=pred, cost_function=cps.CostFunctionWrapper(),
                                  control_limits=([-1.0], [1.0]), seed=1, mpc_horizon=T, num_rollouts=K)
        opt.cost_function.configure(batch_size=K, horizon=T, variable_parameters=vp,
                                    cost_function_specification="quadratic_boundary_grad_minimal")
        opt.configure(num_states=6, num_control_inputs=1, dt=DT, predictor_specification=pred)
        a = np.pi - 1e-3
        s = np.array([a, 0.0, np.cos(a), np.sin(a), 0.0, 0.0], dtype=np.float32)
        for _ in range(50):
            opt.step(s)
        lat = np.empty(n_calls)
        for i in range(n_calls):
            t0 = time.perf_counter()
            opt.step(s)
            lat[i] = time.perf_counter() - t0
        # kernel-only time with CUDA events on the launching stream
        eng = opt.engine
        noise = torch.randn((eng.n_ind, K), device=eng.device)
        s_dev = torch.from_numpy(s).to(eng.device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ks = []
        for i in range(60):
            e0.record()
            eng.mppi_step(s_dev, noise, 1, 0.0)
            e1.record()
            e1.synchronize()
            if i >= 10:
                ks.append(e0.elapsed_time(e1))
        out[pred] = {"latency_ms_median": float(np.median(lat) * 1e3), "latency_ms_p99": float(np.percentile(lat, 99) * 1e3),
                     "kernel_ms_median": float(np.median(ks)),
                     "kernel_ms_in_stream": float(np.median(_stream_times(lambda: eng.mppi_step(s_dev, noise, 1, 0.0)))),
                     "calls": n_calls,
                     "state_steps_per_solve": K * T * N_SUB}
    out["config"] = ("K=2000, T=50, n=10, cost quadratic_boundary_grad_minimal, optimizer_mppi_b200.step(numpy s) -> numpy u; "
                     "kernel_ms_median = CUDA events around one launch on an idle GPU (includes the host's launch latency), "
                     "kernel_ms_in_stream = device time per solve in a stream of 20 back-to-back solves")
    out["neural_GRU_2x64"] = neural_latency(device, n_calls=min(n_calls, 300))
    try:
        out["neural_GRU_2x32"] = neural_latency(device, n_calls=min(n_calls, 300), hidden=32)
    except Exception as ex:
        out["neural_GRU_2x32"] = {"error": repr(ex)}
    out["neural_GRU_2x64_K65536"] = neural_big(device)
    out["ODE_K65536_T100"] = big_solve(device)
    try:
        out["legacy_controller_mppi_cartpole"] = legacy_latency(device, n_calls=min(n_calls, 300))
    except Exception as ex:
        out["legacy_controller_mppi_cartpole"] = {"error": repr(ex)}
    try:
        out["fleet_1024x2000x50"] = fleet_bench(device, E_total=1024, periods=20)
        from oracle import oracle as O
        O.lib().cps_oracle_set_num_threads(os.cpu_count() or 1)
        eps = np.random.default_rng(0).standard_normal((K, 6)).astype(np.float32)
        s = np.array([np.pi - 1e-3, 0.0, np.cos(np.pi - 1e-3), np.sin(np.pi - 1e-3), 0.0, 0.0], dtype=np.float32)
        O.mppi_step("ODE", "quadratic_boundary_grad_minimal", s, np.zeros(T, np.float32), eps=eps[:64])
        t0 = time.perf_counter()
        for _ in range(5):
            r = O.mppi_step("ODE", "quadratic_boundary_grad_minimal", s, np.zeros(T, np.float32), eps=eps)
            O.plant_period(s, float(r["u"]))
        out["fleet_1024x2000x50"]["cpu_port_ms_per_experiment_period"] = (time.perf_counter() - t0) / 5 * 1e3
        out["fleet_1024x2000x50"]["cpu_port_threads"] = O.lib().cps_oracle_num_threads()
    except Exception as ex:
        out["fleet_1024x2000x50"] = {"error": repr(ex)}
    for key, fn in (("forward_optimizers", planner_latency), ("relabel_256_files", relabel_bench)):
        try:
            out[key] = fn(device)
        except Exception as ex:
            out[key] = {"error": repr(ex)}
    return out


def planner_latency(device, n_calls=300):
    """SURVEY 8f row f3: optimizer_cem_b200 / optimizer_random_action_b200 .step(numpy s) -> numpy u with the
    reference's shipped settings (config_optimizers.yml: cem-tf 200 rollouts x 35 steps, 3 outer iterations, 40 elites;
    random-action-tf 640 x 35) and CEM at K = 2000, T = 50; CPU port = the oracle restatement on all host threads."""
    import cartpolesimulation_b200 as cps
    from cartpolesimulation_b200.optimizer_forward_b200 import optimizer_cem_b200, optimizer_random_action_b200
    from oracle import oracle as O
    a = np.pi - 1e-3
    s = np.array([a, 0.0, np.cos(a), np.sin(a), 0.0, 0.0], dtype=np.float32)
    lim = (np.array([-1.0], np.float32), np.array([1.0], np.float32))
    out = {}
    cases = (("cem_200x35_it3", optimizer_cem_b200, 200, 35, dict(cem_outer_it=3, cem_best_k=40)),
             ("cem_2000x50_it3", optimizer_cem_b200, 2000, 50, dict(cem_outer_it=3, cem_best_k=200)),
             ("random_action_640x35", optimizer_random_action_b200, 640, 35, {}))
    for name, cls, K, T, kw in cases:
        vp = cps.VariableParameters(target_position=0.0, target_equilibrium=1.0, L=0.395, m_pole=0.087)
        cost, pred = cps.CostFunctionWrapper(), cps.PredictorWrapper()
        opt = cls(predictor=pred, cost_function=cost, control_limits=lim, seed=1, mpc_horizon=T, num_rollouts=K,
                  device=device, **kw)
        pred.configure(batch_size=K, horizon=T, dt=0.02, variable_parameters=vp, predictor_specification="ODE")
        cost.configure(batch_size=K, horizon=T, variable_parameters=vp, environment_name="CartPole",
                       computation_library=None, cost_function_specification="quadratic_boundary_grad_minimal")
        opt.configure(num_states=6, num_control_inputs=1, dt=0.02, predictor_specification="ODE")
        for _ in range(20):
            opt.step(s)
        lat = []
        for _ in range(n_calls):
            t0 = time.perf_counter()
            opt.step(s)
            lat.append((time.perf_counter() - t0) * 1e3)
        n0 = opt.engine.launch_count()
        opt.step(s)
        rec = {"latency_ms_median": float(np.median(lat)), "latency_ms_p99": float(np.percentile(lat, 99)),
               "launches_per_solve": opt.engine.launch_count() - n0, "calls": n_calls,
               "state_steps_per_solve": K * T * N_SUB * kw.get("cem_outer_it", 1)}
        O.lib().cps_oracle_set_num_threads(os.cpu_count() or 1)
        rng = np.random.default_rng(0)
        t0 = time.perf_counter()
        for _ in range(3):
            if cls is optimizer_cem_b200:
                O.cem_step("ODE", "quadratic_boundary_grad_minimal", s, rng.standard_normal((3, K, T)).astype(np.float32),
                           np.zeros(T, np.float32), np.full(T, 0.5, np.float32), kw["cem_best_k"], 0.01, 0.5)
            else:
                O.random_action_step("ODE", "quadratic_boundary_grad_minimal", s, rng.uniform(-1, 1, (K, T)).astype(np.float32))
        rec["cpu_port_ms"] = (time.perf_counter() - t0) / 3 * 1e3
        rec["cpu_port_threads"] = O.lib().cps_oracle_num_threads()
        out[name] = rec
        opt.engine.close()
    # the reference's shipped default optimizer: RPGD at its shipped configuration (config_optimizers.yml:63-85: 16 plans x 35
    # steps, 4 Adam steps on the adjoint's gradient per solve), and CEM-GMM at its shipped 200 x 35 x 3
    from cartpolesimulation_b200.optimizer_forward_b200 import optimizer_cem_gmm_b200, optimizer_rpgd_b200
    for name, cls, K, T, kw in (("rpgd_16x35_it4", optimizer_rpgd_b200, 16, 35, dict(outer_its=4)),
                                ("rpgd_2000x50_it4", optimizer_rpgd_b200, 2000, 50, dict(outer_its=4)),
                                ("cem_gmm_200x35_it3", optimizer_cem_gmm_b200, 200, 35, dict(cem_outer_it=3, cem_best_k=40))):
        try:
            vp = cps.VariableParameters(target_position=0.0, target_equilibrium=1.0, L=0.395, m_pole=0.087)
            cost, pred = cps.CostFunctionWrapper(), cps.PredictorWrapper()
            opt = cls(predictor=pred, cost_function=cost, control_limits=lim, seed=1, mpc_horizon=T, num_rollouts=K, device=device, **kw)
            pred.configure(batch_size=K, horizon=T, dt=0.02, variable_parameters=vp, predictor_specification="ODE")
            cost.configure(batch_size=K, horizon=T, variable_parameters=vp, environment_name="CartPole",
                           computation_library=None, cost_function_specification="quadratic_boundary_grad_minimal")
            opt.configure(num_states=6, num_control_inputs=1, dt=0.02, predictor_specification="ODE")
            for _ in range(20):
                opt.step(s)
            lat = []
            for _ in range(n_calls):
                t0 = time.perf_counter()
                opt.step(s)
                lat.append((time.perf_counter() - t0) * 1e3)
            n0 = opt.engine.launch_count()
            opt.step(s)
            rec = {"latency_ms_median": float(np.median(lat)), "latency_ms_p99": float(np.percentile(lat, 99)),
                   "launches_per_solve": opt.engine.launch_count() - n0, "calls": n_calls}
            if cls is optimizer_rpgd_b200:   # the adjoint kernel alone
                import torch
                Q = torch.zeros((K, T), device=opt.device).uniform_(-0.5, 0.5)
                s_dev = torch.from_numpy(s).to(opt.device)
                rec["grad_kernel_ms_in_stream"] = float(np.median(_stream_times(lambda: opt.engine.plan_cost_grad(s_dev, Q))))
                rec["state_steps_per_grad"] = K * T * N_SUB
            out[name] = rec
            opt.engine.close()
        except Exception as ex:
            out[name] = {"error": repr(ex)}
    out["api"] = ("optimizer_cem_b200 / optimizer_cem_gmm_b200 / optimizer_random_action_b200 / optimizer_rpgd_b200 .step(numpy s) -> numpy u "
                  "(cps_cem_step_host, cps_cem_gmm_step_host, cps_plan_random_action_host, cps_rpgd_grad_step; plan_kernel, plan_grad_fwd_kernel + plan_grad_jacrev_kernel)")
    return out


def relabel_bench(device, E=256, rows=50, K=2000, T=50):
    """SURVEY 8f row f4: add_control_along_trajectories for E recorded files in lockstep (cps_fleet_relabel), MPPI
    K = 2000, T = 50 per row, per-row pole length, in-kernel noise; host arrays in, labels out."""
    import torch
    from cartpolesimulation_b200.relabel import Relabeller
    from oracle import oracle as O
    rng = np.random.default_rng(0)
    ang = rng.uniform(-np.pi, np.pi, (rows, E))
    s = np.stack([ang, rng.uniform(-3, 3, (rows, E)), np.cos(ang), np.sin(ang), rng.uniform(-0.1, 0.1, (rows, E)),
                  rng.uniform(-0.3, 0.3, (rows, E))], axis=2).astype(np.float32)
    Lr = rng.uniform(0.25, 0.55, (rows, E)).astype(np.float32)
    tp = rng.uniform(-0.1, 0.1, (rows, E)).astype(np.float32)
    rl = Relabeller(E, K, T, noise="philox", seed=1, device=device)
    rl.relabel(s[:5], tp[:5], None, Lr[:5])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    Q = rl.relabel(s, tp, None, Lr)
    dt_s = time.perf_counter() - t0
    out = {"files": E, "rows_per_file": rows, "K": K, "T": T, "ms_per_row_of_all_files": dt_s / rows * 1e3,
           "labels_per_s": E * rows / dt_s, "state_steps_per_s": E * rows * K * T * N_SUB / dt_s,
           "finite": bool(np.isfinite(Q).all()), "launches": rows,
           "api": "Relabeller.relabel (numpy in, numpy out; cps_fleet_relabel, fleet_kernel in replay mode)"}
    O.lib().cps_oracle_set_num_threads(os.cpu_count() or 1)
    eps = rng.standard_normal((4, K, 6)).astype(np.float32)
    t0 = time.perf_counter()
    O.relabel_file("ODE", "quadratic_boundary_grad_minimal", T, s[:4, 0], eps, tp[:4, 0], None, Lr[:4, 0])
    out["cpu_port_ms_per_label"] = (time.perf_counter() - t0) / 4 * 1e3
    out["cpu_port_threads"] = O.lib().cps_oracle_num_threads()
    rl.close()
    return out


def legacy_latency(device, n_calls=300):
    """SURVEY 8f row f2: the legacy controller_mppi_cartpole at its shipped configuration (config_controllers.yml:9-30:
    K=3500, T=35, 'interpolated' sampling, predictor ODE): controller.step(numpy s) -> numpy Q, the host-drawn knot
    perturbations (numpy SFC64, the reference's generator call) included -- the interpolation between the knots, scipy
    interp1d in the reference, runs on the device; kernel-only time from CUDA events; the CPU port of the same iteration
    beside it.  reference_sampler_ms = what the reference's whole host sampler (draws + interp1d) costs on this host."""
    import torch
    from cartpolesimulation_b200.controller_mppi_cartpole_b200 import controller_mppi_cartpole_b200
    ctrl = controller_mppi_cartpole_b200(dict(seed=1), dt=DT, device=device)
    K, T = ctrl.num_rollouts, ctrl.mpc_horizon
    a = np.pi - 1e-3
    s = np.array([a, 0.0, np.cos(a), np.sin(a), 0.0, 0.0], dtype=np.float32)
    for _ in range(20):
        ctrl.step(s)
    lat, samp, knot = np.empty(n_calls), np.empty(n_calls), np.empty(n_calls)
    for i in range(n_calls):
        t0 = time.perf_counter()
        ctrl.step(s)
        lat[i] = time.perf_counter() - t0
    for i in range(n_calls):
        t0 = time.perf_counter()
        ctrl.initialize_perturbations(stdev=ctrl.SQRTRHODTINV, sampling_type=ctrl.SAMPLING_TYPE)
        samp[i] = time.perf_counter() - t0
        t0 = time.perf_counter()
        ctrl._interpolated_knots(stdev=ctrl.SQRTRHODTINV)
        knot[i] = time.perf_counter() - t0
    eng = ctrl.engine
    du = torch.from_numpy(np.ascontiguousarray(ctrl.delta_u.T, dtype=np.float32)).to(eng.device)
    s_dev = torch.from_numpy(s).to(eng.device)
    ks = _event_times(lambda: eng.legacy_step(s_dev, du, 1), 50, warm=10)
    out = {"latency_ms_median": float(np.median(lat) * 1e3), "latency_ms_p99": float(np.percentile(lat, 99) * 1e3),
           "host_sampler_ms_median": float(np.median(knot) * 1e3), "reference_sampler_ms_median": float(np.median(samp) * 1e3),
           "kernel_ms_median": float(np.median(ks)),
           "calls": n_calls, "K": K, "T": T, "state_steps_per_solve": K * T * N_SUB,
           "api": "controller_mppi_cartpole_b200.step(numpy s) -> numpy Q (cps_legacy_step_host_knots: legacy_interp_kernel + "
                  "legacy_mppi_kernel<ODE>)"}
    try:
        from oracle import legacy as OL
        from oracle import oracle as O
        O.lib().cps_oracle_set_num_threads(os.cpu_count() or 1)
        d = np.asarray(ctrl.delta_u, np.float32)
        OL.iteration("ODE", s, np.zeros(T, np.float32), np.zeros(T, np.float32), d[:64])
        t0 = time.perf_counter()
        for _ in range(3):
            OL.iteration("ODE", s, np.zeros(T, np.float32), np.zeros(T, np.float32), d)
        out["cpu_port_ms"] = (time.perf_counter() - t0) / 3 * 1e3
        out["cpu_port_threads"] = O.lib().cps_oracle_num_threads()
    except Exception as ex:
        out["cpu_port_ms"] = repr(ex)
    return out


def _stream_times(fn, n_batches=5, per_batch=20, warm=5):
    """Device time per call inside a stream of back-to-back calls (per_batch calls per CUDA-event pair): what a kernel
    costs without the host's launch latency, which an event pair around ONE launch on an idle GPU includes."""
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n_batches):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(per_batch):
            fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) / per_batch)
    return ts


def _event_times(fn, n, warm=5):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return ts


def neural_latency(device, n_calls=300, hidden=64):
    """BASELINE.json configs[2]: MPPI + autoregressive GRU (2x64 hidden), K=2000, T=50; synthetic seeded weights (no
    dynamics model ships with the reference).  One launch per solve: rollout + cost + update + hidden-state step.
    hidden = 32: the size of the network the reference's configuration names (GRU-6IN-32H1-32H2-5OUT-0)."""
    import torch
    from cartpolesimulation_b200.core import Engine
    from cartpolesimulation_b200.neural import net_flops_per_step, synthetic_net_spec
    K, T = 2000, 50
    spec = synthetic_net_spec((hidden, hidden), "GRU", seed=0)
    eng = Engine(K, T, integrator="neural", cost="quadratic_boundary_grad_minimal", device=device)
    eng.net_load(spec)
    a = np.pi - 1e-3
    s_np = np.array([a, 0.0, np.cos(a), np.sin(a), 0.0, 0.0], dtype=np.float32)
    s = torch.from_numpy(s_np).to(eng.device)
    noise = torch.randn((eng.n_ind, K), device=eng.device)
    ks = _event_times(lambda: eng.mppi_step(s, noise, 1, 0.0), 50)
    lat = np.empty(n_calls)
    for i in range(n_calls):
        t0 = time.perf_counter()
        eng.mppi_step_host(s_np, noise, 1, 0.0)
        lat[i] = time.perf_counter() - t0
    flops = net_flops_per_step(spec) * K * T
    kms = float(np.median(ks))
    out = {"latency_ms_median": float(np.median(lat) * 1e3), "latency_ms_p99": float(np.percentile(lat, 99) * 1e3),
           "kernel_ms_median": kms,
           "kernel_ms_in_stream": float(np.median(_stream_times(lambda: eng.mppi_step(s, noise, 1, 0.0)))),
           "net_steps_per_s": K * T / (kms * 1e-3), "fp32_tflops": flops / (kms * 1e-3) / 1e12,
           "flop_per_solve": flops,
           "api": "cps_mppi_step_host (numpy s -> float u); kernel: %s" % {"tensor": "net_tc_kernel<MPPI> (tcgen05)", "fp32": "net_kernel<16,%d,MPPI> (FP32)" % hidden}.get(eng.net_last_kernel(), "?")}
    try:  # the same solve by the CPU oracle port (C, OpenMP), once, on the host cores
        from oracle import oracle as O
        eps = noise.t().contiguous().cpu().numpy()
        args = (spec["net_type"], spec["hsz"], spec["weights"], spec["in_idx"], spec["out_idx"], spec["norm_a"],
                spec["norm_b"], spec["denorm_A"], spec["denorm_B"])
        O.lib().cps_oracle_set_num_threads(os.cpu_count() or 1)
        O.mppi_step_net("quadratic_boundary_grad_minimal", *args, s_np, np.zeros(T, np.float32), eps[:64])
        t0 = time.perf_counter()
        O.mppi_step_net("quadratic_boundary_grad_minimal", *args, s_np, np.zeros(T, np.float32), eps)
        out["cpu_port_ms"] = (time.perf_counter() - t0) * 1e3
        out["cpu_port_threads"] = O.lib().cps_oracle_num_threads()
    except Exception as ex:
        out["cpu_port_ms"] = repr(ex)
    return out


def neural_big(device):
    """The same GRU solve at K = 65536 (T = 50): tcgen05 tensor-core kernel vs the FP32 CUDA-core kernel."""
    import torch
    from cartpolesimulation_b200.core import Engine
    from cartpolesimulation_b200.neural import net_flops_per_step, synthetic_net_spec
    K, T = 65536, 50
    spec = synthetic_net_spec((64, 64), "GRU", seed=0)
    out = {}
    for kern in ("tensor", "fp32"):
        eng = Engine(K, T, integrator="neural", cost="quadratic_boundary_grad_minimal", device=device, net_kernel=kern)
        eng.net_load(spec)
        a = np.pi - 1e-3
        s = torch.tensor([a, 0.0, np.cos(a), np.sin(a), 0.0, 0.0], device=eng.device, dtype=torch.float32)
        noise = torch.randn((eng.n_ind, K), device=eng.device)
        kms = float(np.median(_event_times(lambda: eng.mppi_step(s, noise, 1, 0.0), 10, warm=3)))
        out[kern] = {"kernel_ms_median": kms, "net_steps_per_s": K * T / (kms * 1e-3),
                     "effective_fp32_tflops": net_flops_per_step(spec) * K * T / (kms * 1e-3) / 1e12}
        eng.close()
    out["note"] = ("tensor = net_tc_kernel (tcgen05.mma kind::f16, fp16 hi/lo 3-pass split, fp32 accumulators in TMEM): "
                   "3x the algorithmic MACs on the tensor pipe; effective_fp32_tflops counts the algorithmic FLOPs only")
    return out


def big_solve(device):
    """BASELINE.json configs[3]: MPPI K=65536, T=100, fused quadratic+barrier cost (quadratic_boundary), one GPU."""
    import torch
    from cartpolesimulation_b200.core import Engine
    K, T = 65536, 100
    out = {}
    for cost in ("quadratic_boundary", "quadratic_boundary_grad_minimal"):
        eng = Engine(K, T, integrator="ODE", cost=cost, device=device)
        a = np.pi - 1e-3
        s = torch.tensor([a, 0.0, np.cos(a), np.sin(a), 0.0, 0.0], device=eng.device, dtype=torch.float32)
        noise = torch.randn((eng.n_ind, K), device=eng.device)
        ks = _event_times(lambda: eng.mppi_step(s, noise, 1, 0.0), 30)
        kms = float(np.median(ks))
        out[cost] = {"kernel_ms_median": kms, "state_steps_per_s": K * T * N_SUB / (kms * 1e-3),
                     "kernel_ms_in_stream": float(np.median(_stream_times(lambda: eng.mppi_step(s, noise, 1, 0.0))))}
        eng.close()
    return out


def fleet_bench(device, E_total=8192, world=1, rank=0, periods=20, K=2000, T=50):
    """BASELINE.json configs[4]: data_generator with 8192 independent MPPI-controlled cartpoles (K=2000, T=50 each),
    sharded over the ranks (no data-path collective).  One launch = one controller period of every local experiment:
    MPPI solve + plant, noise drawn in the kernel (Philox), targets from the host-side data-generator tables."""
    import torch
    from cartpolesimulation_b200.fleet import DataGenConfig, Fleet, make_experiments
    E = E_total // world
    off = rank * E
    cfg = DataGenConfig(length_of_experiment=max(2.0, periods * 0.02 * 2))
    s0, tp, te = make_experiments(E, periods, cfg, seed=0, experiment_offset=off)
    fl = Fleet(E, K, T, integrator="ODE", cost="quadratic_boundary_grad_minimal", noise="philox", seed=0,
               experiment_offset=off, device=device)
    tp_d, te_d = torch.from_numpy(tp).to(fl.device), torch.from_numpy(te).to(fl.device)
    rec = torch.zeros((periods, E, 16), device=fl.device)
    fl.reset(s0)
    fl.run(min(3, periods), tp_d[:3].contiguous(), te_d[:3].contiguous(), None, None)   # warm-up
    fl.reset(s0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fl.run(periods, tp_d, te_d, None, rec)
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1)
    rec_h = rec.cpu().numpy()
    out = {"experiments_total": E_total, "experiments_per_gpu": E, "K": K, "T": T, "periods": periods,
           "ms_per_period": ms / periods, "experiment_periods_per_s_per_gpu": E * periods / (ms * 1e-3),
           "state_steps_per_s_per_gpu": float(E) * K * T * N_SUB * periods / (ms * 1e-3),
           "sim_seconds_per_wall_second_per_gpu": E * periods * 0.02 / (ms * 1e-3),
           "finite": bool(np.isfinite(rec_h).all()), "launches": periods,
           "d2h_record_bytes": int(rec.numel() * 4)}
    fl.close()
    return out


def sharded_solve(local_rank, world, n=30):
    """configs[3] with K sharded over the ranks, both transports of ShardedMPPI: "peer" = ONE launch per solve (local
    rollouts, records pushed over NVLink into every rank's symmetric-memory buffer, update finished on every rank) and
    "allgather" = kernel + NCCL all-gather of n_ind+2 floats + finalize kernel.  Device time of the slowest rank.
    Self-check on every run: all ranks hold bit-identical u_nom, and they agree with a one-GPU solve of the same K
    rollouts (same noise) on rank 0 to 2e-6 (different association order of the block sums only)."""
    import torch
    import torch.distributed as dist
    from cartpolesimulation_b200.core import Engine
    from cartpolesimulation_b200.distributed import ShardedMPPI
    K, T = 65536, 100
    dev = torch.device("cuda", local_rank)
    rank = dist.get_rank() if world > 1 else 0
    a = np.pi - 1e-3
    s = torch.tensor([a, 0.0, np.cos(a), np.sin(a), 0.0, 0.0], device=dev, dtype=torch.float32)
    out = {"K_total": K, "T": T, "ranks": world}
    full = None
    for exchange in ("peer", "allgather"):
        rec = {}
        try:
            sm = ShardedMPPI(K, T, integrator="ODE", cost="quadratic_boundary", device=local_rank, exchange=exchange)
            if full is None:   # the same draws on every rank (seeded device generator), each takes its slice
                g = torch.Generator(device=dev)
                g.manual_seed(7)
                full = torch.randn((sm.engine.n_ind, K), device=dev, generator=g)
            noise = sm.noise_slice(full)
            # ---- parity --------------------------------------------------------------------------------------------
            sm.reset(0.0)
            u = sm.step(s, noise, 1, 0.0)
            mine = torch.cat([torch.from_numpy(sm.get_u_nom()).to(dev), u.reshape(1).float()])
            allr = torch.empty((world, mine.numel()), device=dev)
            if world > 1:
                dist.all_gather_into_tensor(allr, mine)
            else:
                allr[0] = mine
            rec["ranks_bit_identical"] = bool((allr == allr[0]).all().item())
            if rank == 0:
                ref = Engine(K, T, integrator="ODE", cost="quadratic_boundary", device=local_rank)
                ref.mppi_reset(0.0)
                u1 = ref.mppi_step(s, full, 1, 0.0)
                d_nom = float(np.abs(ref.get_u_nom() - sm.get_u_nom()).max())
                d_u = abs(float(u1.cpu()[0]) - float(u.cpu()[0]))
                rec["vs_one_gpu_solve"] = {"u_nom_max_abs_diff": d_nom, "u_abs_diff": d_u, "tol": 2e-6}
                rec["parity_ok"] = bool(rec["ranks_bit_identical"] and d_nom <= 2e-6 and d_u <= 2e-6)
                ref.close()
            # ---- time ----------------------------------------------------------------------------------------------
            ks = _event_times(lambda: sm.step(s, noise, 1, 0.0), n)
            t = torch.tensor([float(np.median(ks))], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            rec["solve_ms_median_max_over_ranks"] = float(t.item())
            rec["state_steps_per_s"] = K * T * N_SUB / (float(t.item()) * 1e-3)
            rec["exchange_bytes_per_rank"] = 4 * sm.rec
            rec["transport"] = sm.exchange
            rec["launches_per_solve"] = 1 if sm.exchange == "peer" else 2
            # ---- where the time goes (this rank; CUDA events around each stream operation) ----------------------------
            if sm.exchange == "allgather":
                eng = sm.engine
                bd = {"local_kernel_us": 1e3 * float(np.median(_event_times(lambda: eng.mppi_step(s, noise, 1, 0.0), n))),
                      "finalize_us": 1e3 * float(np.median(_event_times(lambda: eng.mppi_finalize(sm._gathered), n)))}
                if world > 1:
                    bd["allgather_us"] = 1e3 * float(np.median(_event_times(
                        lambda: dist.all_gather_into_tensor(sm._gathered, sm._partial), n)))
                rec["breakdown"] = bd
            else:
                solo = Engine(sm.K_local, T, integrator="ODE", cost="quadratic_boundary", device=local_rank)
                lk = 1e3 * float(np.median(_event_times(lambda: solo.mppi_step(s, noise, 1, 0.0), n)))
                solo.close()
                rec["breakdown"] = {"local_kernel_us": lk, "exchange_and_wait_us": 1e3 * float(np.median(ks)) - lk,
                                    "note": "local = the same K_local solve without the exchange; the rest is the push "
                                            "over NVLink plus waiting for the slowest rank's record"}
                rec["peer_timeouts"] = sm.engine.peer_timeouts()
            sm.engine.close()
        except Exception as ex:
            rec["error"] = repr(ex)
        out[exchange] = rec
    best = min((out[k] for k in ("peer", "allgather") if "solve_ms_median_max_over_ranks" in out[k]),
               key=lambda r: r["solve_ms_median_max_over_ranks"], default=None)
    if best:
        out["solve_ms_median_max_over_ranks"] = best["solve_ms_median_max_over_ranks"]
        out["state_steps_per_s"] = best["state_steps_per_s"]
        out["parity_ok"] = all(out[k].get("parity_ok", True) and out[k].get("ranks_bit_identical", False)
                               for k in ("peer", "allgather") if "error" not in out[k])
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    from cartpolesimulation_b200.core import Engine
    from cartpolesimulation_b200 import _lib as L

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_cpus, all_cpus = None, os.sched_getaffinity(0)
    if world > 1:   # one process per GPU: keep the pinned host buffers of the e2e leg on the GPU's own NUMA node
        from cartpolesimulation_b200.distributed import bind_to_gpu_numa
        numa_cpus = bind_to_gpu_numa(local_rank)
    if world > 1:
        # stdout carries exactly ONE JSON line: NCCL's banner ("NCCL version ...") goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    B, T = args.batch, args.horizon
    eng = Engine(B, T, dt=DT, substeps=N_SUB, integrator="ODE_v0", cost=None, device=local_rank,
                 fast_sincos=args.fast_sincos, substep_sincos=args.substep_sincos)
    s0_np, Q_np = make_inputs(B, T, seed=1234 + rank)
    s0 = torch.from_numpy(s0_np).to(dev)
    Q = torch.from_numpy(Q_np).to(dev)           # [T, B] time-major, 200 MB > L2 (126 MB): no L2 flush needed
    traj = torch.empty((T + 1, 6, B), device=dev)  # 1.22 GB, written every step

    def one_pass():
        eng.rollout(s0, Q, q_layout=L.TIME_MAJOR, traj_layout=L.TIME_MAJOR, traj_out=traj)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        one_pass()
    barrier()
    # The K timed passes are replayed as ONE CUDA graph (captured before the timed region): the host issues a single
    # launch, so Python / ctypes launch gaps and host-side jitter of N concurrent processes stay out of the device time.
    graph = None
    if not args.no_graph:
        try:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                one_pass()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=side):
                    for _ in range(args.steps):
                        one_pass()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize()
            g.replay()          # one untimed replay (graph upload)
            torch.cuda.synchronize()
            graph = g
        except Exception as ex:   # fall back to K separate launches
            print(f"[bench] CUDA graph capture failed ({ex!r}); timing {args.steps} separate launches", file=sys.stderr)
            graph = None
            torch.cuda.synchronize()
        eng.use_current_stream()
    # per-launch kernel time (CUDA events around single launches on the launching stream) for the roofline
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(min(args.steps, 10))]
    for e0, e1 in evs:
        e0.record()
        one_pass()
        e1.record()
    torch.cuda.synchronize()
    kern_ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = eng.launch_count()
    barrier()
    t_all0 = torch.cuda.Event(enable_timing=True)
    t_all1 = torch.cuda.Event(enable_timing=True)
    t_all0.record()
    if graph is not None:
        graph.replay()
    else:
        for _ in range(args.steps):
            one_pass()
    t_all1.record()
    barrier()
    launches = (args.steps if graph is not None else eng.launch_count() - launches0)
    kernel_label = eng.rollout_last_kernel() or "rollout_kernel"   # what the timed passes dispatched to
    total_ms = t_all0.elapsed_time(t_all1)
    if args.dump_outputs and rank == 0:   # traj still holds the last timed pass
        dump_outputs(args.dump_outputs, traj)
    per_rank = None
    if world > 1:
        # every rank's own device time and per-launch kernel time: with no communication in the timed region, the spread
        # between ranks (GPU-to-GPU clock / power differences) is all there is to the weak-scaling loss
        mine = torch.tensor([total_ms / args.steps, kern_ms], device=dev, dtype=torch.float64)
        allr = torch.empty((world, 2), device=dev, dtype=torch.float64)
        dist.all_gather_into_tensor(allr, mine)
        per_rank = {"ms_per_step": [float(v) for v in allr[:, 0].cpu()], "kernel_ms": [float(v) for v in allr[:, 1].cpu()]}
        total_ms = float(allr[:, 0].max().item()) * args.steps
    steps_per_pass = float(B) * T * N_SUB
    value = steps_per_pass * args.steps * world / (total_ms * 1e-3)

    # ---- e2e: host buffers through cps_rollout_host (pinned), H2D + kernel + D2H inside the timed region --------
    s0_pin = torch.from_numpy(s0_np).pin_memory()
    Q_pin = torch.from_numpy(Q_np).pin_memory()
    traj_pin = torch.empty((T + 1, 6, B), pin_memory=True)
    final_pin = torch.empty((B, 6), pin_memory=True)
    e2e_steps = max(2, min(args.steps, 5))

    def timed_host(fn, n):
        for _ in range(2):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
        dt_s = time.perf_counter() - t0
        if world > 1:   # the slowest rank decides
            t = torch.tensor([dt_s], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt_s = float(t.item())
        return dt_s

    # (1) the full trajectory comes back (what predictor.predict_core returns): PCIe-bound, 1.28 GB D2H per pass
    e2e_s = timed_host(lambda: eng.rollout_host(s0_pin.numpy(), Q_pin.numpy(), L.TIME_MAJOR, L.TIME_MAJOR,
                                                traj_out=traj_pin.numpy()), e2e_steps)
    # (2) only the final states come back (what a cost-only / MPPI caller needs from the rollouts): 25 MB D2H per pass
    e2e_final_s = timed_host(lambda: eng.rollout_host(s0_pin.numpy(), Q_pin.numpy(), L.TIME_MAJOR, L.TIME_MAJOR,
                                                      traj_out=None, final_out=final_pin.numpy()), e2e_steps)
    # (3) the bus itself: pinned device-to-host and host-to-device copies of the same buffers, all ranks at once -- the
    #     ceiling the full-trajectory leg runs against (N ranks share one host memory system and the PCIe root complexes)
    def copy_rate(dst, src, n=3):
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        for _ in range(n):
            dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        dt_s = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt_s], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt_s = float(t.item())
        return src.numel() * 4 * n / dt_s / 1e9   # GB/s per rank, slowest rank
    d2h_gbs = copy_rate(traj_pin, traj)
    h2d_gbs = copy_rate(Q, Q_pin)
    if numa_cpus:
        os.sched_setaffinity(0, all_cpus)   # the CPU baseline below uses every host core again
    sampler.stop_flag = True   # the clock record covers both timed regions (device-resident and e2e)
    sampler.join(timeout=1.0)
    e2e_value = steps_per_pass * e2e_steps * world / e2e_s
    e2e_final_value = steps_per_pass * e2e_steps * world / e2e_final_s
    h2d = s0_pin.numel() * 4 + Q_pin.numel() * 4
    d2h = traj_pin.numel() * 4
    # time the two copies alone would take on this rank at the measured concurrent rates (they do not overlap each other
    # much: the D2H of a chunk follows its kernel, the H2D of the next chunk runs beside it)
    bus_floor_s = d2h / (d2h_gbs * 1e9)
    e2e_bus = {"achieved_gbs_per_rank": (h2d + d2h) / (e2e_s / e2e_steps) / 1e9,
               "d2h_gbs_per_rank_all_ranks_copying": d2h_gbs, "h2d_gbs_per_rank_all_ranks_copying": h2d_gbs,
               "d2h_gbs_all_ranks": d2h_gbs * world,
               "frac_of_d2h_copy_rate": (d2h / (e2e_s / e2e_steps) / 1e9) / d2h_gbs,
               "d2h_floor_ms_per_step": 1e3 * bus_floor_s,
               "note": "full-trajectory leg = 1.28 GB device-to-host per pass: bounded by the pinned D2H copy rate measured here "
                       "with every rank copying at once, not by the 0.8 ms kernel"}

    sharded = None
    fleet = None
    if world > 1 and not args.no_mppi:
        try:
            sharded = sharded_solve(local_rank, world)
        except Exception as ex:
            sharded = {"error": repr(ex)}
        try:  # configs[4]: 8192 experiments over the ranks; the slowest rank's time decides
            fleet = fleet_bench(local_rank, E_total=8192, world=world, rank=rank, periods=10)
            t = torch.tensor([fleet["ms_per_period"]], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            fleet["ms_per_period_max_over_ranks"] = float(t.item())
            fleet["state_steps_per_s_all_gpus"] = 8192.0 * 2000 * 50 * N_SUB / (float(t.item()) * 1e-3)
        except Exception as ex:
            fleet = {"error": repr(ex)}
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (rollout_kernel) ------------------------------------------------------
    fp32_peak, mufu_peak = eng.measure_peaks()
    rate_1gpu = steps_per_pass / (kern_ms * 1e-3)
    achieved_tflops = rate_1gpu * FLOP_PER_STATE_STEP / 1e12
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    alg_bytes = 4.0 * B * T + 24.0 * B * (T + 1) + 24.0 * B   # Q in, trajectory out, s0 in
    traffic, ncu_view = None, None
    try:
        rt = json.load(open(os.path.join(REPO, "profiles", "roofline_traffic.json")))
        traffic = rt.get("rollout_kernel_dram_bytes_per_launch")
        ncu_view = rt.get("ncu")   # pipe utilisation of the same kernel from the committed ncu capture (not measured live)
    except Exception:
        pass
    roofline = {"bound": "fp32", "kernel": "%s<ODE_v0>" % kernel_label, "achieved": achieved_tflops, "peak": fp32_peak,
                "unit": "TFLOP/s", "frac": achieved_tflops / fp32_peak if fp32_peak else None, "traffic": traffic,
                "traffic_source": "committed ncu capture (profiles/roofline_traffic.json), not measured in this run",
                "peak_source": "cps_measure_peaks FFMA microbenchmark, this run (not in MEASURED_PEAKS.json)",
                "flop_per_state_step": FLOP_PER_STATE_STEP, "kernel_ms": kern_ms,
                "fp32_pipe": {"lane_ops_per_state_step": FP32_LANE_OPS_PER_STATE_STEP,
                              "achieved_frac_of_lanes": rate_1gpu * FP32_LANE_OPS_PER_STATE_STEP / (fp32_peak * 1e12 / 2.0)
                              if fp32_peak else None,
                              "note": "FMA-pipe lane operations executed per state-step (FMUL/FADD occupy a lane like an FMA): "
                                      "29 in the substep + ~2.7 amortised per-control-step work; peak = measured FFMA "
                                      "lane rate (roofline.peak / 2)"},
                "frac_of_theoretical": achieved_tflops / (148 * 128 * 2 * 1.965e-3),
                "theoretical_note": "148 SMs x 128 lanes x 2 flops x 1965 MHz = 74.5 TFLOP/s",
                "ncu": ncu_view,
                "mufu": {"achieved_gops": rate_1gpu * (MUFU_PER_STATE_STEP if args.fast_sincos else 1.0) / 1e9,
                         "peak_gops": mufu_peak},
                "hbm": {"achieved_gbs": alg_bytes / (kern_ms * 1e-3) / 1e9, "peak_gbs": hbm_peak,
                        "frac": alg_bytes / (kern_ms * 1e-3) / 1e9 / hbm_peak, "algorithmic_bytes": alg_bytes,
                        "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"}}

    # ---- cpu baseline: oracle port on a bounded sample ---------------------------------------------------------
    rate0, _, threads = cpu_port_rate(4096, T)
    B_sample = int(min(B, max(4096, rate0 * 10.0 / (T * N_SUB))))   # ~10 s of CPU work
    reps = max(1, int(round(10.0 * rate0 / (B_sample * T * N_SUB))))
    cpu_rate, cpu_s, threads = cpu_port_rate(B_sample, T, repeats=reps)
    cpu_baseline = {"value": cpu_rate, "unit": UNIT, "cores": threads, "kind": "port",
                    "sample": f"{reps} x ({B_sample} of {B} cartpoles x {T * N_SUB} substeps), {cpu_s:.1f} s of CPU work",
                    "host_cores": os.cpu_count()}

    mppi = None
    if not args.no_mppi:
        try:
            mppi = mppi_latency(local_rank, n_calls=args.mppi_calls)
        except Exception as ex:  # never lose the headline line because of the secondary measurement
            mppi = {"error": repr(ex)}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(B, T), "per_gpu_batch": B, "l2": "inputs larger than L2 (Q = %d MB)" % (Q.numel() * 4 >> 20),
                       "sincos": ("MUFU every substep" if args.fast_sincos else "sincosf every substep")
                       if (args.fast_sincos or args.substep_sincos) else
                       "rotation substeps + sincosf resync per control step (default)",
                       "timed_region": ("one CUDA graph replay of the %d passes" % args.steps) if graph is not None
                       else ("%d separate launches" % args.steps)},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "ms_per_step": 1e3 * e2e_s / e2e_steps, "api": "cps_rollout_host (pinned host buffers), full trajectory returned",
                    "numa_bound_cpus": len(numa_cpus) if numa_cpus else None, "pcie": e2e_bus,
                    "final_states_only": {"value": e2e_final_value, "unit": UNIT, "h2d_bytes_per_step": h2d,
                                          "d2h_bytes_per_step": int(final_pin.numel() * 4),
                                          "ms_per_step": 1e3 * e2e_final_s / e2e_steps,
                                          "api": "cps_rollout_host(traj_out=NULL, final_out): what a cost-only caller moves"}},
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu_baseline,
            "clocks": sampler.summary(), "per_rank": per_rank, "mppi_solve": mppi, "mppi_sharded": sharded, "fleet_sharded": fleet}
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed passes of the headline figure (the e2e legs time max(2, min(steps, 5)), e2e.steps)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=B_DEFAULT, help="cartpoles per GPU")
    ap.add_argument("--horizon", type=int, default=T_DEFAULT)
    ap.add_argument("--fast-sincos", action="store_true", help="MUFU sin/cos every substep (parity-checked separately)")
    ap.add_argument("--substep-sincos", action="store_true", help="sincosf every substep, literally as the reference")
    ap.add_argument("--no-mppi", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time K separate launches instead of one CUDA graph of K passes")
    ap.add_argument("--mppi-calls", type=int, default=1000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (rank 0's batch) as DIR/<name>.npy; "
                         "--impl reference: the CPU port's rollouts of the same sampled cartpoles")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
