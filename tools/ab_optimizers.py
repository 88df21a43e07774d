"""A/B check of the single-solve drop-ins: closed loops of optimizer_mppi_b200, optimizer_{random_action,cem,cem_gmm,rpgd}_b200
and controller_mppi_cartpole_b200, the plant advanced between solves by oracle.plant_period.  Writes every step's control
and the optimizer's final device-side state to an .npz; `--compare A B` checks two such files bit for bit.

Two trees side by side (e.g. a change and its parent, each with its library built):
    python tools/ab_optimizers.py --root <parent tree> --out parent.npz
    python tools/ab_optimizers.py --root . --out change.npz
    python tools/ab_optimizers.py --compare parent.npz change.npz
300 steps cross the 256-solve refill of the draw rings; CEM-GMM at 2000 x 50 refills its normal and uniform rings at
different steps."""
import argparse
import os
import sys
import tempfile

import numpy as np

GRADMIN = "quadratic_boundary_grad_minimal"
S0 = np.array([np.pi - 0.4, 0.0, np.cos(np.pi - 0.4), np.sin(np.pi - 0.4), 0.05, 0.0], dtype=np.float32)


class SuppliedGenerator:
    """A caller-supplied generator (numpy draws handed over as CPU tensors) that logs the shapes it is asked for."""

    def __init__(self, seed):
        self.rng, self.calls = np.random.default_rng(seed), []

    def normal(self, shape, mean=0.0, stddev=1.0, dtype=None):
        import torch
        self.calls.append(f"normal{tuple(shape)}")
        return torch.from_numpy((self.rng.standard_normal(tuple(shape)) * stddev + mean).astype(np.float32))

    def uniform(self, shape, minval=0.0, maxval=1.0, dtype=None):
        import torch
        self.calls.append(f"uniform{tuple(shape)}")
        return torch.from_numpy(self.rng.uniform(minval, maxval, tuple(shape)).astype(np.float32))


def run(root, out):
    sys.path.insert(0, os.path.abspath(root))
    import torch
    import cartpolesimulation_b200 as cps
    from cartpolesimulation_b200 import optimizer_forward_b200 as F
    from cartpolesimulation_b200.controller_mppi_cartpole_b200 import controller_mppi_cartpole_b200
    from cartpolesimulation_b200.optimizer_mppi_b200 import optimizer_mppi_b200
    from oracle import oracle as O
    from tests.netutil import write_model_dir
    from tests.parity import load_golden
    tmp = tempfile.mkdtemp()
    gru = write_model_dir(tmp, load_golden("net_GRU_6IN_32H1_32H2_5OUT_0")[0])

    def make(cls, K, T, neural=False, **kw):
        vp = cps.VariableParameters(target_position=0.1, target_equilibrium=1.0, L=0.395, m_pole=0.087)
        cost, predictor = cps.CostFunctionWrapper(), cps.PredictorWrapper()
        predictor.configure(batch_size=K, horizon=T, dt=0.02, variable_parameters=vp,
                            predictor_specification=gru if neural else "ODE")
        cost.configure(batch_size=K, horizon=T, variable_parameters=vp, environment_name="CartPole", computation_library=None,
                       cost_function_specification=GRADMIN)
        opt = cls(predictor=predictor, cost_function=cost, seed=7, mpc_horizon=T, num_rollouts=K,
                  control_limits=(np.array([-1.0], np.float32), np.array([1.0], np.float32)), **kw)
        opt.configure(num_states=6, num_control_inputs=1, dt=0.02, predictor_specification="neural" if neural else "ODE")
        return opt

    def state(opt):
        e, st = opt.engine, {}
        if isinstance(opt, optimizer_mppi_b200):
            st["u_nom"] = e.get_u_nom()
            if opt.predictor_type == "neural":
                st["hidden"] = e.net_get_state()
            if opt.optimal_trajectory is not None:
                st["optimal_trajectory"] = opt.optimal_trajectory
        elif isinstance(opt, F.optimizer_cem_b200):
            st["dist_mue"], st["stdev"] = e.cem_get_distribution()
        elif isinstance(opt, F.optimizer_cem_gmm_b200):
            st["loc"], st["scale"], p1 = e.cem_gmm_get_distribution()
            st["p1"] = np.float32(p1)
        elif isinstance(opt, F.optimizer_rpgd_b200):
            m, v, it = e.rpgd_adam_state()
            st.update(Q_tf=opt.Q_tf.cpu().numpy(), adam_m=m.cpu().numpy(), adam_v=v.cpu().numpy(), adam_it=np.int64(it),
                      trajectory_ages=opt.trajectory_ages.cpu().numpy())
        for k, v in opt.logging_values.items():
            st["log_" + k] = np.asarray(v)
        return st

    def loop(opt, steps, supplied=False):
        gen = SuppliedGenerator(11) if supplied else None
        if gen is not None:
            opt.rng = gen
        s, us = S0.copy(), []
        for _ in range(steps):
            u = np.float32(opt.step(s.copy()))
            us.append(u)
            s, _, _ = O.plant_period(s, float(u))
        res = dict(u=np.array(us, dtype=np.float32), **state(opt))
        if gen is not None:
            res["generator_calls"] = np.array(gen.calls)
        return res

    def legacy(sampling, update_every, steps=20):
        ctrl = controller_mppi_cartpole_b200(dict(seed=5, mpc_horizon=35, num_rollouts=1000, update_every=update_every,
                                                  SAMPLING_TYPE=sampling, predictor_specification="ODE"), dt=0.02)
        s, us = S0.copy(), []
        for _ in range(steps):
            u = np.float32(ctrl.step(s.copy()))
            us.append(u)
            s, _, _ = O.plant_period(s, float(u))
        u_next, u_prev = ctrl.engine.legacy_get_inputs()
        return dict(u=np.array(us, dtype=np.float32), legacy_u=u_next, legacy_u_prev=u_prev)

    M, RA, CEM, GMM, RPGD = (optimizer_mppi_b200, F.optimizer_random_action_b200, F.optimizer_cem_b200, F.optimizer_cem_gmm_b200,
                             F.optimizer_rpgd_b200)
    configs = {
        "mppi_ode_2000x50": lambda: loop(make(M, 2000, 50), 300),
        "mppi_ode_logging": lambda: loop(make(M, 2000, 50, optimizer_logging=True), 20),
        "mppi_gru32_optimal_trajectory": lambda: loop(make(M, 2000, 50, neural=True, calculate_optimal_trajectory=True), 20),
        "mppi_supplied": lambda: loop(make(M, 2000, 50), 20, supplied=True),
        "random_action_640x35": lambda: loop(make(RA, 640, 35), 300),
        "random_action_supplied": lambda: loop(make(RA, 640, 35), 20, supplied=True),
        "cem_200x35": lambda: loop(make(CEM, 200, 35, cem_outer_it=3), 300),
        "cem_warmup": lambda: loop(make(CEM, 200, 35, warmup=True), 300),
        "cem_logging": lambda: loop(make(CEM, 200, 35, optimizer_logging=True), 20),
        "cem_supplied": lambda: loop(make(CEM, 200, 35), 20, supplied=True),
        "cem_gmm_200x35": lambda: loop(make(GMM, 200, 35), 300),
        "cem_gmm_2000x50": lambda: loop(make(GMM, 2000, 50), 120),
        "cem_gmm_supplied": lambda: loop(make(GMM, 200, 35), 20, supplied=True),
        "rpgd_16x35": lambda: loop(make(RPGD, 16, 35), 300),
        "rpgd_2000x50": lambda: loop(make(RPGD, 2000, 50), 300),
        "rpgd_8192x35_torch_path": lambda: loop(make(RPGD, 8192, 35), 20),
        "rpgd_gru32": lambda: loop(make(RPGD, 16, 35, neural=True, calculate_optimal_trajectory=True), 20),
        "rpgd_supplied": lambda: loop(make(RPGD, 16, 35), 20, supplied=True),
    }
    for sampling in ("iid", "random_walk", "uniform", "repeated", "interpolated"):
        configs[f"legacy_{sampling}"] = lambda sampling=sampling: legacy(sampling, 2)
    configs["legacy_interpolated_every_step"] = lambda: legacy("interpolated", 1)
    arrays = {}
    for name, fn in configs.items():
        for k, v in fn().items():
            arrays[f"{name}/{k}"] = v
        print(f"{name}: {len(arrays[name + '/u'])} steps, last u {float(arrays[name + '/u'][-1]):+.7f}", flush=True)
    np.savez(out, **arrays)


def compare(a_path, b_path):
    a, b = np.load(a_path), np.load(b_path)
    bad = sorted(set(a.files) ^ set(b.files))
    by_config = {}
    for k in sorted(set(a.files) & set(b.files)):
        x, y = a[k], b[k]
        same = x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes()
        by_config.setdefault(k.split("/")[0], []).append((k.split("/")[1], same))
        if not same:
            bad.append(k)
    for cfg, fields in by_config.items():
        n_u = a[cfg + "/u"].size
        verdict = "bitwise equal" if all(s for _, s in fields) else "DIFFERS: " + ", ".join(f for f, s in fields if not s)
        print(f"{cfg:32s} {n_u:4d} steps, {len(fields)} arrays ({', '.join(f for f, _ in fields)}): {verdict}")
    print("ALL BITWISE EQUAL" if not bad else f"MISMATCH in {len(bad)} arrays: {bad}")
    return 0 if not bad else 1


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument("--out")
    ap.add_argument("--compare", nargs=2, metavar=("A", "B"))
    args = ap.parse_args()
    sys.exit(compare(*args.compare) if args.compare else run(args.root, args.out))
