"""optimizer_random_action_b200, optimizer_cem_b200 and optimizer_cem_gmm_b200 on a PredictorWrapper configured with the
shipped GRU 2 x 32 model directory, with a non-zero stored hidden state: five solves each against oracle.random_action_step
/ cem_step / cem_gmm_step on the float64 network restatement (tests/plan_neural_oracle.py), teacher-forced per solve (each
solve starts from the oracle's distribution and u_prev), with injected draws; then the optimizers' own draws.  The
engine's stored hidden state is never written."""
import numpy as np
import pytest

from tests.netutil import net_spec_from_golden
from tests.parity import load_golden
from tests.test_gpu_net_grad import GRADMIN, J_BOUND, NETS, _h_after, _state

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

K, T, TP = 200, 35, 0.02
LIMITS = (np.array([-1.0], np.float32), np.array([1.0], np.float32))


class _Gen:
    """The reference's generator calls (tf.random.Generator.normal / uniform) answered from a seeded numpy stream; every
    array handed out is kept in `log`."""

    def __init__(self, seed):
        self.rng, self.log = np.random.default_rng(seed), []

    def normal(self, shape, mean=0.0, stddev=1.0, dtype=None):
        d = (self.rng.normal(0, 1, tuple(shape)) * stddev + mean).astype(np.float32)
        self.log.append(d)
        return torch.from_numpy(d)

    def uniform(self, shape, minval=0.0, maxval=1.0, dtype=None):
        d = self.rng.uniform(minval, maxval, tuple(shape)).astype(np.float32)
        self.log.append(d)
        return torch.from_numpy(d)


def _optimizer(tmp_path, cls, **kw):
    import cartpolesimulation_b200 as cps
    from tests.netutil import write_model_dir
    z, _ = load_golden(NETS["gru32"])
    vp = cps.VariableParameters(target_position=TP, target_equilibrium=1.0, L=0.395, m_pole=0.087)
    cost, predictor = cps.CostFunctionWrapper(), cps.PredictorWrapper()
    predictor.configure(batch_size=K, horizon=T, dt=0.02, variable_parameters=vp,
                        predictor_specification=write_model_dir(str(tmp_path), z))
    cost.configure(batch_size=K, horizon=T, variable_parameters=vp, environment_name="CartPole", computation_library=None,
                   cost_function_specification=GRADMIN)
    opt = cls(predictor=predictor, cost_function=cost, control_limits=LIMITS, seed=3, mpc_horizon=T, num_rollouts=K,
              optimizer_logging=True, **kw)
    opt.configure(num_states=6, num_control_inputs=1, dt=0.02, predictor_specification="neural")
    assert opt.predictor_type == "neural"
    h = _h_after("gru32")
    opt.engine.net_set_state(h)
    return opt, net_spec_from_golden(z), h


def _rel(a, b):
    return float(np.abs(np.asarray(a, np.float64) - b).max() / np.abs(b).max())


@pytest.mark.parametrize("kind", ["random_action", "cem", "cem_gmm"])
def test_forward_optimizer_neural_predictor_wrapper(tmp_path, monkeypatch, kind):
    from cartpolesimulation_b200 import optimizer_forward_b200 as F
    from oracle import oracle as O
    from tests.plan_neural_oracle import neural_plan_cost
    kw = dict(cem_outer_it=3, cem_best_k=40) if kind != "random_action" else {}
    if kind == "cem":
        kw.update(warmup=True, warmup_iterations=5)   # the first solve runs 5 iterations, the others 3
    opt, sp, h = _optimizer(tmp_path, getattr(F, f"optimizer_{kind}_b200"), **kw)
    monkeypatch.setattr(O, "plan_cost", neural_plan_cost(sp, h))
    gen = _Gen(7)
    opt.rng = gen
    ref = None
    for i in range(5):
        s = _state(80 + i)
        opt.optimizer_logging = i % 2 == 0   # the device form with logging, and the host form
        if ref is not None:   # teacher forcing: the solve starts from the oracle's state
            opt.u = np.array(ref["u"], dtype=np.float32)
            if kind == "cem":
                opt.dist_mue, opt.stdev = torch.from_numpy(ref["mean"]), torch.from_numpy(ref["stdev"])
            if kind == "cem_gmm":
                opt.engine.cem_gmm_set_distribution(ref["loc"].T, ref["scale"].T, ref["p1"])
        u_prev = float(np.asarray(opt.u).reshape(-1)[0])
        if kind == "cem":
            mean, stdev = opt.dist_mue.numpy().reshape(-1), opt.stdev.numpy().reshape(-1)
        if kind == "cem_gmm":
            loc, scale, p1 = opt.engine.cem_gmm_get_distribution()
        n0 = len(gen.log)
        u = float(opt.step(s.copy()))
        draws = gen.log[n0:]
        if kind == "random_action":
            assert len(draws) == 1
            ref = O.random_action_step("neural", GRADMIN, s, draws[0][:, :, 0], u_prev, target_position=TP)
            ref["Q"] = draws[0][:, :, 0]   # the plans as drawn
        elif kind == "cem":
            assert len(draws) == (5 if i == 0 else 3)
            ref = O.cem_step("neural", GRADMIN, s, np.stack([d[:, :, 0] for d in draws]), mean, stdev, 40, 0.01, 0.5, u_prev,
                             target_position=TP)
            np.testing.assert_allclose(opt.dist_mue.numpy().reshape(-1), ref["mean"], rtol=0, atol=1e-5)
            np.testing.assert_allclose(opt.stdev.numpy().reshape(-1), ref["stdev"], rtol=0, atol=1e-5)
        else:
            assert len(draws) == 6
            ref = O.cem_gmm_step("neural", GRADMIN, s, np.stack([d[:, :, 0, :] for d in draws[0::2]]),
                                 np.stack([d[:, :, 0] for d in draws[1::2]]), loc.T, scale.T, p1, 40, 0.01, u_prev,
                                 target_position=TP)
            g_loc, g_scale, g_p1 = opt.engine.cem_gmm_get_distribution()
            np.testing.assert_allclose(g_loc.T, ref["loc"], rtol=0, atol=1e-5)
            np.testing.assert_allclose(g_scale.T, ref["scale"], rtol=0, atol=1e-5)
            assert abs(g_p1 - ref["p1"]) < 1e-6
        assert abs(u - ref["u"]) < 2e-6, (i, u, ref["u"])
        if opt.optimizer_logging:   # _log_rollouts on the network: the last iteration's plans and their costs
            Q_log, J_log = opt.logging_values["Q_logged"][:, :, 0], opt.logging_values["J_logged"]
            np.testing.assert_allclose(Q_log, ref["Q"], rtol=0, atol=1e-5)
            assert _rel(J_log, ref["J"]) < (J_BOUND if kind == "random_action" else 2e-5)
            assert opt.logging_values["rollout_trajectories_logged"].shape == (K, T + 1, 6)
        np.testing.assert_array_equal(opt.engine.net_get_state(), h)


@pytest.mark.parametrize("kind", ["random_action", "cem", "cem_gmm"])
def test_forward_optimizer_neural_own_draws(tmp_path, monkeypatch, kind):
    """The optimizers' own device draws (time-major rings): over five solves u is the first input of the cheapest logged
    plan, the logged costs are the float64 restatement's on the logged plans, and the stored hidden state stays."""
    from cartpolesimulation_b200 import optimizer_forward_b200 as F
    from tests.plan_neural_oracle import neural_plan_cost
    opt, sp, h = _optimizer(tmp_path, getattr(F, f"optimizer_{kind}_b200"))
    pc = neural_plan_cost(sp, h)
    for i in range(5):
        s = _state(90 + i)
        u_prev = float(np.asarray(opt.u).reshape(-1)[0])
        u = float(opt.step(s.copy()))
        Q_log, J_log = opt.logging_values["Q_logged"][:, :, 0], opt.logging_values["J_logged"]
        assert np.all(np.isfinite(J_log)) and np.all(np.abs(Q_log) <= 1.0)
        assert u == Q_log[int(np.argsort(J_log, kind="stable")[0]), 0]
        assert _rel(J_log, pc("neural", GRADMIN, s, Q_log, u_prev, target_position=TP)) < J_BOUND
        np.testing.assert_array_equal(opt.engine.net_get_state(), h)
