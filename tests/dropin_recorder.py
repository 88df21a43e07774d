"""Stand-in for cartpolesimulation_b200's Engine in the drop-in tests: records how optimizer_mppi_b200 drives the C-ABI
layer (what it extracts from the controller's wrapper objects), without a GPU; and the assertions both drop-in tests make
on that record."""
import numpy as np


def recording_engine(calls):
    """An Engine class whose instances append (name, arguments) to `calls`; mppi_step_host returns 0.25."""

    class FakeEngine:
        def __init__(self, **kw):
            import torch
            calls.append(("create", {k: v for k, v in kw.items()}))
            self.device = torch.device("cpu")
            self.K, self.T, self.p = kw["num_rollouts"], kw["horizon"], kw["interp_period"]
            self.n_ind = int(np.ceil((self.T - 1) / self.p)) + 1
            self.u_nom = np.zeros(self.T, np.float32)

        def set_cost_params(self, v):
            calls.append(("cost_params", [float(x) for x in v]))

        def set_mppi_params(self, *a):
            calls.append(("mppi_params", [float(x) for x in a]))

        def set_variable_parameters(self, *a):
            calls.append(("variable", [float(x) for x in a]))

        def mppi_reset(self, v):
            calls.append(("reset", float(v)))

        def mppi_step_host(self, s, noise, layout, u_prev):
            calls.append(("step", dict(s=[float(x) for x in s], noise_shape=list(noise.shape), layout=int(layout),
                                       u_prev=float(u_prev))))
            return 0.25

        def get_u_nom(self):
            return self.u_nom

    return FakeEngine


def check_record(r):
    """What controller_mpc's configuration (optimizer mppi-b200, ODE predictor, quadratic_boundary_grad_minimal with
    ep_weight_up = 41.5, K = 2000, T = 50), two controller.step calls and a controller_reset must make reach the Engine."""
    assert r["optimizer_name"] == "mppi-b200"
    assert (r["num_rollouts"], r["mpc_horizon"]) == (2000, 50)
    calls = r["calls"]
    create = [c for c in calls if c[0] == "create"][0][1]
    assert create["integrator"] == "ODE" and create["substeps"] == 10 and create["cost"] == "quadratic_boundary_grad_minimal"
    assert create["num_rollouts"] == 2000 and create["horizon"] == 50 and create["interp_period"] == 10
    assert abs(create["dt"] - 0.02) < 1e-12
    # weights were read from the cost plugin's own YAML block (edited ep_weight_up = 41.5)
    cost = [c for c in calls if c[0] == "cost_params"][0][1]
    np.testing.assert_allclose(cost, [10.0, 10000.0, 41.5, 1.0, 5.0, 1.0, 0.85], rtol=1e-6)
    mp = [c for c in calls if c[0] == "mppi_params"][0][1]
    np.testing.assert_allclose(mp, [1.0, 1.0, 100.0, 1000.0, 0.03, -1.0, 1.0], rtol=1e-6)
    # variable parameters: re-read every step from the controller's VariableParameters, uploaded only on change
    var = [c[1] for c in calls if c[0] == "variable"]
    assert len(var) == 1
    np.testing.assert_allclose(var[0], [0.1, -1.0, 0.3, 0.1], rtol=1e-6)
    steps = [c[1] for c in calls if c[0] == "step"]
    assert len(steps) == 2
    assert steps[0]["u_prev"] == 0.0 and steps[1]["u_prev"] == 0.25      # last RETURNED control
    assert steps[0]["noise_shape"] == [6, 2000] and steps[0]["layout"] == 1
    np.testing.assert_allclose(steps[0]["s"][:2], [3.1, 0.1], rtol=1e-6)
    assert r["u1"] == 0.25 and r["u_type"] == "ndarray"
    resets = [c for c in calls if c[0] == "reset"]
    assert len(resets) == 2 and resets[-1][1] == 0.0                   # configure + controller_reset
