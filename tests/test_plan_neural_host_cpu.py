"""Host-side refusals of the forward-only planners on the neural predictor that need no GPU: a fleet with
integrator="neural" and no network, and a drop-in optimizer handed a bare "neural" predictor with no network to take
over, raise NotImplementedError before any device work."""
import numpy as np
import pytest


@pytest.mark.parametrize("cls", ["CemFleet", "CemGmmFleet", "RandomActionFleet"])
def test_neural_fleet_without_network_is_refused(cls):
    from cartpolesimulation_b200 import fleet
    with pytest.raises(NotImplementedError):
        getattr(fleet, cls)(4, integrator="neural")
    with pytest.raises(ValueError):
        getattr(fleet, cls)(4, integrator="ODE", network={})


@pytest.mark.parametrize("cls", ["optimizer_cem_b200", "optimizer_cem_gmm_b200", "optimizer_random_action_b200"])
def test_bare_neural_predictor_is_refused(cls):
    from cartpolesimulation_b200 import optimizer_forward_b200 as F
    assert "neural" in getattr(F, cls).PREDICTORS
    opt = getattr(F, cls)(predictor="neural", cost_function="quadratic_boundary_grad_minimal",
                          control_limits=(np.array([-1.0], np.float32), np.array([1.0], np.float32)), num_rollouts=8,
                          mpc_horizon=5)
    with pytest.raises(NotImplementedError):
        opt.configure(num_states=6, num_control_inputs=1, dt=0.02)
    assert opt.engine is None
