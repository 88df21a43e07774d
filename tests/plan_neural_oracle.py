"""A neural path for oracle.plan_cost, and so for oracle.random_action_step, cem_step and cem_gmm_step, which call it:
predict_and_cost of the forward-only optimizers with predictor_autoregressive_neural (optimizer_random_action_tf.py:42-49,
optimizer_cem_tf.py:57-61: predict_core, then get_trajectory_cost), restated in float64 over oracle/net_grad.py -- every
rollout from the stored hidden state h0, then the gradient plugins' stage costs, J = their sum / (T + 1).  The
restatement is pinned to the reference's network recordings by tests/test_oracle_net_grad.py.

    monkeypatch.setattr(O, "plan_cost", neural_plan_cost(spec, h0))
    O.cem_step("neural", cost, s, eps, mean, stdev, ...)
"""
import numpy as np
import torch

from oracle import net_grad as NG
from oracle import oracle as O


def neural_plan_cost(spec, h0=None, ode_plan_cost=O.plan_cost):
    """A function with oracle.plan_cost's signature: integrator "neural" runs `spec` from h0 ([Htot] or None: zeros);
    any other integrator goes to `ode_plan_cost` (oracle.plan_cost as imported)."""
    h = None if h0 is None else torch.from_numpy(np.asarray(h0, np.float64))

    def plan_cost(integrator, cost_name, s, Q, u_prev=0.0, target_position=0.0, target_equilibrium=1.0, cost_cfg=None,
                  want_traj=False, **kw):
        if integrator != "neural":
            return ode_plan_cost(integrator, cost_name, s, Q, u_prev, target_position, target_equilibrium, cost_cfg=cost_cfg,
                                 want_traj=want_traj, **kw)
        Qt = torch.from_numpy(np.asarray(Q, np.float64).reshape(np.shape(Q)[0], -1))
        traj = NG.predict(spec, np.asarray(s, np.float64).reshape(-1)[:6], Qt, h)
        st = NG.stage_costs(cost_name, traj, Qt, float(u_prev), target_position, target_equilibrium, cost_cfg)
        J = (st.sum(dim=1) / (Qt.shape[1] + 1)).numpy()
        return (J, traj.numpy()) if want_traj else J
    return plan_cost
