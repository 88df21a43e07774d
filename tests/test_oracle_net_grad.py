"""The torch restatement of predict_and_cost with the neural predictor (oracle/net_grad.py), the gradient oracle of
cps_plan_cost_grad for CPS_PREDICTOR_NEURAL, pinned without a GPU: its trajectories against the recordings of the live
reference's torch Sequence (tests/golden/net_*.npz; bound of test_gpu_net.py, measured <= 5e-7 range-relative), its costs
against oracle.trajectory_cost, its autograd gradient against central finite differences in float64."""
import numpy as np
import pytest

from tests.netutil import net_spec_from_golden
from tests.parity import load_golden, record, traj_err

torch = pytest.importorskip("torch")

NETS = ["net_GRU_6IN_32H1_32H2_5OUT_0", "net_GRU_6IN_64H1_64H2_5OUT_0", "net_Dense_6IN_32H1_32H2_5OUT_0"]
COSTS = ["quadratic_boundary_grad_minimal", "quadratic_boundary_grad"]


@pytest.mark.parametrize("name", NETS)
def test_restatement_reproduces_reference_recordings(name):
    from oracle import net_grad as NG
    z, _ = load_golden(name)
    sp = net_spec_from_golden(z)
    Q = torch.from_numpy(z["Q"].astype(np.float64))
    h_upd = z["h_after_updates"].reshape(-1) if "h_after_updates" in z.files else None
    errs = dict(zero_h=max(traj_err(NG.predict(sp, z["s0"], Q).numpy(), z["traj_zero_h"]).values()),
                after_updates=max(traj_err(NG.predict(sp, z["s_after"], Q, h_upd).numpy(), z["traj_after_updates"]).values()),
                rand=max(traj_err(NG.predict(sp, z["s_rand"], Q, h_upd).numpy(), z["traj_rand"]).values()))
    record("net_grad_oracle_vs_reference_golden", name, **errs)
    assert max(errs.values()) < 1e-5


@pytest.mark.parametrize("name", NETS)
@pytest.mark.parametrize("cost", COSTS)
def test_restatement_costs_match_oracle_trajectory_cost(name, cost):
    from oracle import net_grad as NG
    from oracle import oracle as O
    z, _ = load_golden(name)
    traj, Q = z["traj_zero_h"], z["Q"]
    st = NG.stage_costs(cost, torch.from_numpy(traj.astype(np.float64)), torch.from_numpy(Q.astype(np.float64)), 0.2, 0.03, 1.0)
    J = (st.sum(dim=1) / (Q.shape[1] + 1)).numpy()
    Jr = O.trajectory_cost(cost, traj, Q, 0.2, 0.03, 1.0)
    e = float(np.abs(J - Jr).max() / np.abs(Jr).max())
    record("net_grad_oracle_cost_vs_trajectory_cost", f"{name}/{cost}", J=e)
    assert e < 2e-6   # float32 oracle against a float64 sum: measured <= 4.9e-7


@pytest.mark.parametrize("name", NETS)
@pytest.mark.parametrize("cost", COSTS)
def test_autograd_gradient_matches_finite_differences(name, cost):
    from oracle import net_grad as NG
    z, _ = load_golden(name)
    sp = net_spec_from_golden(z)
    rng = np.random.default_rng(3)
    K, T = 3, 6
    Q = np.clip(rng.normal(0, 0.5, (K, T)), -1, 1)
    h0 = z["h_after_updates"].reshape(-1) if "h_after_updates" in z.files else None
    kw = dict(u_prev=-0.3, target_position=0.03, target_equilibrium=1.0, h0=h0)
    if cost == "quadratic_boundary_grad":
        from oracle import oracle as O
        cfg = dict(O.DEFAULT_COST_CONFIG[cost])
        # the kinetic term's target is under stop_gradient, which a finite difference does not see: weight 0 here
        cfg.update({"dd_linear_weight_up": 25.0, "ccrc_weight_up": 1.5, "ekp_weight_up": 0.0})
        kw["cost_cfg"] = cfg
    _, G = NG.plan_cost_grad(sp, cost, z["s0"], Q, **kw)
    eps = 1e-6
    Gfd = np.zeros_like(Q)
    for t in range(T):
        d = np.zeros_like(Q)
        d[:, t] = eps
        Jp = NG.plan_cost(sp, cost, z["s0"], torch.from_numpy(Q + d), **kw).numpy()
        Jm = NG.plan_cost(sp, cost, z["s0"], torch.from_numpy(Q - d), **kw).numpy()
        Gfd[:, t] = (Jp - Jm) / (2 * eps)
    e = float(np.abs(G - Gfd).max() / np.abs(Gfd).max())
    record("net_grad_oracle_vs_finite_differences", f"{name}/{cost}", G=e)
    assert e < 1e-6
