"""CPU tests of the host side of relabelling under RPGD (cartpolesimulation_b200/relabel.py): the argument checks that
run before any device work, the rpgd block's keywords, the row expansion handed to the device (recorded), and the
oracle's per-file loop."""
import numpy as np
import pandas as pd
import pytest

from cartpolesimulation_b200 import relabel as RL
from oracle import oracle as O
from oracle.rpgd_relabel import relabel_file_rpgd
from tests.test_relabel_host_cpu import Recorder

STATE = ["angle", "angleD", "angle_cos", "angle_sin", "position", "positionD"]


def _df(n, seed=0):
    rng = np.random.default_rng(seed)
    d = pd.DataFrame(rng.uniform(-0.1, 0.1, (n, 6)), columns=STATE)
    d["L"] = np.linspace(0.3, 0.5, n)
    return d


def test_mppi_and_rpgd_together_raise():
    cfg = dict(state_components=STATE, environment_attributes_dict={"L": "L"}, mppi={}, rpgd={})
    with pytest.raises(ValueError):
        RL.add_control_along_trajectories([_df(3)], cfg, relabeller=Recorder(1))


def test_nquad_under_rpgd_raises_before_any_step():
    rec = Recorder(2)
    cfg = dict(state_components=STATE, environment_attributes_dict={"L": "L_integrate_0.3_0.5_"}, rpgd={})
    with pytest.raises(NotImplementedError):
        RL.add_control_along_trajectories([_df(3), _df(2)], cfg, integration_method="nquad", relabeller=rec)
    assert rec.resets == 0 and not rec.calls


@pytest.mark.parametrize("env,extra,ev", [({"L": "L"}, {}, 1), ({"L": "L_integrate_0.3_0.5_"}, dict(integration_num_evals=4), 4),
                                          ({"L": "L_differentiate_"}, {}, 5)])
def test_rpgd_block_feeds_the_rows_mppi_would(env, extra, ev):
    """The expansion does not depend on the optimizer: the same rows, states and attributes reach the relabeller."""
    calls = []
    for opt in ("mppi", "rpgd"):
        rec = Recorder(2)
        cfg = dict(state_components=STATE, environment_attributes_dict=env, **{opt: {}})
        RL.add_control_along_trajectories([_df(4, 1), _df(3, 2)], cfg, relabeller=rec, seed=3, **extra)
        calls.append(rec.calls[0])
    assert calls[0]["states"].shape == (4 * ev, 2, 6)
    for k in ("states", "L"):
        np.testing.assert_array_equal(calls[0][k], calls[1][k])


def test_rpgd_block_keywords():
    block = dict(seed=None, mpc_horizon=35, num_rollouts=16, outer_its=4, sample_stdev=0.5, sample_mean=0.0,
                 sample_whole_control_space=False, uniform_dist_min=-0.8, uniform_dist_max=0.8, resamp_per=10,
                 period_interpolation_inducing_points=4, SAMPLING_DISTRIBUTION="normal", shift_previous=1, warmup=False,
                 warmup_iterations=250, learning_rate=0.05, opt_keep_k_ratio=0.75, gradmax_clip=5, rtol=1.0e-3,
                 adam_beta_1=0.9, adam_beta_2=0.999, adam_epsilon=1.0e-08, optimizer_logging=False,
                 calculate_optimal_trajectory=False, integrator="ODE", cost="quadratic_boundary_grad")
    kw = RL.rpgd_relabeller_keywords(block)
    for k in ("seed", "rtol", "optimizer_logging", "calculate_optimal_trajectory", "sample_whole_control_space",
              "uniform_dist_min", "uniform_dist_max"):
        assert k not in kw
    assert kw["mpc_horizon"] == 35 and kw["integrator"] == "ODE" and kw["cost"] == "quadratic_boundary_grad"
    assert RL.rpgd_relabeller_keywords(dict(seed=5))["seed"] == 5


@pytest.mark.parametrize("kw", [dict(optimizer="cem"), dict(optimizer="rpgd", horizon=35),
                                dict(optimizer="rpgd", interp_period=4), dict(optimizer="rpgd", mppi={}),
                                dict(optimizer="rpgd", no_pairs=True)])
def test_relabeller_argument_checks(kw):
    with pytest.raises(ValueError):
        RL.Relabeller(2, **kw)


def test_rpgd_keywords_without_the_switch_raise():
    with pytest.raises(TypeError):
        RL.Relabeller(2, outer_its=4)


def test_oracle_relabel_file_rpgd_is_rpgd_step_row_by_row():
    """relabel_file_rpgd = optimizer_reset + rpgd_step per row with the row's physics; the handle's own L / m_pole give the
    run without attributes exactly."""
    K, R, keep, p = 16, 4, 12, 4
    rng = np.random.default_rng(0)
    n_ind = O.num_inducing(35, p)
    init = rng.standard_normal((K, n_ind))
    draws = rng.standard_normal((R, K - keep, n_ind))
    s = rng.uniform(-0.2, 0.2, (R, 6)).astype(np.float32)
    tp = np.full(R, 0.02)
    u0 = relabel_file_rpgd("quadratic_boundary_grad_minimal", 35, s, init, draws, tp, resamp_per=2, period=p)
    u1 = relabel_file_rpgd("quadratic_boundary_grad_minimal", 35, s, init, draws, tp, L=np.full(R, 0.395),
                           m_pole=np.full(R, 0.087), resamp_per=2, period=p)
    np.testing.assert_array_equal(u0, u1)
    Q = np.clip(init * 0.5, -1, 1) @ O.interp_matrix(35, p).astype(np.float64)
    m = v = np.zeros_like(Q)
    it, up = 0, 0.0
    for r in range(R):
        res = O.rpgd_step("quadratic_boundary_grad_minimal", s[r], Q, m, v, it, r, up, resamp_draw=draws[r],
                          resamp_per=2, period=p, target_position=0.02)
        Q, m, v, it, up = res["Q_next"], res["m"], res["v"], res["iterations"], float(np.float32(res["u"]))
        assert u0[r] == np.float32(res["u"])
    u2 = relabel_file_rpgd("quadratic_boundary_grad_minimal", 35, s, init, draws, tp, L=np.full(R, 0.3), resamp_per=2,
                           period=p)
    assert not np.array_equal(u0, u2)
