"""Offline relabelling under RPGD: add_control_along_trajectories around optimizer_rpgd_tf, restated for one file.

oracle.relabel_file is the same loop around optimizer_mppi; here every row is one oracle.rpgd_step (float64).  For a
network, monkeypatch oracle.plan_cost_grad with oracle.net_grad's gradient, as the neural RPGD tests do; the network
takes no physical parameters, so pass L / m_pole only for predictor "ODE"."""
import numpy as np

from oracle import oracle as O


def relabel_file_rpgd(cost_name, T, states, init_draws, resamp_draws, target_position=None, target_equilibrium=None,
                      L=None, m_pole=None, outer_its=4, resamp_per=10, opt_keep_k=12, period=4, sample_stdev=0.5,
                      sample_mean=0.0, lo=-1.0, hi=1.0, **kw):
    """One recorded file (preprocess_data_add_control_along_trajectories.py:108-140): controller.reset() -- plans
    clip(init_draws * sample_stdev + sample_mean) at the inducing points, interpolated (init_draws [K, n_ind]); zero Adam
    moments, iteration count and solve counter; u_prev = 0 (optimizer_rpgd_tf.optimizer_reset, :379-408) -- then one
    optimizer_rpgd_tf.step per row from the recorded state states[r] with the row's attributes ([R] or None) and the
    resampling draws resamp_draws[r] [K - opt_keep_k, n_ind] (read on resampling rows).  Between rows the file keeps its
    plans, moments, Adam iteration count and last control.  L / m_pole change the model of predictor "ODE" (the physics
    vector of plan_cost_grad).  kw: further keywords of oracle.rpgd_step (n, dt, cost_cfg, learning_rate, ...).
    Returns the controls [R] (float32)."""
    states = np.asarray(states, dtype=np.float32)
    R = states.shape[0]
    W = O.interp_matrix(T, period).astype(np.float64)
    Q = np.clip(np.asarray(init_draws, dtype=np.float64) * sample_stdev + sample_mean, lo, hi) @ W
    m, v = np.zeros_like(Q), np.zeros_like(Q)
    iterations, u_prev = 0, 0.0
    out = np.zeros(R, dtype=np.float32)
    for r in range(R):
        rkw = dict(kw)
        if L is not None or m_pole is not None:
            ph = O.physics_vector()
            if L is not None:
                ph[6] = np.float32(L[r])
            if m_pole is not None:
                ph[2] = np.float32(m_pole[r])
            rkw["phys"] = ph
        res = O.rpgd_step(cost_name, states[r], Q, m, v, iterations, r, u_prev, resamp_draw=resamp_draws[r],
                          outer_its=outer_its, resamp_per=resamp_per, opt_keep_k=opt_keep_k, period=period,
                          sample_stdev=sample_stdev, sample_mean=sample_mean, lo=lo, hi=hi,
                          target_position=0.0 if target_position is None else float(target_position[r]),
                          target_equilibrium=1.0 if target_equilibrium is None else float(target_equilibrium[r]), **rkw)
        Q, m, v, iterations = res["Q_next"], res["m"], res["v"], res["iterations"]
        u_prev = float(np.float32(res["u"]))   # template_optimizer.u: the float32 control enters the next cost
        out[r] = np.float32(res["u"])
    return out
