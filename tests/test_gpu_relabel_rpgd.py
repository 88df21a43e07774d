"""Offline relabelling under RPGD (cps_rpgd_fleet_relabel, RpgdFleet.relabel, Relabeller(optimizer="rpgd"),
add_control_along_trajectories with controller_config["rpgd"]): against the closed-loop RpgdFleet's own records (bit for
bit), the float64 oracle (oracle.rpgd_step, oracle.rpgd_relabel.relabel_file_rpgd), the single-experiment kernels with
the row's L / m_pole folded on the host, and itself split over handles, files of different lengths and NaN attributes.
Predictor "ODE" and the GRU / Dense networks of tests/golden/net_*.npz."""
import numpy as np
import pytest
import torch

from oracle import net_grad as NG
from oracle import oracle as O
from oracle.rpgd_relabel import relabel_file_rpgd
from tests.netutil import net_spec_from_golden
from tests.parity import load_golden, record

pytestmark = pytest.mark.gpu

GRADMIN, GRAD = "quadratic_boundary_grad_minimal", "quadratic_boundary_grad"
NETS = {"gru32": "net_GRU_6IN_32H1_32H2_5OUT_0", "dense32": "net_Dense_6IN_32H1_32H2_5OUT_0"}
T, P_IND = 35, 4
STATE_COLS = [1, 2, 4, 5, 6, 7]   # angle, angleD, cos, sin, position, positionD of a record row
STATE = ["angle", "angleD", "angle_cos", "angle_sin", "position", "positionD"]


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def random_states(E, seed):
    from cartpolesimulation_b200.fleet import DataGenConfig, random_initial_state
    rng = np.random.default_rng(seed)
    return np.stack([random_initial_state(rng, DataGenConfig()) for _ in range(E)])


def targets(P, E, seed, flip=None):
    rng = np.random.default_rng(seed)
    tp = np.repeat(rng.uniform(-0.1, 0.1, E)[None], P, axis=0).astype(np.float32)
    te = np.ones((P, E), np.float32)
    if flip is not None:
        te[flip:, 1::2] = -1.0
    return tp, te


def _spec(net):
    z, _ = load_golden(NETS[net])
    return net_spec_from_golden(z)


def _engine_spec(sp):
    d = dict(sp)
    d["weights"] = O.pack_net_weights(sp["net_type"], sp["layers"], sp["out_layer"])
    return d


def fleet_kw(pred):
    return {} if pred == "ode" else dict(integrator="neural", network=_engine_spec(_spec(pred)))


def make(E, K, cost, pred="ode", noise="philox", **kw):
    from cartpolesimulation_b200.fleet import RpgdFleet
    return RpgdFleet(E, num_rollouts=K, mpc_horizon=T, cost=cost, noise=noise, period_interpolation_inducing_points=P_IND,
                     **fleet_kw(pred), **kw)


def recorded_states(rec):
    return rec[:, :, STATE_COLS].contiguous()


@pytest.mark.parametrize("pred", ["ode", "gru32", "dense32"])
@pytest.mark.parametrize("cost", [GRADMIN, GRAD])
@pytest.mark.parametrize("E,K", [(1, 16), (1, 64), (3, 16), (3, 64), (37, 16), (37, 64)])
def test_relabelling_a_closed_loop_run_reproduces_its_controls(pred, cost, E, K):
    """25 closed-loop periods of an RpgdFleet (resampling every 5, target equilibrium flipped at period 8 for the odd
    experiments), then its recorded states and targets relabelled from a reset: with the same seed and offset, and on a
    'supplied' relabeller fed the closed loop's own draws.  The controller sees the same states, so Q_calculated must come
    back bit for bit, and the optimizer state must end where the closed loop's did."""
    P, resamp, seed = 25, 5, 17
    s0 = random_states(E, 3)
    tp, te = targets(P, E, 4, flip=8)
    loop = make(E, K, cost, pred, seed=seed, resamp_per=resamp)
    loop.reset(s0)
    rec = torch.zeros((P, E, 16), device="cuda")
    loop.run(P, cuda(tp), cuda(te), None, rec)
    states = recorded_states(rec)
    want = rec[:, :, 9].clone()
    launches0 = None
    for noise in ("philox", "supplied"):
        rl = make(E, K, cost, pred, noise=noise, seed=seed, resamp_per=resamp)
        if noise == "philox":
            rl.reset(np.zeros((E, 6), np.float32))
            draws = None
        else:
            rl.reset(np.zeros((E, 6), np.float32), init_draws=loop.draws(-1))
            draws = torch.stack([loop.draws(j) for j in range(P)]).contiguous()
        launches0 = rl.engine.launch_count()
        Q = rl.relabel(states, cuda(tp), cuda(te), draws=draws)
        torch.cuda.synchronize()
        assert torch.equal(Q, want), (noise, float((Q - want).abs().max()))
        pl, pr = loop.plans(), rl.plans()
        for k in ("Q", "m", "v", "ages"):
            np.testing.assert_array_equal(pl[k], pr[k])
        assert pl["adam_iterations"] == pr["adam_iterations"] and pl["solves"] == pr["solves"] == P
        np.testing.assert_array_equal(rl.states(), states[-1].cpu().numpy())   # the last row's recorded states
        assert rl.period == P
        per_row = (3 + (4 if pred == "ode" else 2) * 4) * P   # launches per row as per period, whatever E
        assert rl.engine.launch_count() - launches0 == per_row


def _row_states(R, E, seed):
    rng = np.random.default_rng(seed)
    ang = rng.uniform(-np.pi, np.pi, (R, E))
    return np.stack([ang, rng.uniform(-3, 3, (R, E)), np.cos(ang), np.sin(ang), rng.uniform(-0.15, 0.15, (R, E)),
                     rng.uniform(-0.5, 0.5, (R, E))], axis=2).astype(np.float32)


def _oracle_grad(sp):
    def f(cost_name, s, Q, u_prev, dtype=np.float64, phys=None, **kw):   # the network takes no physical parameters
        return NG.plan_cost_grad(sp, cost_name, s, Q, u_prev, dtype=torch.float32 if dtype == np.float32 else torch.float64,
                                 **kw)
    return f


@pytest.mark.parametrize("pred,cost,E,K", [("ode", GRADMIN, 3, 16), ("ode", GRAD, 3, 16), ("ode", GRADMIN, 5, 64),
                                           ("gru32", GRADMIN, 3, 16), ("dense32", GRAD, 3, 16)])
def test_relabel_rows_match_oracle_teacher_forced(monkeypatch, pred, cost, E, K):
    """Each row starts oracle.rpgd_step from the relabeller's own optimizer state (plans, moments, ages, counters, u_prev)
    with the row's recorded state, targets and -- predictor "ODE" -- its own L / m_pole (the oracle's physics vector).
    12 rows, resampling at 0 and 10.  Bounds, the near-tie rule and the float32 allowance of quadratic_boundary_grad are
    those of the closed-loop fleet tests."""
    R, resamp = 12, 10
    if pred != "ode":
        monkeypatch.setattr(O, "plan_cost_grad", _oracle_grad(_spec(pred)))
    fl = make(E, K, cost, pred, noise="supplied", resamp_per=resamp)
    keep, n_ind = fl.opt_keep_k, fl.n_ind
    rng = np.random.default_rng(5)
    init = rng.standard_normal((E, K, n_ind)).astype(np.float32)
    draws = rng.standard_normal((R, E, K - keep, n_ind)).astype(np.float32)
    states = _row_states(R, E, 6)
    tp, te = targets(R, E, 7, flip=4)
    Lr = rng.uniform(0.25, 0.55, (R, E)).astype(np.float32)
    mr = rng.uniform(0.05, 0.12, (R, E)).astype(np.float32)
    fl.reset(np.zeros((E, 6), np.float32), init_draws=cuda(init))
    worst = dict(u=0.0, Q_next=0.0)
    order_skips = n_checked = 0
    for r in range(R):
        st = fl.plans()
        _, u_prev = fl.states(with_u_prev=True)
        J_out = torch.zeros((1, E, K), device="cuda")
        Q = fl.relabel(cuda(states[r:r + 1]), cuda(tp[r:r + 1]), cuda(te[r:r + 1]), cuda(Lr[r:r + 1]), cuda(mr[r:r + 1]),
                       cuda(draws[r:r + 1]), J_out=J_out).cpu().numpy()[0]
        nxt = fl.plans()
        _, u_next = fl.states(with_u_prev=True)
        J_out = J_out.cpu().numpy()[0]
        for e in range(E):
            n_checked += 1
            okw = dict(resamp_draw=draws[r, e], outer_its=4, resamp_per=resamp, opt_keep_k=keep, period=P_IND,
                       target_position=float(tp[r, e]), target_equilibrium=float(te[r, e]))
            if pred == "ode":
                okw["phys"] = O.physics_vector(L=float(Lr[r, e]), m_pole=float(mr[r, e]))
            args = (cost, states[r, e], st["Q"][e], st["m"][e], st["v"][e], st["adam_iterations"], r, float(u_prev[e]))
            ref = O.rpgd_step(*args, **okw)
            r32 = O.rpgd_step(*args, dtype=np.float32, **okw) if cost == GRAD else ref
            floor = lambda key: 2.0 * np.abs(r32[key] - ref[key])
            assert u_next[e] == Q[e]
            order = np.argsort(J_out[e], kind="stable")
            eu = abs(float(Q[e]) - float(ref["Q_opt"][order[0], 0]))
            assert eu < 1e-4 + float(floor("Q_opt")[order[0], 0]), (r, e, eu)
            J_ref = ref["J"]
            tol = 1e-5 * float(np.abs(J_ref).max()) + 2.0 * np.abs(r32["J"] - J_ref) + 1e-4 * np.abs(J_ref)
            same = np.array_equal(order[:keep], ref["best"]) if r % resamp == 0 else order[0] == ref["best"][0]
            if not same:   # a near-tie: the oracle's own costs of the two orders agree within rounding
                assert np.all(np.diff(J_ref[order]) > -(tol[order][1:] + tol[order][:-1])), (r, e)
                order_skips += 1
                continue
            dQ = np.abs(nxt["Q"][e] - ref["Q_next"])
            assert np.all(dQ <= 2e-4 + floor("Q_next")), (r, e, float(dQ.max()))
            worst.update(u=max(worst["u"], eu), Q_next=max(worst["Q_next"], float(dQ.max())))
    record("rpgd_relabel_oracle", f"{pred}/{cost}/E{E}/K{K}", order_skips=order_skips, **worst)
    assert order_skips <= max(1, n_checked // 10), (order_skips, n_checked)


def test_device_fold_equals_host_fold():
    """L / m_pole arrays holding the handle's own values give the run with NULL arrays bit for bit (labels, plans,
    moments); and each row's labels with varying L / m_pole equal Engine.rpgd_grad_step x 4 + plan_cost + rpgd_finish on
    an engine whose variable parameters (folded on the host) are that row's."""
    from cartpolesimulation_b200.core import Engine
    E, K, R, cost = 4, 16, 3, GRAD
    states = _row_states(R, E, 9)
    tp, te = targets(R, E, 10, flip=1)
    runs = []
    for L, mp in ((None, None), (np.full((R, E), 0.395, np.float32), np.full((R, E), 0.087, np.float32))):
        fl = make(E, K, cost, seed=3)
        fl.reset(np.zeros((E, 6), np.float32))
        Q = fl.relabel(cuda(states), cuda(tp), cuda(te), None if L is None else cuda(L), None if mp is None else cuda(mp))
        runs.append((Q.cpu().numpy(), fl.plans()))
    np.testing.assert_array_equal(runs[0][0], runs[1][0])
    for k in ("Q", "m", "v", "ages"):
        np.testing.assert_array_equal(runs[0][1][k], runs[1][1][k])

    rng = np.random.default_rng(11)
    Lr = rng.uniform(0.25, 0.55, (R, E)).astype(np.float32)
    mr = rng.uniform(0.05, 0.12, (R, E)).astype(np.float32)
    fl = make(E, K, cost, seed=3)
    fl.reset(np.zeros((E, 6), np.float32))
    eng = Engine(K, T, cost=cost, interp_period=P_IND)
    for r in range(R):
        st = fl.plans()
        _, u_prev = fl.states(with_u_prev=True)
        Q = fl.relabel(cuda(states[r:r + 1]), cuda(tp[r:r + 1]), cuda(te[r:r + 1]), cuda(Lr[r:r + 1]),
                       cuda(mr[r:r + 1])).cpu().numpy()[0]
        for e in range(E):
            eng.set_variable_parameters(target_position=float(tp[r, e]), target_equilibrium=float(te[r, e]),
                                        L=float(Lr[r, e]), m_pole=float(mr[r, e]))
            eng.rpgd_reset()
            m, v, _ = eng.rpgd_adam_state()
            m.copy_(torch.from_numpy(st["m"][e]).cuda())
            v.copy_(torch.from_numpy(st["v"][e]).cuda())
            eng.rpgd_set_iterations(st["adam_iterations"])
            Qe = torch.from_numpy(st["Q"][e].copy()).cuda()
            s_dev = cuda(states[r, e])
            for _ in range(4):
                eng.rpgd_grad_step(s_dev, Qe, float(u_prev[e]), 0.05, 0.9, 0.999, 1e-8, 5.0)
            J = eng.plan_cost(s_dev, Qe, u_prev=float(u_prev[e]))[0]
            ages = torch.from_numpy(st["ages"][e].copy()).cuda()
            u_nom = eng.rpgd_finish(J, Qe, None, fl.opt_keep_k, 1, ages)
            assert u_nom[0] == Q[e], (r, e, float(u_nom[0]), float(Q[e]))


def test_split_over_relabellers_equals_one():
    from cartpolesimulation_b200.relabel import Relabeller
    E, K, R = 5, 16, 14
    states = _row_states(R, E, 12)
    tp, te = targets(R, E, 13, flip=6)
    Lr = np.random.default_rng(14).uniform(0.25, 0.55, (R, E)).astype(np.float32)
    kw = dict(optimizer="rpgd", num_rollouts=K, mpc_horizon=T, period_interpolation_inducing_points=P_IND, resamp_per=4,
              seed=21, cost=GRAD)
    whole = Relabeller(E, **kw)
    whole.reset()
    Q = whole.relabel(states, tp, te, Lr, chunk_rows=5)
    parts = []
    for lo, hi in ((0, 2), (2, 5)):
        rl = Relabeller(hi - lo, file_offset=lo, **kw)
        rl.reset()
        parts.append(rl.relabel(states[:, lo:hi], tp[:, lo:hi], te[:, lo:hi], Lr[:, lo:hi]))
    np.testing.assert_array_equal(Q, np.concatenate(parts, axis=1))


def test_nan_attribute_stays_in_its_file():
    E, K, R = 4, 16, 12
    states = _row_states(R, E, 15)
    tp, te = targets(R, E, 16)
    out = []
    for bad in (False, True):
        t = tp.copy()
        if bad:
            t[3:, 2] = np.nan
        fl = make(E, K, GRAD, seed=8, resamp_per=5)
        fl.reset(np.zeros((E, 6), np.float32))
        out.append(fl.relabel(cuda(states), cuda(t), cuda(te)).cpu().numpy())
        if bad:
            assert fl.nonfinite_costs() > 0
    np.testing.assert_array_equal(out[0][:, [0, 1, 3]], out[1][:, [0, 1, 3]])
    np.testing.assert_array_equal(out[0][:3, 2], out[1][:3, 2])


@pytest.mark.parametrize("pred", ["gru32", "dense32"])
def test_neural_labels_do_not_depend_on_L_or_m_pole(pred):
    E, K, R = 3, 16, 8
    states = _row_states(R, E, 17)
    rng = np.random.default_rng(18)
    out = []
    for L, mp in ((None, None), (rng.uniform(0.2, 0.6, (R, E)), rng.uniform(0.05, 0.12, (R, E)))):
        fl = make(E, K, GRADMIN, pred, seed=2)
        fl.reset(np.zeros((E, 6), np.float32))
        out.append(fl.relabel(cuda(states), None, None, None if L is None else cuda(L),
                              None if mp is None else cuda(mp)).cpu().numpy())
    np.testing.assert_array_equal(out[0], out[1])


def test_files_of_different_lengths_keep_their_own_labels():
    import pandas as pd
    from cartpolesimulation_b200.relabel import Relabeller, add_control_along_trajectories
    rows, E, K = (9, 4, 6), 3, 16
    dfs = []
    for f, n in enumerate(rows):
        s = _row_states(n, 1, 30 + f)[:, 0]
        d = pd.DataFrame(s, columns=STATE)
        d["target_position"] = np.linspace(-0.05, 0.05, n)
        d["L"] = np.linspace(0.3, 0.5, n)
        dfs.append(d)
    cfg = dict(state_components=STATE, environment_attributes_dict={"target_position": "target_position", "L": "L"})
    kw = dict(optimizer="rpgd", num_rollouts=K, mpc_horizon=T, period_interpolation_inducing_points=P_IND, resamp_per=3,
              seed=4)
    together = add_control_along_trajectories(dfs, cfg, relabeller=Relabeller(E, **kw), save_output_only=True)
    for f in range(E):
        alone = add_control_along_trajectories(dfs[f], cfg, relabeller=Relabeller(1, file_offset=f, **kw),
                                               save_output_only=True)
        assert len(together[f]) == rows[f]
        np.testing.assert_array_equal(together[f].to_numpy(), alone.to_numpy())


class _Capture:
    """Wraps a Relabeller: records what add_control_along_trajectories feeds it, or answers with given controls."""

    def __init__(self, rl, answer=None):
        self.rl, self.E, self.optimizer, self.answer, self.calls = rl, rl.E, "rpgd", answer, []

    def reset(self, period=0):
        self.rl.reset(period)

    def relabel(self, states, tp, te, L, mp, noise=None):
        self.calls.append(dict(states=states, tp=tp, te=te, L=L, mp=mp))
        return self.rl.relabel(states, tp, te, L, mp) if self.answer is None else self.answer


@pytest.mark.parametrize("mode", ["plain", "random", "integrate", "differentiate"])
def test_add_control_along_trajectories_rpgd_matches_oracle(mode):
    """Plain rows, `_random_uniform_`, Monte-Carlo `_integrate_` and `_differentiate_` of an rpgd block against a per-file
    loop of oracle.relabel_file_rpgd fed the relabeller's Philox draws (float64; the labels after the same averaging /
    Savitzky-Golay step)."""
    import pandas as pd
    from cartpolesimulation_b200.relabel import Relabeller, add_control_along_trajectories
    E, K, rows = 2, 16, (5, 3)
    dfs = []
    for f, n in enumerate(rows):
        d = pd.DataFrame(_row_states(n, 1, 40 + f)[:, 0], columns=STATE)
        d["target_position"] = np.linspace(-0.05, 0.05, n)
        d["target_equilibrium"] = 1.0
        d["L"] = np.linspace(0.35, 0.45, n)
        dfs.append(d)
    env = {"target_position": "target_position", "target_equilibrium": "target_equilibrium", "L": "L"}
    extra = {}
    if mode == "random":
        env["L"] = "L_random_uniform_0.3_0.5"
    elif mode == "integrate":
        env["L"] = "L_integrate_0.3_0.5_"
        extra = dict(integration_num_evals=4)
    elif mode == "differentiate":
        env["L"] = "L_differentiate_"
    rpgd = dict(num_rollouts=K, mpc_horizon=T, period_interpolation_inducing_points=P_IND, resamp_per=3, seed=6,
                outer_its=4, rtol=1e-3, optimizer_logging=False, calculate_optimal_trajectory=False)
    cfg = dict(state_components=STATE, environment_attributes_dict=env, rpgd=rpgd)
    from cartpolesimulation_b200.relabel import rpgd_relabeller_keywords
    rl = Relabeller(E, optimizer="rpgd", **rpgd_relabeller_keywords(rpgd))
    cap = _Capture(rl)
    got = add_control_along_trajectories(dfs, cfg, "Q", relabeller=cap, seed=1, save_output_only=True, **extra)
    c = cap.calls[0]
    n = c["states"].shape[0]
    keep = rl.fleet.opt_keep_k
    init = rl.fleet.draws(-1).cpu().numpy()
    draws = np.stack([rl.fleet.draws(j).cpu().numpy() for j in range(n)])
    Q_ref = np.zeros((n, E), np.float32)
    for e in range(E):
        Q_ref[:, e] = relabel_file_rpgd(GRADMIN, T, c["states"][:, e], init[e], draws[:, e], c["tp"][:, e], c["te"][:, e],
                                        c["L"][:, e], None, resamp_per=3, opt_keep_k=keep, period=P_IND)
    ref = add_control_along_trajectories(dfs, cfg, "Q", relabeller=_Capture(rl, answer=Q_ref), seed=1,
                                         save_output_only=True, **extra)
    worst = 0.0
    for f in range(E):
        assert got[f].shape == ref[f].shape and list(got[f].columns) == list(ref[f].columns)
        d = np.abs(got[f].to_numpy() - ref[f].to_numpy())
        # the derivative columns divide the control's error by the five-point stencil's step (0.5e-3)
        scale = np.array([1.0 / 0.5e-3 if "_dL" in col and not col.startswith("_") else 1.0 for col in got[f].columns]) \
            if mode == "differentiate" else 1.0
        worst = max(worst, float((d / scale).max()))
        assert np.all(d <= 1e-6 * scale), (f, float((d / scale).max()))   # measured <= 2.1e-7 on a B200
    record("rpgd_relabel_add_control", mode, u=worst)


def test_rejections():
    import pandas as pd
    from cartpolesimulation_b200.relabel import Relabeller, add_control_along_trajectories
    rl = Relabeller(2, optimizer="rpgd")
    with pytest.raises(NotImplementedError):
        rl.relabel_device(torch.zeros((1, 2, 6), device="cuda"), active=torch.ones((1, 2), dtype=torch.int32, device="cuda"))
    with pytest.raises(ValueError):
        rl.fleet.relabel(torch.zeros((1, 3, 6), device="cuda"))
    with pytest.raises(ValueError):
        rl.fleet.relabel(torch.zeros((2, 2, 6), device="cuda"), Q_out=torch.zeros((1, 2), device="cuda"))
    with pytest.raises(RuntimeError):   # CPS_ERR_NOT_CONFIGURED before reset()
        rl.fleet.relabel(torch.zeros((1, 2, 6), device="cuda"))
    df = pd.DataFrame(np.zeros((2, 7)), columns=STATE + ["L"])
    cfg = dict(state_components=STATE, environment_attributes_dict={"L": "L_integrate_0.3_0.5_"}, rpgd={})
    with pytest.raises(NotImplementedError):
        add_control_along_trajectories([df, df], cfg, integration_method="nquad", relabeller=rl)
    assert rl.engine.lib.cps_rpgd_fleet_relabel(rl.engine._h, 1, None, None, None, None, None, None, None, None) == 1
