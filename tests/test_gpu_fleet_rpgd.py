"""RPGD fleets (cps_rpgd_fleet_*, fleet.RpgdFleet): E closed-loop experiments under the reference's default optimizer, against
the float64 oracle (oracle.rpgd_step + oracle.plant_period), the single-experiment kernels (Engine.rpgd_grad_step /
Engine.plan_cost), their own Philox draws, a split over two fleets and optimizer_rpgd_b200."""
import csv
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import oracle as O
from tests.parity import close_except_few, record

pytestmark = pytest.mark.gpu

GRADMIN, GRAD = "quadratic_boundary_grad_minimal", "quadratic_boundary_grad"
RANGES = np.array([np.pi, 18.38, 1.0, 1.0, 0.198, 1.125], dtype=np.float64)  # the reference's normalisation ranges
T, P_IND = 35, 4


def state_err(a, b):
    d = np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64))
    d[..., 0] = np.minimum(d[..., 0], 2 * np.pi - d[..., 0])
    return float((d / RANGES).max())


def random_states(E, seed):
    from cartpolesimulation_b200.fleet import DataGenConfig, random_initial_state
    rng = np.random.default_rng(seed)
    return np.stack([random_initial_state(rng, DataGenConfig()) for _ in range(E)])


def targets(P, E, seed, flip=None):
    """tp [P, E] within the track, te [P, E] = +1, or -1 from period `flip` on for the odd experiments."""
    rng = np.random.default_rng(seed)
    tp = np.repeat(rng.uniform(-0.1, 0.1, E)[None], P, axis=0).astype(np.float32)
    te = np.ones((P, E), np.float32)
    if flip is not None:
        te[flip:, 1::2] = -1.0
    return tp, te


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def make(E, K, cost, noise="supplied", **kw):
    from cartpolesimulation_b200.fleet import RpgdFleet
    return RpgdFleet(E, num_rollouts=K, mpc_horizon=T, cost=cost, noise=noise,
                     period_interpolation_inducing_points=P_IND, **kw)


@pytest.mark.parametrize("cost,E,K,flip,checked", [(GRADMIN, 1, 16, None, None), (GRAD, 3, 16, 5, None),
                                                    (GRAD, 37, 64, 4, 2)])
def test_rpgd_fleet_matches_oracle_teacher_forced(cost, E, K, flip, checked):
    """Every period starts the oracle from the fleet's own state (plans, moments, ages, counters, u_prev, plant state):
    12 periods, resampling at 0 and 10.  `checked`: experiments compared per period (rotating), None: all of them."""
    P, resamp = 12, 10
    fl = make(E, K, cost, resamp_per=resamp)
    keep, n_ind = fl.opt_keep_k, fl.n_ind
    rng = np.random.default_rng(7)
    init = rng.standard_normal((E, K, n_ind)).astype(np.float32)
    draws = rng.standard_normal((P, E, K - keep, n_ind)).astype(np.float32)
    tp, te = targets(P, E, 3, flip)
    fl.reset(random_states(E, 11), init_draws=cuda(init))
    W = O.interp_matrix(T, P_IND).astype(np.float64)
    np.testing.assert_allclose(fl.plans()["Q"], np.clip(init.astype(np.float64) * 0.5, -1, 1) @ W, rtol=0, atol=1e-6)
    d_draws, d_tp, d_te = cuda(draws), cuda(tp), cuda(te)
    worst = dict(Q_opt=0.0, J=0.0, u=0.0, Q_next=0.0, m=0.0, v=0.0, state=0.0)
    order_skips = floor_used = n_checked = 0
    for j in range(P):
        st = fl.plans()
        s, u_prev = fl.states(with_u_prev=True)
        rec, J_out, Q_opt = (torch.zeros(shape, device="cuda") for shape in ((1, E, 16), (1, E, K), (1, E, K, T)))
        fl.run(1, d_tp[j:j + 1].contiguous(), d_te[j:j + 1].contiguous(), d_draws[j:j + 1].contiguous(), rec, J_out, Q_opt)
        nxt = fl.plans()
        s_next, u_next = fl.states(with_u_prev=True)
        rec, J_out, Q_opt = rec.cpu().numpy()[0], J_out.cpu().numpy()[0], Q_opt.cpu().numpy()[0]
        assert st["solves"] == j and nxt["solves"] == j + 1
        assert nxt["adam_iterations"] == st["adam_iterations"] + 4
        exps = range(E) if checked is None else [(j * checked + i) % E for i in range(checked)]
        for e in exps:
            n_checked += 1
            args = (cost, s[e], st["Q"][e], st["m"][e], st["v"][e], st["adam_iterations"], j, float(u_prev[e]))
            okw = dict(resamp_draw=draws[j, e], outer_its=4, resamp_per=resamp, opt_keep_k=keep, period=P_IND,
                       target_position=float(tp[j, e]), target_equilibrium=float(te[j, e]))
            ref = O.rpgd_step(*args, **okw)
            # the same step with the gradient evaluated in float32: where quadratic_boundary_grad is ill-conditioned
            # (see the costs below) float32 arithmetic itself moves the result, and each entry is allowed twice that spread
            r32 = O.rpgd_step(*args, dtype=np.float32, **okw)
            few = dict(max_outliers=2, outlier_atol=2e-3) if cost == GRAD else {}

            def close(got, key, atol):
                d = np.abs(np.asarray(got, np.float64) - ref[key])
                floor = 2.0 * np.abs(r32[key] - ref[key])
                bad = d > atol + floor   # as close_except_few, with the float32 spread added to both bounds
                ok = int(bad.sum()) <= few.get("max_outliers", 0) and bool(
                    (d[bad] <= few.get("outlier_atol", atol) + floor[bad]).all())
                return ok, float(d.max())
            ok, eQ = close(Q_opt[e], "Q_opt", 2e-4)
            assert ok, eQ
            # the costs of the fleet's own improved plans (float32 plans that differ from the oracle's by the Adam steps'
            # rounding), evaluated in float64.  Fast-spinning states with target_equilibrium = -1 make quadratic_boundary_grad
            # ill-conditioned (its kinetic term switches on the angle): the oracle's own float32 evaluation then differs
            # from float64 by up to ~2e-3, so each plan is allowed twice that float32 spread on top of 1e-5
            kw = dict(target_position=float(tp[j, e]), target_equilibrium=float(te[j, e]))
            J_chk, _ = O.plan_cost_grad(cost, s[e], Q_opt[e], float(u_prev[e]), **kw)
            J_f32, _ = O.plan_cost_grad(cost, s[e], Q_opt[e], float(u_prev[e]), dtype=np.float32, **kw)
            scale = float(np.abs(J_chk).max())
            tol = 1e-5 * scale + 2.0 * np.abs(J_f32 - J_chk)
            dJ = np.abs(J_out[e] - J_chk)
            assert np.all(dJ <= tol), float((dJ / tol).max())
            eJ = float(dJ.max()) / scale
            floor_used += int((dJ > 1e-5 * scale).sum())
            order = np.argsort(J_out[e], kind="stable")
            u = rec[e, 9]
            assert u == Q_opt[e, order[0], 0] and u_next[e] == u
            eu = abs(float(u) - float(ref["Q_opt"][order[0], 0]))
            assert eu < 1e-4 + 2.0 * abs(float(r32["Q_opt"][order[0], 0] - ref["Q_opt"][order[0], 0]))
            # a near-tie (oracle costs within rounding) may order two plans the other way; then the warm start differs
            # legitimately in those rows -- otherwise plans, moments and ages must follow the oracle's bookkeeping
            same = np.array_equal(order[:keep], ref["best"]) if j % resamp == 0 else order[0] == ref["best"][0]
            if not same:
                assert np.all(np.diff(J_chk[order]) > -(tol[order][1:] + tol[order][:-1])), \
                    "the fleet's cost order is wrong beyond rounding"
                order_skips += 1
            else:
                ok, eN = close(nxt["Q"][e], "Q_next", 2e-4)
                assert ok, eN
                mscale, vscale = max(1.0, float(np.abs(ref["m"]).max())), max(1.0, float(np.abs(ref["v"]).max()))
                okm, em = close(nxt["m"][e], "m", 2e-4 * mscale)
                okv, ev = close(nxt["v"][e], "v", 2e-4 * vscale)
                em, ev = em / mscale, ev / vscale
                assert okm and okv, (em, ev)
                if j % resamp == 0:
                    exp_ages = np.concatenate([np.ones(K - keep, np.int32), st["ages"][e][ref["best"]] + 1])
                else:
                    exp_ages = st["ages"][e] + 1
                np.testing.assert_array_equal(nxt["ages"][e], exp_ages)
                worst.update(Q_next=max(worst["Q_next"], eN), m=max(worst["m"], em), v=max(worst["v"], ev))
            s_ref, _, dd = O.plant_period(s[e], u)
            es = state_err(s_next[e], s_ref)
            assert es < 1e-5, es
            np.testing.assert_array_equal(rec[e, [1, 2, 4, 5, 6, 7]], s[e])
            np.testing.assert_allclose(rec[e, [3, 8]], dd[0], rtol=1e-5, atol=1e-5)
            assert rec[e, 10] == u and rec[e, 12] == tp[j, e] and rec[e, 13] == te[j, e]
            np.testing.assert_allclose(rec[e, 0], j * 0.02, rtol=1e-6)
            worst.update(Q_opt=max(worst["Q_opt"], eQ), J=max(worst["J"], eJ), u=max(worst["u"], eu),
                         state=max(worst["state"], es))
    record("rpgd_fleet_oracle", f"{cost}/E{E}/K{K}", order_skips=order_skips, J_beyond_1e_5=floor_used, **worst)
    # near-ties are rare (none measured on a B200); many skipped comparisons would hide a bookkeeping error
    assert order_skips <= max(1, n_checked // 10), (order_skips, n_checked)


def test_rpgd_fleet_is_bit_identical_to_the_single_experiment_kernels():
    """Per experiment, the fleet's plans after the Adam steps equal outer_its calls of Engine.rpgd_grad_step on the same
    (s, Q, m, v, iterations, u_prev, targets), and its costs equal Engine.plan_cost, bit for bit (two periods: the
    second has a non-zero u_prev and moments).  quadratic_boundary_grad with both target equilibria."""
    from cartpolesimulation_b200.core import Engine
    E, K, P = 5, 16, 2
    fl = make(E, K, GRAD)
    keep, n_ind = fl.opt_keep_k, fl.n_ind
    rng = np.random.default_rng(21)
    fl.reset(random_states(E, 22), init_draws=cuda(rng.standard_normal((E, K, n_ind))))
    draws = cuda(rng.standard_normal((P, E, K - keep, n_ind)))
    tp, te = targets(P, E, 23, flip=0)
    eng = Engine(K, T, cost=GRAD, interp_period=P_IND)
    for j in range(P):
        st = fl.plans()
        s, u_prev = fl.states(with_u_prev=True)
        J_out, Q_opt = torch.zeros((1, E, K), device="cuda"), torch.zeros((1, E, K, T), device="cuda")
        fl.run(1, cuda(tp[j:j + 1]), cuda(te[j:j + 1]), draws[j:j + 1].contiguous(), None, J_out, Q_opt)
        for e in range(E):
            eng.set_variable_parameters(target_position=float(tp[j, e]), target_equilibrium=float(te[j, e]))
            eng.rpgd_reset()
            m, v, _ = eng.rpgd_adam_state()
            m.copy_(torch.from_numpy(st["m"][e]).cuda())
            v.copy_(torch.from_numpy(st["v"][e]).cuda())
            eng.rpgd_set_iterations(st["adam_iterations"])
            Q = torch.from_numpy(st["Q"][e].copy()).cuda()
            s_dev = cuda(s[e])
            for _ in range(4):
                eng.rpgd_grad_step(s_dev, Q, float(u_prev[e]), 0.05, 0.9, 0.999, 1e-8, 5.0)
            J = eng.plan_cost(s_dev, Q, u_prev=float(u_prev[e]))[0]
            assert torch.equal(Q, Q_opt[0, e]), (j, e)
            assert torch.equal(J, J_out[0, e]), (j, e)


def test_rpgd_fleet_philox_draws_match_supplied():
    """A Philox fleet and a supplied fleet fed its draws(-1) / draws(period) give bit-identical records and plans."""
    E, K, P, resamp = 4, 16, 12, 5
    a = make(E, K, GRADMIN, noise="philox", seed=99, resamp_per=resamp)
    b = make(E, K, GRADMIN, resamp_per=resamp)
    s0 = random_states(E, 5)
    tp, te = targets(P, E, 6, flip=3)
    a.reset(s0)
    b.reset(s0, init_draws=a.draws(-1))
    draws = torch.stack([a.draws(j) for j in range(P)]).contiguous()
    assert draws.shape == (P, E, K - a.opt_keep_k, a.n_ind)
    assert abs(float(draws.mean())) < 0.1 and abs(float(draws.std()) - 1.0) < 0.1
    ra, rb = torch.zeros((P, E, 16), device="cuda"), torch.zeros((P, E, 16), device="cuda")
    a.run(P, cuda(tp), cuda(te), None, ra)
    b.run(P, cuda(tp), cuda(te), draws, rb)
    assert torch.equal(ra, rb)
    pa, pb = a.plans(), b.plans()
    for k in ("Q", "m", "v", "ages"):
        np.testing.assert_array_equal(pa[k], pb[k])
    assert a.period == b.period == P


def test_rpgd_fleet_split_independence():
    """One fleet of E experiments and two fleets covering the halves (experiment_offset) give bit-identical records."""
    E, K, P = 6, 16, 12
    s0 = random_states(E, 8)
    tp, te = targets(P, E, 9, flip=4)
    whole = make(E, K, GRAD, noise="philox", seed=4)
    whole.reset(s0)
    r = torch.zeros((P, E, 16), device="cuda")
    whole.run(P, cuda(tp), cuda(te), None, r)
    parts = []
    for lo, hi in ((0, 2), (2, 6)):
        f = make(hi - lo, K, GRAD, noise="philox", seed=4, experiment_offset=lo)
        f.reset(s0[lo:hi])
        rp = torch.zeros((P, hi - lo, 16), device="cuda")
        f.run(P, cuda(tp[:, lo:hi]), cuda(te[:, lo:hi]), None, rp)
        parts.append(rp)
    assert torch.equal(r, torch.cat(parts, dim=1))


def test_rpgd_fleet_nan_target_stays_in_its_experiment():
    """A NaN target makes every cost of that experiment NaN.  NaN costs sort after every number (torch.sort's order), so
    the ranks stay a permutation: the run completes, the experiment's ages stay those of a valid permutation, the other
    experiments' records are bit-identical to a run without the NaN, and the NaN costs are counted."""
    E, K, P, resamp = 4, 16, 12, 5
    s0 = random_states(E, 41)
    tp, te = targets(P, E, 42)
    tp_nan = tp.copy()
    tp_nan[:, 1] = np.nan
    recs, fleets = [], []
    for table in (tp, tp_nan):
        fl = make(E, K, GRAD, noise="philox", seed=5, resamp_per=resamp)
        fl.reset(s0)
        r = torch.zeros((P, E, 16), device="cuda")
        fl.run(P, cuda(table), cuda(te), None, r)
        torch.cuda.synchronize()
        recs.append(r.cpu().numpy())
        fleets.append(fl)
    others = [0, 2, 3]
    np.testing.assert_array_equal(recs[1][:, others], recs[0][:, others])
    ages = fleets[1].plans()["ages"]
    assert ages.min() >= 1 and ages.max() <= P, (ages.min(), ages.max())
    # every resampling solve rebuilds ages 1 (fresh) and the kept ones; the last resampled at period 10
    assert (ages[1] == 2).sum() == K - fleets[1].opt_keep_k
    assert fleets[0].nonfinite_costs() == 0 and fleets[1].nonfinite_costs() > 0


class _Draws:
    def __init__(self, draws):
        self.draws, self.i = list(draws), 0

    def normal(self, shape, mean=0.0, stddev=1.0, dtype=None):
        d = self.draws[self.i]
        self.i += 1
        assert list(d.shape) == list(shape)
        return d * stddev + mean


def test_rpgd_fleet_agrees_with_optimizer_rpgd_b200():
    """optimizer_rpgd_b200 driven with the same draws and the fleet's plant states, closed loop over 7 periods (resampling
    at 0, 3, 6).  Its fresh plans come from a torch matmul, so they may differ from the kernel's in the last bit."""
    import cartpolesimulation_b200 as cps
    from cartpolesimulation_b200.optimizer_forward_b200 import optimizer_rpgd_b200
    K, P, resamp, tp = 16, 7, 3, 0.03
    fl = make(1, K, GRADMIN, resamp_per=resamp)
    keep, n_ind = fl.opt_keep_k, fl.n_ind
    rng = np.random.default_rng(31)
    init = rng.standard_normal((1, K, n_ind)).astype(np.float32)
    draws = rng.standard_normal((P, 1, K - keep, n_ind)).astype(np.float32)
    vp = cps.VariableParameters(target_position=tp, target_equilibrium=1.0, L=0.395, m_pole=0.087)
    cost, predictor = cps.CostFunctionWrapper(), cps.PredictorWrapper()
    opt = optimizer_rpgd_b200(predictor=predictor, cost_function=cost,
                              control_limits=(np.array([-1.0], np.float32), np.array([1.0], np.float32)), seed=1,
                              mpc_horizon=T, num_rollouts=K, resamp_per=resamp, period_interpolation_inducing_points=P_IND)
    predictor.configure(batch_size=K, horizon=T, dt=0.02, variable_parameters=vp, predictor_specification="ODE")
    cost.configure(batch_size=K, horizon=T, variable_parameters=vp, environment_name="CartPole", computation_library=None,
                   cost_function_specification=GRADMIN)
    opt.configure(num_states=6, num_control_inputs=1, default_configure=False, dt=0.02, predictor_specification="ODE")
    opt.rng = _Draws([torch.from_numpy(init[0][:, :, None].copy())] +
                     [torch.from_numpy(draws[j, 0][:, :, None].copy()) for j in range(0, P, resamp)])
    opt.optimizer_reset()
    fl.reset(random_states(1, 32), init_draws=cuda(init))
    eQ = eu = 0.0
    for j in range(P):
        s = fl.states()[0]
        u_opt = float(opt.step(s.copy()))
        rec = torch.zeros((1, 1, 16), device="cuda")
        fl.run(1, cuda(np.full((1, 1), tp)), None, cuda(draws[j:j + 1]), rec)
        u = float(rec[0, 0, 9])
        Q = fl.plans()["Q"][0]
        eu, eQ = max(eu, abs(u - u_opt)), max(eQ, float(np.abs(Q - opt.Q_tf.cpu().numpy()).max()))
        assert abs(u - u_opt) < 1e-4, (j, u, u_opt)
        assert close_except_few(Q, opt.Q_tf.cpu().numpy(), 2e-4), j
    record("rpgd_fleet_optimizer", "gradmin_K16", Q=eQ, u=eu)


def test_rpgd_fleet_rejections():
    from cartpolesimulation_b200 import _lib as L
    from cartpolesimulation_b200.core import Engine
    from cartpolesimulation_b200.fleet import RpgdFleet
    for kw in (dict(integrator="ODE_v0"), dict(integrator="neural"), dict(cost="quadratic_boundary"),
               dict(cost="default"), dict(num_rollouts=4097), dict(SAMPLING_DISTRIBUTION="uniform")):
        args = dict(num_rollouts=16, cost=GRADMIN)
        args.update(kw)
        with pytest.raises(NotImplementedError):
            RpgdFleet(2, **args)
    for kw in (dict(opt_keep_k_ratio=2.0), dict(shift_previous=-1), dict(dt_simulation=0.003)):
        with pytest.raises(ValueError):
            RpgdFleet(2, **kw)
    fl = RpgdFleet(2)
    with pytest.raises(NotImplementedError):
        fl.set_plant_models(latency=0.01)
    with pytest.raises(RuntimeError):          # CPS_ERR_NOT_CONFIGURED before reset()
        fl.run(1)
    with pytest.raises(RuntimeError):
        fl.states()
    with pytest.raises(ValueError):            # a Philox fleet draws its own numbers
        fl.reset(np.zeros((2, 6), np.float32), init_draws=torch.zeros((2, 16, fl.n_ind), device="cuda"))
    eng = Engine(16, T, cost=GRADMIN, interp_period=P_IND)
    assert eng.lib.cps_rpgd_fleet_step(eng._h, 1, None, None, None, None, None, None) == 4
    assert eng.lib.cps_rpgd_fleet_draws(eng._h, 0, None) == 4
    # the C ABI's own checks (the Python class validates dt before it gets there)
    c = L.cps_rpgd_fleet_config(C.sizeof(L.cps_rpgd_fleet_config), 2, 7, L.FLEET_NOISE_PHILOX, 0.002, 0, 0, 4, 4, 10, 12, 1,
                                0.05, 0.9, 0.999, 1e-8, 5.0, 0.5, 0.0)
    assert eng.lib.cps_rpgd_fleet_create(eng._h, C.byref(c)) == 1
    c.sim_substeps, c.opt_keep_k = 10, 0
    assert eng.lib.cps_rpgd_fleet_create(eng._h, C.byref(c)) == 1
    c.opt_keep_k = 12
    assert eng.lib.cps_rpgd_fleet_create(eng._h, C.byref(c)) == 0


def test_rpgd_fleet_records_write_the_reference_csv(tmp_path):
    from cartpolesimulation_b200.fleet import make_experiments
    from cartpolesimulation_b200.recording import save_fleet_recordings
    E, P = 3, 20
    s0, tp, te = make_experiments(E, P, seed=2)
    fl = make(E, 16, GRADMIN, noise="philox", seed=2)
    fl.reset(s0)
    rec = torch.zeros((P, E, 16), device="cuda")
    fl.run(P, cuda(tp), cuda(te), None, rec)
    r = rec.cpu().numpy()
    assert np.all(np.isfinite(r)) and np.all(np.abs(r[:, :, 9]) <= 1.0)
    paths = save_fleet_recordings(rec, str(tmp_path), optimizer_name="rpgd-b200", run_for_ML_Pipeline=False)
    assert len(paths) == E
    with open(paths[1]) as f:
        rows = [row for row in csv.reader(line for line in f if not line.startswith("#"))]
    assert rows[0][:15] == ["time", "angle", "angleD", "angleDD", "angle_cos", "angle_sin", "position", "positionD",
                            "positionDD", "Q_calculated", "Q_applied", "Q_ccrc", "u", "target_position", "target_equilibrium"]
    assert len(rows) == P + 1
    np.testing.assert_allclose(np.array([float(x[1]) for x in rows[1:]]), r[:, 1, 1], rtol=1e-6, atol=1e-6)
    assert fl.engine.launch_count() > 0
