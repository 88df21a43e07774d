"""RPGD fleets on the neural predictor (cps_rpgd_fleet_* on a CPS_PREDICTOR_NEURAL handle, fleet.RpgdFleet(integrator=
"neural", network=...)): E closed-loop experiments whose controller plans with a GRU / Dense network while the plant stays
the CartPole ODE.  Against the float64 oracle (oracle.rpgd_step with oracle.net_grad's autograd gradient +
oracle.plant_period), the single-experiment kernels (Engine.rpgd_grad_step / Engine.plan_cost on a neural engine), their
own Philox draws, a split over two fleets and optimizer_rpgd_b200 on a neural PredictorWrapper.
Networks: the weights and normalisation of tests/golden/net_*.npz; non-zero stored states: h_after of
tests/golden/mppi_net_*.npz."""
import csv
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import net_grad as NG
from oracle import oracle as O
from tests.netutil import net_spec_from_golden
from tests.parity import close_except_few, load_golden, record

pytestmark = pytest.mark.gpu

GRADMIN, GRAD = "quadratic_boundary_grad_minimal", "quadratic_boundary_grad"
NETS = {"gru32": "net_GRU_6IN_32H1_32H2_5OUT_0", "gru64": "net_GRU_6IN_64H1_64H2_5OUT_0",
        "dense32": "net_Dense_6IN_32H1_32H2_5OUT_0"}
H_AFTER = {"gru32": "mppi_net_gru32_grad", "gru64": "mppi_net_gru64_gradmin"}
RANGES = np.array([np.pi, 18.38, 1.0, 1.0, 0.198, 1.125], dtype=np.float64)  # the reference's normalisation ranges
T, P_IND = 35, 4


def _spec(net):
    z, _ = load_golden(NETS[net])
    return net_spec_from_golden(z)


def _engine_spec(sp):
    d = dict(sp)
    d["weights"] = O.pack_net_weights(sp["net_type"], sp["layers"], sp["out_layer"])
    return d


def _h_after(net):
    z, _ = load_golden(H_AFTER[net])
    return z["h_after"][0].astype(np.float32)


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


def make(E, K, cost, net="gru32", noise="supplied", h0=None, spec=None, **kw):
    from cartpolesimulation_b200.fleet import RpgdFleet
    fl = RpgdFleet(E, num_rollouts=K, mpc_horizon=T, cost=cost, noise=noise, period_interpolation_inducing_points=P_IND,
                   integrator="neural", network=spec if spec is not None else _engine_spec(_spec(net)), **kw)
    if h0 is not None:
        fl.engine.net_set_state(h0)
    return fl


def _oracle_grad(sp):
    """oracle.plan_cost_grad's signature over oracle.net_grad (numpy dtypes mapped to torch's)."""
    def f(cost_name, s, Q, u_prev, dtype=np.float64, **kw):
        return NG.plan_cost_grad(sp, cost_name, s, Q, u_prev, dtype=torch.float32 if dtype == np.float32 else torch.float64,
                                 **kw)
    return f


@pytest.mark.parametrize("net,cost,E,K,flip,checked", [("gru32", GRADMIN, 1, 16, None, None),
                                                       ("gru32", GRAD, 3, 16, 5, None),
                                                       ("dense32", GRADMIN, 9, 64, 4, 3),
                                                       ("gru64", GRADMIN, 3, 64, 4, None)])
def test_neural_rpgd_fleet_matches_oracle_teacher_forced(monkeypatch, net, cost, E, K, flip, checked):
    """Every period starts the oracle from the fleet's own state (plans, moments, ages, counters, u_prev, plant state):
    12 periods, resampling at 0 and 10.  `checked`: experiments compared per period (rotating), None: all of them.
    quadratic_boundary_grad with target_equilibrium = -1 is ill-conditioned on fast-spinning states: there each entry is
    also allowed twice the spread of the oracle's own float32 evaluation (as the ODE fleet's oracle test)."""
    P, resamp = 12, 10
    sp = _spec(net)
    monkeypatch.setattr(O, "plan_cost_grad", _oracle_grad(sp))
    fl = make(E, K, cost, spec=_engine_spec(sp), resamp_per=resamp)
    keep, n_ind = fl.opt_keep_k, fl.n_ind
    rng = np.random.default_rng(7)
    init = rng.standard_normal((E, K, n_ind)).astype(np.float32)
    draws = rng.standard_normal((P, E, K - keep, n_ind)).astype(np.float32)
    tp, te = targets(P, E, 3, flip)
    fl.reset(random_states(E, 11), init_draws=cuda(init))
    d_draws, d_tp, d_te = cuda(draws), cuda(tp), cuda(te)
    worst = dict(Q_opt=0.0, J=0.0, u=0.0, Q_next=0.0, m=0.0, v=0.0, state=0.0)
    failures = []
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
            r32 = O.rpgd_step(*args, dtype=np.float32, **okw) if cost == GRAD else ref

            def close(got, key, atol):
                d = np.abs(np.asarray(got, np.float64) - ref[key])
                return bool(np.all(d <= atol + 2.0 * np.abs(r32[key] - ref[key]))), float(d.max())
            ok, eQ = close(Q_opt[e], "Q_opt", 1.6e-5)
            if not ok:
                failures.append(("Q_opt", j, e, eQ))
            kw = dict(target_position=float(tp[j, e]), target_equilibrium=float(te[j, e]))
            J_chk, _ = O.plan_cost_grad(cost, s[e], Q_opt[e], float(u_prev[e]), **kw)
            J_f32 = O.plan_cost_grad(cost, s[e], Q_opt[e], float(u_prev[e]), dtype=np.float32, **kw)[0] if cost == GRAD else J_chk
            scale = float(np.abs(J_chk).max())
            tol = 3.5e-6 * scale + 2.0 * np.abs(J_f32 - J_chk)
            dJ = np.abs(J_out[e] - J_chk)
            if not np.all(dJ <= tol):
                failures.append(("J", j, e, float((dJ / tol).max())))
            eJ = float(dJ.max()) / scale
            floor_used += int((dJ > 3.5e-6 * scale).sum())
            order = np.argsort(J_out[e], kind="stable")
            u = rec[e, 9]
            assert u == Q_opt[e, order[0], 0] and u_next[e] == u
            eu = abs(float(u) - float(ref["Q_opt"][order[0], 0]))
            if not eu < 2.2e-6 + 2.0 * abs(float(r32["Q_opt"][order[0], 0] - ref["Q_opt"][order[0], 0])):
                failures.append(("u", j, e, eu))
            # a near-tie (oracle costs within rounding) may order two plans the other way; then the warm start differs
            # legitimately in those rows -- otherwise plans, moments and ages must follow the oracle's bookkeeping
            same = np.array_equal(order[:keep], ref["best"]) if j % resamp == 0 else order[0] == ref["best"][0]
            if not same:
                assert np.all(np.diff(J_chk[order]) > -(tol[order][1:] + tol[order][:-1])), \
                    "the fleet's cost order is wrong beyond rounding"
                order_skips += 1
            else:
                ok, eN = close(nxt["Q"][e], "Q_next", 1.6e-5)
                mscale, vscale = max(1.0, float(np.abs(ref["m"]).max())), max(1.0, float(np.abs(ref["v"]).max()))
                okm, em = close(nxt["m"][e], "m", 2e-4 * mscale)
                okv, ev = close(nxt["v"][e], "v", 2e-4 * vscale)
                em, ev = em / mscale, ev / vscale
                if not (ok and okm and okv):
                    failures.append(("Q_next/m/v", j, e, (eN, em, ev)))
                if j % resamp == 0:
                    exp_ages = np.concatenate([np.ones(K - keep, np.int32), st["ages"][e][ref["best"]] + 1])
                else:
                    exp_ages = st["ages"][e] + 1
                np.testing.assert_array_equal(nxt["ages"][e], exp_ages)
                worst.update(Q_next=max(worst["Q_next"], eN), m=max(worst["m"], em), v=max(worst["v"], ev))
            # the plant is the CartPole ODE whatever the controller predicts with
            s_ref, _, dd = O.plant_period(s[e], u)
            es = state_err(s_next[e], s_ref)
            assert es < 1e-5, es
            np.testing.assert_array_equal(rec[e, [1, 2, 4, 5, 6, 7]], s[e])
            np.testing.assert_allclose(rec[e, [3, 8]], dd[0], rtol=1e-5, atol=1e-5)
            assert rec[e, 10] == u and rec[e, 12] == tp[j, e] and rec[e, 13] == te[j, e]
            worst.update(Q_opt=max(worst["Q_opt"], eQ), J=max(worst["J"], eJ), u=max(worst["u"], eu),
                         state=max(worst["state"], es))
    record("rpgd_fleet_neural_oracle", f"{net}/{cost}/E{E}/K{K}", order_skips=order_skips, J_beyond_bound=floor_used,
           **worst)
    assert not failures, failures[:5]
    # near-ties are rare (measured on a B200: 3 of 36 checked experiment-periods for GRU 2 x 64 at K = 64, 1 of 36 for
    # Dense 2 x 32 at K = 64, none at K = 16); many skipped comparisons would hide a bookkeeping error
    assert order_skips <= max(2, n_checked // 8), (order_skips, n_checked)


@pytest.mark.parametrize("net,K,cost,stored", [("gru32", 16, GRAD, True), ("gru32", 64, GRADMIN, False),
                                               ("gru32", 20, GRADMIN, True), ("dense32", 20, GRAD, False),
                                               ("dense32", 64, GRADMIN, False)])
def test_neural_rpgd_fleet_is_bit_identical_to_the_single_experiment_kernels(net, K, cost, stored):
    """Per experiment, the fleet's plans after the Adam steps equal outer_its calls of Engine.rpgd_grad_step on a neural
    engine with the same network and stored state, on the same (s, Q, m, v, iterations, u_prev, targets), and its costs
    equal Engine.plan_cost, bit for bit (two periods: the second has a non-zero u_prev and moments).  K = 64: several
    CTAs per experiment; K = 20: a partial tile."""
    from cartpolesimulation_b200.core import Engine
    E, P = 5, 2
    spec = _engine_spec(_spec(net))
    h0 = _h_after(net) if stored else None
    fl = make(E, K, cost, spec=spec, h0=h0)
    keep, n_ind = fl.opt_keep_k, fl.n_ind
    rng = np.random.default_rng(21)
    fl.reset(random_states(E, 22), init_draws=cuda(rng.standard_normal((E, K, n_ind))))
    draws = cuda(rng.standard_normal((P, E, K - keep, n_ind)))
    tp, te = targets(P, E, 23, flip=0)
    eng = Engine(K, T, integrator="neural", cost=cost, interp_period=P_IND)
    eng.net_load(spec)
    if h0 is not None:
        eng.net_set_state(h0)
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


def test_neural_rpgd_fleet_philox_draws_match_supplied():
    """A Philox fleet and a supplied fleet fed its draws(-1) / draws(period) give bit-identical records and plans."""
    E, K, P, resamp = 4, 16, 12, 5
    a = make(E, K, GRADMIN, noise="philox", seed=99, resamp_per=resamp)
    b = make(E, K, GRADMIN, resamp_per=resamp)
    s0 = random_states(E, 5)
    tp, te = targets(P, E, 6, flip=3)
    a.reset(s0)
    b.reset(s0, init_draws=a.draws(-1))
    draws = torch.stack([a.draws(j) for j in range(P)]).contiguous()
    ra, rb = torch.zeros((P, E, 16), device="cuda"), torch.zeros((P, E, 16), device="cuda")
    a.run(P, cuda(tp), cuda(te), None, ra)
    b.run(P, cuda(tp), cuda(te), draws, rb)
    assert torch.equal(ra, rb)
    pa, pb = a.plans(), b.plans()
    for k in ("Q", "m", "v", "ages"):
        np.testing.assert_array_equal(pa[k], pb[k])


def test_neural_rpgd_fleet_split_independence():
    """One fleet of E experiments and two fleets covering the halves (experiment_offset) give bit-identical records."""
    E, K, P = 6, 16, 12
    s0 = random_states(E, 8)
    tp, te = targets(P, E, 9, flip=4)
    h0 = _h_after("gru32")
    whole = make(E, K, GRAD, noise="philox", seed=4, h0=h0)
    whole.reset(s0)
    r = torch.zeros((P, E, 16), device="cuda")
    whole.run(P, cuda(tp), cuda(te), None, r)
    parts = []
    for lo, hi in ((0, 2), (2, 6)):
        f = make(hi - lo, K, GRAD, noise="philox", seed=4, experiment_offset=lo, h0=h0)
        f.reset(s0[lo:hi])
        rp = torch.zeros((P, hi - lo, 16), device="cuda")
        f.run(P, cuda(tp[:, lo:hi]), cuda(te[:, lo:hi]), None, rp)
        parts.append(rp)
    assert torch.equal(r, torch.cat(parts, dim=1))


def test_neural_rpgd_fleet_nan_target_stays_in_its_experiment():
    """A NaN target makes every cost of that experiment NaN; they sort after every number, so the run completes, the
    experiment's ages stay those of a valid permutation, the other experiments' records are bit-identical to a run
    without the NaN, and the NaN costs are counted."""
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
    for e in range(E):   # each experiment's ages: the last resampling (period 10) left K - keep fresh plans, now aged 2
        assert (ages[e] == 2).sum() == K - fleets[1].opt_keep_k
    assert fleets[0].nonfinite_costs() == 0 and fleets[1].nonfinite_costs() > 0


class _Draws:
    def __init__(self, draws):
        self.draws, self.i = list(draws), 0

    def normal(self, shape, mean=0.0, stddev=1.0, dtype=None):
        d = self.draws[self.i]
        self.i += 1
        assert list(d.shape) == list(shape)
        return d * stddev + mean


def test_neural_rpgd_fleet_agrees_with_optimizer_rpgd_b200(tmp_path):
    """optimizer_rpgd_b200 on a PredictorWrapper configured with a GRU 2 x 32 model directory, driven with the same draws
    and the fleet's plant states, closed loop over 7 periods (resampling at 0, 3, 6); the fleet runs the network the
    optimizer loaded.  Its fresh plans come from a torch matmul, so they may differ from the kernel's in the last bit."""
    import cartpolesimulation_b200 as cps
    from cartpolesimulation_b200.optimizer_forward_b200 import optimizer_rpgd_b200
    from cartpolesimulation_b200.optimizer_mppi_b200 import _extract_net_spec
    from tests.netutil import write_model_dir
    z, _ = load_golden(NETS["gru32"])
    K, P, resamp, tp = 16, 7, 3, 0.03
    vp = cps.VariableParameters(target_position=tp, target_equilibrium=1.0, L=0.395, m_pole=0.087)
    cost, predictor = cps.CostFunctionWrapper(), cps.PredictorWrapper()
    predictor.configure(batch_size=K, horizon=T, dt=0.02, variable_parameters=vp,
                        predictor_specification=write_model_dir(str(tmp_path), z))
    cost.configure(batch_size=K, horizon=T, variable_parameters=vp, environment_name="CartPole", computation_library=None,
                   cost_function_specification=GRADMIN)
    opt = optimizer_rpgd_b200(predictor=predictor, cost_function=cost,
                              control_limits=(np.array([-1.0], np.float32), np.array([1.0], np.float32)), seed=1,
                              mpc_horizon=T, num_rollouts=K, resamp_per=resamp, period_interpolation_inducing_points=P_IND)
    opt.configure(num_states=6, num_control_inputs=1, default_configure=False, dt=0.02, predictor_specification="neural")
    assert opt.predictor_type == "neural"
    fl = make(1, K, GRADMIN, spec=_extract_net_spec(predictor), resamp_per=resamp)
    keep, n_ind = fl.opt_keep_k, fl.n_ind
    rng = np.random.default_rng(31)
    init = rng.standard_normal((1, K, n_ind)).astype(np.float32)
    draws = rng.standard_normal((P, 1, K - keep, n_ind)).astype(np.float32)
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
    record("rpgd_fleet_neural_optimizer", "gru32_gradmin_K16", Q=eQ, u=eu)


def test_neural_rpgd_fleet_leaves_the_stored_state_and_counts_its_launches():
    """The stored hidden state is read, never written; a period takes 3 + 2 x (Adam steps) launches whatever E
    (first_iter_count Adam steps on the first solve after a reset, outer_its after that)."""
    E, K = 37, 16
    h0 = _h_after("gru32")
    fl = make(E, K, GRAD, noise="philox", seed=3, h0=h0, warmup=True, warmup_iterations=7)
    assert fl.first_iter_count == 7 and fl.outer_its == 4
    h_before = fl.engine.net_get_state().copy()
    np.testing.assert_array_equal(h_before, h0)
    tp, te = targets(3, E, 4, flip=1)
    fl.reset(random_states(E, 5))
    n0 = fl.engine.launch_count()
    fl.run(1, cuda(tp[:1]), cuda(te[:1]))
    assert fl.engine.launch_count() - n0 == 3 + 2 * 7
    n1 = fl.engine.launch_count()
    fl.run(2, cuda(tp[1:]), cuda(te[1:]))
    assert fl.engine.launch_count() - n1 == 2 * (3 + 2 * 4)
    np.testing.assert_array_equal(fl.engine.net_get_state(), h_before)
    assert fl.nonfinite_costs() == 0


def test_neural_rpgd_fleet_rejections():
    from cartpolesimulation_b200 import _lib as L
    from cartpolesimulation_b200.core import Engine
    from cartpolesimulation_b200.fleet import RpgdFleet
    K = 16
    # differential (D_*) network
    zd, _ = load_golden("net_diff_GRU_6IN_32H1_32H2_5OUT_1")
    spd = net_spec_from_golden(zd)
    d = _engine_spec(spd)
    f = spd["diff"]
    d.update(differential=True, diff_p1=f["p1"], diff_p2=f["p2"], out_norm_a=f["on_a"], out_norm_b=f["on_b"],
             out_to_in=f["out_to_in"])
    with pytest.raises(NotImplementedError):
        RpgdFleet(2, num_rollouts=K, integrator="neural", network=d)
    # a network whose image with the adjoint's buffers exceeds 227 KB of shared memory (GRU 2 x 72)
    sp = dict(_spec("gru32"))
    rng = np.random.default_rng(0)
    H, n_in = 72, len(sp["in_idx"]) + 1
    sp["hsz"] = [H, H]
    sp["layers"] = [tuple(rng.normal(0, 0.1, shp).astype(np.float32) for shp in ((3 * H, i), (3 * H, H), (3 * H,), (3 * H,)))
                    for i in (n_in, H)]
    sp["out_layer"] = (rng.normal(0, 0.1, (len(sp["out_idx"]), H)).astype(np.float32),
                       np.zeros(len(sp["out_idx"]), np.float32))
    with pytest.raises(NotImplementedError):
        RpgdFleet(2, num_rollouts=K, integrator="neural", network=_engine_spec(sp))
    # cost plugins without an adjoint
    for cost in ("default", "quadratic_boundary"):
        with pytest.raises(NotImplementedError):
            RpgdFleet(2, num_rollouts=K, cost=cost, integrator="neural", network=_engine_spec(_spec("gru32")))
    # the C ABI: the tensor-core flag (CPS_ERR_UNSUPPORTED), a neural handle without a network (CPS_ERR_NOT_CONFIGURED)
    c = L.cps_rpgd_fleet_config(C.sizeof(L.cps_rpgd_fleet_config), 2, 10, L.FLEET_NOISE_PHILOX, 0.002, 0, 0, 4, 4, 10, 12, 1,
                                0.05, 0.9, 0.999, 1e-8, 5.0, 0.5, 0.0)
    eng = Engine(K, T, integrator="neural", cost=GRADMIN, interp_period=P_IND, net_kernel="tensor")
    eng.net_load(_engine_spec(_spec("gru64")))
    with pytest.raises(NotImplementedError):
        eng._chk(eng.lib.cps_rpgd_fleet_create(eng._h, C.byref(c)))
    eng = Engine(K, T, integrator="neural", cost=GRADMIN, interp_period=P_IND)
    assert eng.lib.cps_rpgd_fleet_create(eng._h, C.byref(c)) == 4
    eng.net_load(_engine_spec(_spec("gru32")))
    assert eng.lib.cps_rpgd_fleet_create(eng._h, C.byref(c)) == 0


def test_neural_rpgd_fleet_records_write_the_reference_csv(tmp_path):
    from cartpolesimulation_b200.fleet import make_experiments
    from cartpolesimulation_b200.recording import save_fleet_recordings
    E, P = 3, 20
    s0, tp, te = make_experiments(E, P, seed=2)
    fl = make(E, 16, GRADMIN, net="dense32", noise="philox", seed=2)
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
