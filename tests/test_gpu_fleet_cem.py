"""CEM fleets (cps_cem_fleet_*, fleet.CemFleet): E closed-loop experiments under optimizer_cem_tf, against the float64
oracle (oracle.cem_step + oracle.plant_period), the single solve (Engine.cem_step), their own Philox draws, a split over
two fleets, a permutation of the experiments and optimizer_cem_b200."""
import csv
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import oracle as O
from tests.parity import record, shifted_cost_ok, vec_err

pytestmark = pytest.mark.gpu

GRADMIN, GRAD = "quadratic_boundary_grad_minimal", "quadratic_boundary_grad"
SHIFTED = ("default", "quadratic_boundary")   # MAX_COST plugins: order below the 6e9 shift is noise (DESIGN.md 6.3)
RANGES = np.array([np.pi, 18.38, 1.0, 1.0, 0.198, 1.125], dtype=np.float64)   # the reference's normalisation ranges
T = 35


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


def make(E, K, best_k, cost=GRADMIN, integrator="ODE", noise="philox", **kw):
    from cartpolesimulation_b200.fleet import CemFleet
    return CemFleet(E, num_rollouts=K, mpc_horizon=T, cem_best_k=best_k, cost=cost, integrator=integrator, noise=noise, **kw)


def elite_update(Q, J, best_k, stdev_min, initial_stdev):
    """The last iteration's update from the fleet's own plans Q [K, T] and costs J: stable order, mean / population
    stdev, clip, shift.  Returns (elites ascending, mean, stdev, u)."""
    order = np.argsort(J, kind="stable")[:best_k]
    eq = Q[order].astype(np.float64)
    mean, std = eq.mean(0), np.maximum(eq.std(0), stdev_min)
    return np.sort(order), np.r_[mean[1:], 0.0], np.r_[std[1:], initial_stdev], Q[order[0], 0]


CASES = [  # integrator, cost, E, K, best_k, flip, warmup_iterations, checked
    ("ODE", GRADMIN, 1, 200, 40, None, None, None),
    ("ODE_v0", GRAD, 3, 64, 10, 5, None, None),
    ("ODE", GRAD, 37, 300, 64, 4, None, 3),              # best_k x T = 2240: statistics in cem_update_fleet_kernel
    ("ODE", "default", 3, 200, 40, 4, None, None),
    ("ODE_v0", "quadratic_boundary", 3, 300, 70, None, None, None),
    ("ODE", GRADMIN, 3, 64, 8, 6, 5, None),              # warmup: the first period runs 5 iterations
]


@pytest.mark.parametrize("integ,cost,E,K,best_k,flip,warm,checked", CASES)
def test_cem_fleet_matches_oracle_teacher_forced(integ, cost, E, K, best_k, flip, warm, checked):
    """Every period starts the oracle from the fleet's own state, distribution, u_prev, targets and draws(period): 12
    periods.  `checked`: experiments compared per period (rotating), None: all of them."""
    P, sd0, sd_min = 12, 0.5, 0.01
    kw = dict(warmup=True, warmup_iterations=warm) if warm else {}
    fl = make(E, K, best_k, cost, integ, seed=3, **kw)
    tp, te = targets(P, E, 3, flip)
    fl.reset(random_states(E, 11))
    mu0, s0 = fl.distribution()
    assert np.all(mu0 == 0.0) and np.all(s0 == np.float32(sd0))
    d_tp, d_te = cuda(tp), cuda(te)
    worst = dict(u=0.0, mean=0.0, stdev=0.0, Q=0.0, J=0.0, state=0.0)
    skips = n_checked = 0
    for j in range(P):
        s, u_prev = fl.states(with_u_prev=True)
        mu, sd = fl.distribution()
        draws = fl.draws(j).cpu().numpy()
        assert draws.shape[0] == (warm if (warm and j == 0) else 3)
        rec, J_out, Q_out = (torch.zeros(shape, device="cuda") for shape in ((1, E, 16), (1, E, K), (1, E, T, K)))
        fl.run(1, d_tp[j:j + 1].contiguous(), d_te[j:j + 1].contiguous(), None, rec, J_out, Q_out)
        mu_n, sd_n = fl.distribution()
        s_next, u_next = fl.states(with_u_prev=True)
        rec, J_out, Q_out = rec.cpu().numpy()[0], J_out.cpu().numpy()[0], Q_out.cpu().numpy()[0]
        exps = range(E) if checked is None else [(j * checked + i) % E for i in range(checked)]
        for e in exps:
            n_checked += 1
            Qe = Q_out[e].T   # [K, T]
            kw = dict(target_position=float(tp[j, e]), target_equilibrium=float(te[j, e]))
            # the last iteration's costs of the fleet's own plans, and its update from them
            J_chk = O.plan_cost(integ, cost, s[e], Qe, float(u_prev[e]), **kw)
            assert shifted_cost_ok(J_out[e], J_chk) if cost in SHIFTED else vec_err(J_out[e], J_chk) < 3e-5, (j, e)
            el, m_chk, s_chk, u_chk = elite_update(Qe, J_out[e], best_k, sd_min, sd0)
            np.testing.assert_allclose(mu_n[e], m_chk, rtol=0, atol=2e-6)
            np.testing.assert_allclose(sd_n[e], s_chk, rtol=0, atol=2e-6)
            u = rec[e, 9]
            assert u == u_chk and u_next[e] == u and rec[e, 10] == u
            # the whole solve from the same inputs
            ref = O.cem_step(integ, cost, s[e], draws[:, e].transpose(0, 2, 1), mu[e], sd[e], best_k, sd_min, sd0,
                             u_prev=float(u_prev[e]), **kw)
            if cost in SHIFTED or not np.array_equal(el, ref["elites"]):
                # MAX_COST plugins: the order below the shift is rounding noise, so the solve is followed only through the
                # fleet's own plans above; otherwise a near-tie in an earlier iteration may pick other elites
                skips += cost not in SHIFTED
            else:
                eQ, eJ = float(np.abs(Qe - ref["Q"]).max()), vec_err(J_out[e], ref["J"])
                em, es_ = float(np.abs(mu_n[e] - ref["mean"]).max()), float(np.abs(sd_n[e] - ref["stdev"]).max())
                assert eQ < 2e-6 and eJ < 3e-5 and em < 3e-6 and es_ < 3e-6, (j, e, eQ, eJ, em, es_)
                assert abs(float(u) - float(ref["u"])) < 1e-4
                worst.update(u=max(worst["u"], abs(float(u) - float(ref["u"]))), mean=max(worst["mean"], em),
                             stdev=max(worst["stdev"], es_), Q=max(worst["Q"], eQ), J=max(worst["J"], eJ))
            s_ref, _, dd = O.plant_period(s[e], u)
            es = state_err(s_next[e], s_ref)
            assert es < 1e-5, es
            np.testing.assert_array_equal(rec[e, [1, 2, 4, 5, 6, 7]], s[e])
            np.testing.assert_allclose(rec[e, [3, 8]], dd[0], rtol=1e-5, atol=1e-5)
            assert rec[e, 12] == tp[j, e] and rec[e, 13] == te[j, e]
            np.testing.assert_allclose(rec[e, 0], j * 0.02, rtol=1e-6)
            worst.update(state=max(worst["state"], es))
    assert fl.period == P
    record("cem_fleet_oracle", f"{integ}/{cost}/E{E}/K{K}/bk{best_k}", skips=skips, checked=n_checked, **worst)
    # float32 and float64 costs order a near-tie at the elite boundary differently in a few solves (measured on a B200: 2
    # of 12 and 4 of 36); the fleet's own update is checked in every one of them above, and most solves must follow the
    # oracle end to end
    assert skips <= n_checked // 4, (skips, n_checked)


@pytest.mark.parametrize("cost,best_k", [(GRAD, 40), (GRADMIN, 64), ("quadratic_boundary", 40)])
def test_cem_fleet_is_bit_identical_to_the_single_solve(cost, best_k):
    """Per experiment and period, cps_cem_step on an Engine given the experiment's distribution, targets, state, u_prev and
    draws gives the fleet's u, distribution, last-iteration J and Q bit for bit (two periods, both target equilibria)."""
    from cartpolesimulation_b200 import _lib as L
    from cartpolesimulation_b200.core import Engine
    E, K, P = 4, 200, 2
    fl = make(E, K, best_k, cost, noise="supplied")
    rng = np.random.default_rng(21)
    fl.reset(random_states(E, 22))
    draws = rng.standard_normal((P, 3, E, T, K)).astype(np.float32)
    tp, te = targets(P, E, 23, flip=0)
    eng = Engine(K, T, cost=cost)
    eng.cem_configure(best_k, 0.5, 0.01)
    for j in range(P):
        s, u_prev = fl.states(with_u_prev=True)
        mu, sd = fl.distribution()
        J_out, Q_out = torch.zeros((1, E, K), device="cuda"), torch.zeros((1, E, T, K), device="cuda")
        fl.run(1, cuda(tp[j:j + 1]), cuda(te[j:j + 1]), cuda(draws[j]), None, J_out, Q_out)
        mu_n, sd_n = fl.distribution()
        _, u_n = fl.states(with_u_prev=True)
        for e in range(E):
            eng.set_variable_parameters(target_position=float(tp[j, e]), target_equilibrium=float(te[j, e]))
            eng.cem_set_distribution(mu[e], sd[e])
            J, Q = torch.empty(K, device="cuda"), torch.empty((T, K), device="cuda")
            u = eng.cem_step(cuda(s[e]), cuda(draws[j][:, e]), L.TIME_MAJOR, float(u_prev[e]), Q_out=Q, J_out=J)
            m1, s1 = eng.cem_get_distribution()
            assert float(u.cpu()[0]) == float(u_n[e]), (j, e)
            assert np.array_equal(m1, mu_n[e]) and np.array_equal(s1, sd_n[e]), (j, e)
            assert torch.equal(J, J_out[0, e]) and torch.equal(Q, Q_out[0, e]), (j, e)


def test_cem_fleet_philox_draws_match_supplied():
    """A Philox fleet and a supplied fleet fed its draws(period) give bit-identical records and distributions (the first
    period runs warmup_iterations)."""
    E, K, P = 4, 200, 6
    a = make(E, K, 40, seed=99, warmup=True, warmup_iterations=4)
    b = make(E, K, 40, noise="supplied", warmup=True, warmup_iterations=4)
    s0 = random_states(E, 5)
    tp, te = targets(P, E, 6, flip=3)
    a.reset(s0)
    b.reset(s0)
    draws = torch.cat([a.draws(j) for j in range(P)]).contiguous()
    assert draws.shape == (4 + 3 * (P - 1), E, T, K)
    assert abs(float(draws.mean())) < 0.01 and abs(float(draws.std()) - 1.0) < 0.01
    ra, rb = torch.zeros((P, E, 16), device="cuda"), torch.zeros((P, E, 16), device="cuda")
    a.run(P, cuda(tp), cuda(te), None, ra)
    b.run(P, cuda(tp), cuda(te), draws, rb)
    assert torch.equal(ra, rb)
    for x, y in zip(a.distribution(), b.distribution()):
        np.testing.assert_array_equal(x, y)
    assert a.period == b.period == P


def test_cem_fleet_split_and_permutation():
    """One fleet of E experiments equals two fleets split by experiment_offset (Philox), and permuting the experiments of a
    supplied fleet permutes every output, bit for bit."""
    E, K, P = 6, 64, 8
    s0 = random_states(E, 8)
    tp, te = targets(P, E, 9, flip=4)
    whole = make(E, K, 10, GRAD, seed=4)
    whole.reset(s0)
    r = torch.zeros((P, E, 16), device="cuda")
    whole.run(P, cuda(tp), cuda(te), None, r)
    parts = []
    for lo, hi in ((0, 2), (2, 6)):
        f = make(hi - lo, K, 10, GRAD, seed=4, experiment_offset=lo)
        f.reset(s0[lo:hi])
        rp = torch.zeros((P, hi - lo, 16), device="cuda")
        f.run(P, cuda(tp[:, lo:hi]), cuda(te[:, lo:hi]), None, rp)
        parts.append(rp)
    assert torch.equal(r, torch.cat(parts, dim=1))
    perm = np.array([3, 0, 5, 1, 4, 2])
    draws = np.random.default_rng(10).standard_normal((3 * P, E, T, K)).astype(np.float32)
    outs = []
    for p in (np.arange(E), perm):
        f = make(E, K, 10, GRAD, noise="supplied")
        f.reset(s0[p])
        rec, J = torch.zeros((P, E, 16), device="cuda"), torch.zeros((P, E, K), device="cuda")
        Q = torch.zeros((P, E, T, K), device="cuda")
        f.run(P, cuda(tp[:, p]), cuda(te[:, p]), cuda(draws[:, p]), rec, J, Q)
        outs.append([x.cpu().numpy() for x in (rec, J, Q)] + list(f.distribution()) + list(f.states(with_u_prev=True)))
    for x, y in zip(outs[0][:3], outs[1][:3]):
        np.testing.assert_array_equal(x[:, perm], y)
    for x, y in zip(outs[0][3:], outs[1][3:]):
        np.testing.assert_array_equal(x[perm], y)


def test_cem_fleet_nan_target_stays_in_its_experiment():
    """A NaN target makes every cost of that experiment NaN (sorted last): the run completes, the other experiments'
    records are bit-identical to a run without the NaN, and the NaN costs are counted."""
    E, K, P = 4, 200, 6
    s0 = random_states(E, 41)
    tp, te = targets(P, E, 42)
    tp_nan = tp.copy()
    tp_nan[:, 1] = np.nan
    recs, fleets = [], []
    for table in (tp, tp_nan):
        fl = make(E, K, 40, GRAD, seed=5)
        fl.reset(s0)
        r = torch.zeros((P, E, 16), device="cuda")
        fl.run(P, cuda(table), cuda(te), None, r)
        torch.cuda.synchronize()
        recs.append(r.cpu().numpy())
        fleets.append(fl)
    others = [0, 2, 3]
    np.testing.assert_array_equal(recs[1][:, others], recs[0][:, others])
    assert np.all(np.abs(recs[1][:, 1, 9]) <= 1.0)   # the NaN experiment still picks a clipped control
    assert fleets[0].nonfinite_costs() == 0 and fleets[1].nonfinite_costs() >= P * 3 * K


class _Draws:
    def __init__(self, draws):
        self.draws, self.i = list(draws), 0

    def normal(self, shape, dtype=None):
        d = self.draws[self.i]
        self.i += 1
        assert list(d.shape) == list(shape)
        return d


def test_cem_fleet_agrees_with_optimizer_cem_b200():
    """optimizer_cem_b200 driven with the fleet's draws and states, closed loop over 5 periods with warm-up: the same
    controls and distributions, and the plant as oracle.plant_period."""
    import cartpolesimulation_b200 as cps
    from cartpolesimulation_b200.optimizer_forward_b200 import optimizer_cem_b200
    K, P, tp = 200, 5, 0.03
    fl = make(1, K, 40, seed=12, warmup=True, warmup_iterations=6)
    fl.reset(random_states(1, 32))
    vp = cps.VariableParameters(target_position=tp, target_equilibrium=1.0, L=0.395, m_pole=0.087)
    cost, predictor = cps.CostFunctionWrapper(), cps.PredictorWrapper()
    opt = optimizer_cem_b200(predictor=predictor, cost_function=cost,
                             control_limits=(np.array([-1.0], np.float32), np.array([1.0], np.float32)), seed=1,
                             mpc_horizon=T, num_rollouts=K, warmup=True, warmup_iterations=6)
    predictor.configure(batch_size=K, horizon=T, dt=0.02, variable_parameters=vp, predictor_specification="ODE")
    cost.configure(batch_size=K, horizon=T, variable_parameters=vp, environment_name="CartPole", computation_library=None,
                   cost_function_specification=GRADMIN)
    opt.configure(num_states=6, num_control_inputs=1, dt=0.02, predictor_specification="ODE")
    opt.rng = _Draws([torch.from_numpy(np.ascontiguousarray(d[0].T)[:, :, None]) for j in range(P)
                      for d in fl.draws(j).cpu().numpy()])
    es = eu = 0.0
    for j in range(P):
        s = fl.states()[0]
        u_opt = float(opt.step(s.copy()))
        rec = torch.zeros((1, 1, 16), device="cuda")
        fl.run(1, cuda(np.full((1, 1), tp)), None, None, rec)
        u = float(rec[0, 0, 9])
        eu = max(eu, abs(u - u_opt))
        assert abs(u - u_opt) < 1e-6, (j, u, u_opt)
        mu, sd = fl.distribution()
        np.testing.assert_allclose(mu[0], opt.dist_mue.numpy().reshape(-1), rtol=0, atol=1e-6)
        np.testing.assert_allclose(sd[0], opt.stdev.numpy().reshape(-1), rtol=0, atol=1e-6)
        s_ref, _, _ = O.plant_period(s, u)
        es = max(es, state_err(fl.states()[0], s_ref))
        assert es < 1e-5, es
    assert opt.count == P
    record("cem_fleet_optimizer", "gradmin_K200", u=eu, state=es)


@pytest.mark.parametrize("best_k,per_it", [(40, 1), (64, 2)])
def test_cem_fleet_launches_per_period(best_k, per_it):
    """n_it x (1, or 2 with the statistics deferred: best_k x T > 2048) + 1 launches per period, whatever E."""
    for E in (1, 300):
        fl = make(E, 200, best_k, warmup=True, warmup_iterations=5)
        fl.reset(random_states(E, 1))
        n0 = fl.engine.launch_count()
        fl.run(1)
        n1 = fl.engine.launch_count()
        fl.run(2)
        assert n1 - n0 == 5 * per_it + 1
        assert fl.engine.launch_count() - n1 == 2 * (3 * per_it + 1)


def test_cem_fleet_rejections():
    from cartpolesimulation_b200 import _lib as L
    from cartpolesimulation_b200.core import Engine
    from cartpolesimulation_b200.fleet import CemFleet
    for kw in (dict(integrator="neural"), dict(cost=None), dict(num_rollouts=8193)):
        with pytest.raises(NotImplementedError):
            CemFleet(2, **kw)
    for kw in (dict(cem_best_k=0), dict(cem_best_k=201), dict(cem_initial_action_stdev=-0.1), dict(cem_stdev_min=-1.0),
               dict(dt_simulation=0.003), dict(cem_outer_it=0)):
        with pytest.raises(ValueError):
            CemFleet(2, **kw)
    fl = CemFleet(2)
    with pytest.raises(NotImplementedError):
        fl.set_plant_models(latency=0.01)
    with pytest.raises(RuntimeError):          # CPS_ERR_NOT_CONFIGURED before reset()
        fl.run(1)
    with pytest.raises(RuntimeError):
        fl.states()
    fl.reset(np.zeros((2, 6), np.float32))
    with pytest.raises(ValueError):            # a Philox fleet draws its own numbers
        fl.run(1, draws=torch.zeros((3, 2, T, 200), device="cuda"))
    sup = CemFleet(2, noise="supplied")
    sup.reset(np.zeros((2, 6), np.float32))
    with pytest.raises(ValueError):            # and a supplied one needs them
        sup.run(1)
    with pytest.raises(ValueError):            # of the right size
        sup.run(1, draws=torch.zeros((2, 2, T, 200), device="cuda"))
    # the C ABI's own checks
    def cfg(**kw):
        c = L.cps_cem_fleet_config(C.sizeof(L.cps_cem_fleet_config), 2, 10, L.FLEET_NOISE_PHILOX, 0.002, 0, 0, 3, 3, 40,
                                   0.5, 0.01)
        for k, v in kw.items():
            setattr(c, k, v)
        return C.byref(c)
    eng = Engine(200, T)
    assert eng.lib.cps_cem_fleet_step(eng._h, 1, None, None, None, None, None, None) == 4
    assert eng.lib.cps_cem_fleet_create(eng._h, cfg(sim_substeps=7)) == 1
    assert eng.lib.cps_cem_fleet_create(eng._h, cfg(best_k=0)) == 1
    assert eng.lib.cps_cem_fleet_create(eng._h, cfg(stdev_min=-0.5)) == 1
    assert eng.lib.cps_cem_fleet_create(eng._h, cfg(first_iter_count=0)) == 1
    assert eng.lib.cps_cem_fleet_create(eng._h, cfg(struct_size=8)) == 1
    assert eng.lib.cps_cem_fleet_create(eng._h, cfg()) == 0
    assert eng.lib.cps_cem_fleet_step(eng._h, 1, None, None, None, None, None, None) == 4   # no states yet
    for args, kw in (((200, T), dict(substep_sincos=True)), ((200, T), dict(fast_div=True)),
                     ((200, T), dict(integrator="neural")), ((9000, T), {}), ((200, T), dict(cost="legacy_mppi", noise_mode="direct")),
                     ((64, 13000), {})):   # T = 13000: mean, stdev and their updates alone exceed the shared memory
        other = Engine(*args, **kw)
        assert other.lib.cps_cem_fleet_create(other._h, cfg(best_k=4)) == 3, (args, kw)


def test_cem_fleet_records_write_the_reference_csv(tmp_path):
    from cartpolesimulation_b200.fleet import make_experiments
    from cartpolesimulation_b200.recording import save_fleet_recordings
    E, P = 3, 20
    s0, tp, te = make_experiments(E, P, seed=2)
    fl = make(E, 200, 40, seed=2)
    fl.reset(s0)
    rec = torch.zeros((P, E, 16), device="cuda")
    fl.run(P, cuda(tp), cuda(te), None, rec)
    r = rec.cpu().numpy()
    assert np.all(np.isfinite(r)) and np.all(np.abs(r[:, :, 9]) <= 1.0)
    paths = save_fleet_recordings(rec, str(tmp_path), optimizer_name="cem-b200", run_for_ML_Pipeline=False)
    assert len(paths) == E
    with open(paths[1]) as f:
        rows = [row for row in csv.reader(line for line in f if not line.startswith("#"))]
    assert rows[0][:15] == ["time", "angle", "angleD", "angleDD", "angle_cos", "angle_sin", "position", "positionD",
                            "positionDD", "Q_calculated", "Q_applied", "Q_ccrc", "u", "target_position", "target_equilibrium"]
    assert len(rows) == P + 1
    np.testing.assert_allclose(np.array([float(x[1]) for x in rows[1:]]), r[:, 1, 1], rtol=1e-6, atol=1e-6)
