"""Random-action fleets (cps_random_action_fleet_*, fleet.RandomActionFleet): E closed-loop experiments under
optimizer_random_action_tf, against the float64 oracle (oracle.random_action_step + oracle.plant_period), the single solve
(Engine.plan_random_action), their own Philox draws, a numpy restatement of the Philox uniforms, a split over two fleets,
a permutation of the experiments and optimizer_random_action_b200."""
import csv
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import oracle as O
from tests.parity import record, shifted_cost_ok, vec_err
from tests.test_gpu_fleet_core import OFFSET, SEED, philox4x32_10

pytestmark = pytest.mark.gpu

GRADMIN, GRAD = "quadratic_boundary_grad_minimal", "quadratic_boundary_grad"
SHIFTED = ("default", "quadratic_boundary")   # MAX_COST plugins: order below the 6e9 shift is noise (DESIGN.md 6.3)
RANGES = np.array([np.pi, 18.38, 1.0, 1.0, 0.198, 1.125], dtype=np.float64)   # the reference's normalisation ranges
RA_DRAWS = 0xE0000000   # cps_plant.cuh
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


def make(E, K, cost=GRADMIN, integrator="ODE", noise="philox", **kw):
    from cartpolesimulation_b200.fleet import RandomActionFleet
    return RandomActionFleet(E, num_rollouts=K, mpc_horizon=T, cost=cost, integrator=integrator, noise=noise, **kw)


def uniforms(w0, w1, period, e_global, n, lo, hi):
    """philox_uniforms: n values lo + (hi - lo) u per (w0, e_global) (broadcast), u = (word >> 8) 2^-24, four per counter
    (w0, w1 + group, period, e); float32 multiply and add rounded separately."""
    out = []
    for g in range((n + 3) // 4):
        out += philox4x32_10(w0, w1 + g, period, e_global, SEED)
    u = [(w >> np.uint64(8)).astype(np.float32) * np.float32(2.0 ** -24) for w in out[:n]]
    span = np.float32(hi) - np.float32(lo)
    return np.stack([np.float32(lo) + span * x for x in u], axis=-1).astype(np.float32)


CASES = [  # integrator, cost, E, K, flip, checked
    ("ODE", GRADMIN, 1, 200, None, None),
    ("ODE_v0", GRAD, 3, 64, 5, None),
    ("ODE", GRAD, 37, 300, 4, 3),
    ("ODE", "default", 3, 200, 4, None),
    ("ODE_v0", "quadratic_boundary", 3, 300, None, None),
]


@pytest.mark.parametrize("integ,cost,E,K,flip,checked", CASES)
def test_random_action_fleet_matches_oracle_teacher_forced(integ, cost, E, K, flip, checked):
    """Every period starts the oracle from the fleet's own state, u_prev, targets and draws(period): 12 periods.
    `checked`: experiments compared per period (rotating), None: all of them."""
    P = 12
    fl = make(E, K, cost, integ, seed=3)
    tp, te = targets(P, E, 3, flip)
    fl.reset(random_states(E, 11))
    d_tp, d_te = cuda(tp), cuda(te)
    worst = dict(J=0.0, state=0.0)
    skips = n_checked = 0
    for j in range(P):
        s, u_prev = fl.states(with_u_prev=True)
        plans = fl.draws(j).cpu().numpy()
        assert np.all(plans >= -1.0) and np.all(plans < 1.0)
        rec, J_out, Q_out = (torch.zeros(shape, device="cuda") for shape in ((1, E, 16), (1, E, K), (1, E, T, K)))
        fl.run(1, d_tp[j:j + 1].contiguous(), d_te[j:j + 1].contiguous(), None, rec, J_out, Q_out)
        s_next, u_next = fl.states(with_u_prev=True)
        rec, J_out, Q_out = rec.cpu().numpy()[0], J_out.cpu().numpy()[0], Q_out.cpu().numpy()[0]
        np.testing.assert_array_equal(Q_out, plans)
        exps = range(E) if checked is None else [(j * checked + i) % E for i in range(checked)]
        for e in exps:
            n_checked += 1
            Qe = plans[e].T   # [K, T]
            kw = dict(target_position=float(tp[j, e]), target_equilibrium=float(te[j, e]))
            ref = O.random_action_step(integ, cost, s[e], Qe, float(u_prev[e]), **kw)
            ok = shifted_cost_ok(J_out[e], ref["J"]) if cost in SHIFTED else vec_err(J_out[e], ref["J"]) < 3e-5
            assert ok, (j, e)
            if cost not in SHIFTED:
                worst.update(J=max(worst["J"], vec_err(J_out[e], ref["J"])))
            # u is the first input of the fleet's own cheapest plan (stable: lowest index among equal costs) ...
            u = rec[e, 9]
            assert u == Qe[np.argsort(J_out[e], kind="stable")[0], 0] and u_next[e] == u and rec[e, 10] == u
            # ... and the oracle's, unless float32 and float64 costs order a near-tie differently
            if u != ref["u"]:
                skips += 1
            s_ref, _, dd = O.plant_period(s[e], u)
            es = state_err(s_next[e], s_ref)
            assert es < 1e-5, es
            np.testing.assert_array_equal(rec[e, [1, 2, 4, 5, 6, 7]], s[e])
            np.testing.assert_allclose(rec[e, [3, 8]], dd[0], rtol=1e-5, atol=1e-5)
            assert rec[e, 12] == tp[j, e] and rec[e, 13] == te[j, e]
            np.testing.assert_allclose(rec[e, 0], j * 0.02, rtol=1e-6)
            worst.update(state=max(worst["state"], es))
    assert fl.period == P
    record("random_action_fleet_oracle", f"{integ}/{cost}/E{E}/K{K}", skips=skips, checked=n_checked, **worst)
    # the MAX_COST plugins order plans below the shift by rounding noise, so there the fleet is followed through its own
    # costs only; elsewhere most solves must pick the oracle's plan
    if cost not in SHIFTED:
        assert skips <= n_checked // 4, (skips, n_checked)


@pytest.mark.parametrize("cost", [GRAD, GRADMIN, "quadratic_boundary"])
def test_random_action_fleet_is_bit_identical_to_the_single_solve(cost):
    """Per experiment and period, cps_plan_random_action on an Engine given the experiment's targets, state, u_prev and
    plans gives the fleet's u and J bit for bit (two periods, both target equilibria)."""
    from cartpolesimulation_b200 import _lib as L
    from cartpolesimulation_b200.core import Engine
    E, K, P = 4, 200, 2
    fl = make(E, K, cost, noise="supplied")
    rng = np.random.default_rng(21)
    fl.reset(random_states(E, 22))
    plans = rng.uniform(-1.0, 1.0, (P, E, T, K)).astype(np.float32)
    tp, te = targets(P, E, 23, flip=0)
    eng = Engine(K, T, cost=cost)
    for j in range(P):
        s, u_prev = fl.states(with_u_prev=True)
        J_out = torch.zeros((1, E, K), device="cuda")
        fl.run(1, cuda(tp[j:j + 1]), cuda(te[j:j + 1]), cuda(plans[j:j + 1]), None, J_out)
        _, u_n = fl.states(with_u_prev=True)
        for e in range(E):
            eng.set_variable_parameters(target_position=float(tp[j, e]), target_equilibrium=float(te[j, e]))
            J = torch.empty(K, device="cuda")
            u = eng.plan_random_action(cuda(s[e]), cuda(plans[j, e]), L.TIME_MAJOR, float(u_prev[e]), J_out=J)
            assert float(u.cpu()[0]) == float(u_n[e]), (j, e)
            assert torch.equal(J, J_out[0, e]), (j, e)


def test_random_action_fleet_philox_draws_match_supplied():
    """A Philox fleet and a supplied fleet fed its draws(period) give bit-identical records, costs and states."""
    E, K, P = 4, 200, 6
    a = make(E, K, seed=99, control_limits=(-0.8, 0.6))
    b = make(E, K, noise="supplied", control_limits=(-0.8, 0.6))
    s0 = random_states(E, 5)
    tp, te = targets(P, E, 6, flip=3)
    a.reset(s0)
    b.reset(s0)
    plans = torch.stack([a.draws(j) for j in range(P)]).contiguous()
    assert plans.shape == (P, E, T, K)
    assert float(plans.min()) >= -0.8 and float(plans.max()) < 0.6 and abs(float(plans.mean()) + 0.1) < 0.01
    ra, rb = torch.zeros((P, E, 16), device="cuda"), torch.zeros((P, E, 16), device="cuda")
    Ja, Jb = torch.zeros((P, E, K), device="cuda"), torch.zeros((P, E, K), device="cuda")
    Qa = torch.zeros((P, E, T, K), device="cuda")
    a.run(P, cuda(tp), cuda(te), None, ra, Ja, Qa)
    b.run(P, cuda(tp), cuda(te), plans, rb, Jb)
    assert torch.equal(ra, rb) and torch.equal(Ja, Jb) and torch.equal(Qa, plans)
    for x, y in zip(a.states(with_u_prev=True), b.states(with_u_prev=True)):
        np.testing.assert_array_equal(x, y)
    assert a.period == b.period == P


def test_random_action_fleet_draws_match_restated_philox():
    from cartpolesimulation_b200.fleet import RandomActionFleet
    E, K = 3, 64
    assert T % 4 != 0
    fl = RandomActionFleet(E, num_rollouts=K, mpc_horizon=T, seed=SEED, experiment_offset=OFFSET,
                           control_limits=(-0.7, 0.9))
    fl.reset(np.zeros((E, 6), np.float32), period=2)
    k, e = np.arange(K)[None, :], OFFSET + np.arange(E)[:, None]
    for p in (2, 5):
        want = uniforms(k, RA_DRAWS, p, e, T, -0.7, 0.9).transpose(0, 2, 1)   # [E][T][K]
        np.testing.assert_array_equal(fl.draws(p).cpu().numpy(), want)
    fl.close()


def test_random_action_fleet_split_and_permutation():
    """One fleet of E experiments equals two fleets split by experiment_offset (Philox), and permuting the experiments of a
    supplied fleet permutes every output, bit for bit."""
    E, K, P = 6, 64, 8
    s0 = random_states(E, 8)
    tp, te = targets(P, E, 9, flip=4)
    whole = make(E, K, GRAD, seed=4)
    whole.reset(s0)
    r = torch.zeros((P, E, 16), device="cuda")
    whole.run(P, cuda(tp), cuda(te), None, r)
    parts = []
    for lo, hi in ((0, 2), (2, 6)):
        f = make(hi - lo, K, GRAD, seed=4, experiment_offset=lo)
        f.reset(s0[lo:hi])
        rp = torch.zeros((P, hi - lo, 16), device="cuda")
        f.run(P, cuda(tp[:, lo:hi]), cuda(te[:, lo:hi]), None, rp)
        parts.append(rp)
    assert torch.equal(r, torch.cat(parts, dim=1))
    perm = np.array([3, 0, 5, 1, 4, 2])
    plans = np.random.default_rng(10).uniform(-1.0, 1.0, (P, E, T, K)).astype(np.float32)
    outs = []
    for p in (np.arange(E), perm):
        f = make(E, K, GRAD, noise="supplied")
        f.reset(s0[p])
        rec, J = torch.zeros((P, E, 16), device="cuda"), torch.zeros((P, E, K), device="cuda")
        f.run(P, cuda(tp[:, p]), cuda(te[:, p]), cuda(plans[:, p]), rec, J)
        outs.append([x.cpu().numpy() for x in (rec, J)] + list(f.states(with_u_prev=True)))
    for x, y in zip(outs[0][:2], outs[1][:2]):
        np.testing.assert_array_equal(x[:, perm], y)
    for x, y in zip(outs[0][2:], outs[1][2:]):
        np.testing.assert_array_equal(x[perm], y)


def test_random_action_fleet_nan_target_stays_in_its_experiment():
    """A NaN target makes every cost of that experiment NaN (sorted last): the run completes, the other experiments'
    records are bit-identical to a run without the NaN, and the NaN costs are counted."""
    E, K, P = 4, 200, 6
    s0 = random_states(E, 41)
    tp, te = targets(P, E, 42)
    tp_nan = tp.copy()
    tp_nan[:, 1] = np.nan
    recs, fleets = [], []
    for table in (tp, tp_nan):
        fl = make(E, K, GRAD, seed=5)
        fl.reset(s0)
        r = torch.zeros((P, E, 16), device="cuda")
        fl.run(P, cuda(table), cuda(te), None, r)
        torch.cuda.synchronize()
        recs.append(r.cpu().numpy())
        fleets.append(fl)
    others = [0, 2, 3]
    np.testing.assert_array_equal(recs[1][:, others], recs[0][:, others])
    assert np.all(np.abs(recs[1][:, 1, 9]) <= 1.0)   # the NaN experiment still picks a plan's control
    assert fleets[0].nonfinite_costs() == 0 and fleets[1].nonfinite_costs() >= P * K


class _Draws:
    def __init__(self, draws):
        self.draws, self.i = list(draws), 0

    def uniform(self, shape, minval=0.0, maxval=1.0, dtype=None):
        d = self.draws[self.i]
        self.i += 1
        assert list(d.shape) == list(shape) and (minval, maxval) == (-1.0, 1.0)
        return d


def test_random_action_fleet_agrees_with_optimizer_random_action_b200():
    """optimizer_random_action_b200 driven with the fleet's plans and states, closed loop over 5 periods: the same
    controls, and the plant as oracle.plant_period."""
    import cartpolesimulation_b200 as cps
    from cartpolesimulation_b200.optimizer_forward_b200 import optimizer_random_action_b200
    K, P, tp = 200, 5, 0.03
    fl = make(1, K, seed=12)
    fl.reset(random_states(1, 32))
    vp = cps.VariableParameters(target_position=tp, target_equilibrium=1.0, L=0.395, m_pole=0.087)
    cost, predictor = cps.CostFunctionWrapper(), cps.PredictorWrapper()
    opt = optimizer_random_action_b200(predictor=predictor, cost_function=cost,
                                       control_limits=(np.array([-1.0], np.float32), np.array([1.0], np.float32)), seed=1,
                                       mpc_horizon=T, num_rollouts=K)
    predictor.configure(batch_size=K, horizon=T, dt=0.02, variable_parameters=vp, predictor_specification="ODE")
    cost.configure(batch_size=K, horizon=T, variable_parameters=vp, environment_name="CartPole", computation_library=None,
                   cost_function_specification=GRADMIN)
    opt.configure(num_states=6, num_control_inputs=1, dt=0.02, predictor_specification="ODE")
    opt.rng = _Draws([torch.from_numpy(np.ascontiguousarray(fl.draws(j).cpu().numpy()[0].T)[:, :, None]) for j in range(P)])
    es = 0.0
    for j in range(P):
        s = fl.states()[0]
        u_opt = float(opt.step(s.copy()))
        rec = torch.zeros((1, 1, 16), device="cuda")
        fl.run(1, cuda(np.full((1, 1), tp)), None, None, rec)
        u = float(rec[0, 0, 9])
        assert u == u_opt, (j, u, u_opt)
        s_ref, _, _ = O.plant_period(s, u)
        es = max(es, state_err(fl.states()[0], s_ref))
        assert es < 1e-5, es
    assert opt.rng.i == P
    record("random_action_fleet_optimizer", "gradmin_K200", state=es)


def test_random_action_fleet_launches_per_period():
    """Two launches per period (rollouts with the argmin, plant), whatever E."""
    for E in (1, 300):
        fl = make(E, 200)
        fl.reset(random_states(E, 1))
        n0 = fl.engine.launch_count()
        fl.run(1)
        n1 = fl.engine.launch_count()
        fl.run(3)
        assert n1 - n0 == 2 and fl.engine.launch_count() - n1 == 6


def test_random_action_fleet_rejections():
    from cartpolesimulation_b200 import _lib as L
    from cartpolesimulation_b200.core import Engine
    from cartpolesimulation_b200.fleet import RandomActionFleet
    for kw in (dict(integrator="neural"), dict(cost=None), dict(num_rollouts=8193)):
        with pytest.raises(NotImplementedError):
            RandomActionFleet(2, **kw)
    with pytest.raises(ValueError):
        RandomActionFleet(2, dt_simulation=0.003)
    fl = RandomActionFleet(2)
    with pytest.raises(NotImplementedError):
        fl.set_plant_models(latency=0.01)
    with pytest.raises(RuntimeError):          # CPS_ERR_NOT_CONFIGURED before reset()
        fl.run(1)
    with pytest.raises(RuntimeError):
        fl.states()
    fl.reset(np.zeros((2, 6), np.float32))
    with pytest.raises(ValueError):            # a Philox fleet draws its own numbers
        fl.run(1, plans=torch.zeros((1, 2, T, 200), device="cuda"))
    sup = RandomActionFleet(2, noise="supplied")
    sup.reset(np.zeros((2, 6), np.float32))
    with pytest.raises(ValueError):            # and a supplied one needs them
        sup.run(1)
    with pytest.raises(ValueError):            # of the right size
        sup.run(1, plans=torch.zeros((1, 2, T, 100), device="cuda"))
    # the C ABI's own checks
    def cfg(**kw):
        c = L.cps_random_action_fleet_config(C.sizeof(L.cps_random_action_fleet_config), 2, 10, L.FLEET_NOISE_PHILOX,
                                             0.002, 0, 0)
        for k, v in kw.items():
            setattr(c, k, v)
        return C.byref(c)
    eng = Engine(200, T)
    assert eng.lib.cps_random_action_fleet_step(eng._h, 1, None, None, None, None, None, None) == 4
    assert eng.lib.cps_random_action_fleet_create(eng._h, cfg(sim_substeps=7)) == 1
    assert eng.lib.cps_random_action_fleet_create(eng._h, cfg(n_experiments=65536)) == 1
    assert eng.lib.cps_random_action_fleet_create(eng._h, cfg(struct_size=8)) == 1
    assert eng.lib.cps_random_action_fleet_create(eng._h, cfg(draw_source=7)) == 1
    assert eng.lib.cps_random_action_fleet_create(eng._h, cfg()) == 0
    assert eng.lib.cps_random_action_fleet_step(eng._h, 1, None, None, None, None, None, None) == 4   # no states yet
    for args, kw in (((200, T), dict(substep_sincos=True)), ((200, T), dict(fast_div=True)),
                     ((200, T), dict(integrator="neural")), ((9000, T), {}),
                     ((200, T), dict(cost="legacy_mppi", noise_mode="direct"))):
        other = Engine(*args, **kw)
        assert other.lib.cps_random_action_fleet_create(other._h, cfg()) == 3, (args, kw)


def test_random_action_fleet_records_write_the_reference_csv(tmp_path):
    from cartpolesimulation_b200.fleet import make_experiments
    from cartpolesimulation_b200.recording import save_fleet_recordings
    E, P = 3, 20
    s0, tp, te = make_experiments(E, P, seed=2)
    fl = make(E, 200, seed=2)
    fl.reset(s0)
    rec = torch.zeros((P, E, 16), device="cuda")
    fl.run(P, cuda(tp), cuda(te), None, rec)
    r = rec.cpu().numpy()
    assert np.all(np.isfinite(r)) and np.all(np.abs(r[:, :, 9]) <= 1.0)
    paths = save_fleet_recordings(rec, str(tmp_path), optimizer_name="random-action-b200", run_for_ML_Pipeline=False)
    assert len(paths) == E
    with open(paths[1]) as f:
        rows = [row for row in csv.reader(line for line in f if not line.startswith("#"))]
    assert rows[0][:15] == ["time", "angle", "angleD", "angleDD", "angle_cos", "angle_sin", "position", "positionD",
                            "positionDD", "Q_calculated", "Q_applied", "Q_ccrc", "u", "target_position", "target_equilibrium"]
    assert len(rows) == P + 1
    np.testing.assert_allclose(np.array([float(x[1]) for x in rows[1:]]), r[:, 1, 1], rtol=1e-6, atol=1e-6)
