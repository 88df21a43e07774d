"""Legacy controller fleets (cps_legacy_fleet_*, fleet.LegacyFleet): E closed-loop experiments under
controller_mppi_cartpole, against the single controller (controller_mppi_cartpole_b200 fed the fleet's draws through a
stub generator, bit for bit), the single solve (Engine.legacy_step), the float64 oracle (oracle/legacy.py iteration +
oracle.plant_period), a numpy restatement of the Philox draws, a supplied fleet, a split over two fleets and a
permutation of the experiments."""
import csv

import numpy as np
import pytest
import torch

from oracle import legacy as OL
from oracle import oracle as O
from tests.test_gpu_fleet_core import OFFSET, SEED, normals, philox4x32_10

pytestmark = pytest.mark.gpu

LEGACY_DRAWS, LEGACY_ACT = 0xF0000000, 0xFFFFFF00   # cps_plant.cuh
RANGES = np.array([np.pi, 18.38, 1.0, 1.0, 0.198, 1.125], dtype=np.float64)
SAMPLINGS = ["iid", "random_walk", "uniform", "repeated", "interpolated"]


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def state_err(a, b):
    d = np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64))
    d[..., 0] = np.minimum(d[..., 0], 2 * np.pi - d[..., 0])
    return float((d / RANGES).max())


def random_states(E, seed):
    from cartpolesimulation_b200.fleet import DataGenConfig, random_initial_state
    rng = np.random.default_rng(seed)
    return np.stack([random_initial_state(rng, DataGenConfig()) for _ in range(E)])


def make(E, K=300, T=35, sampling="interpolated", predictor="ODE", update_every=1, p_Q=0.0, **kw):
    from cartpolesimulation_b200.fleet import LegacyFleet
    return LegacyFleet(E, dict(num_rollouts=K, mpc_horizon=T, SAMPLING_TYPE=sampling, predictor_specification=predictor,
                               update_every=update_every, seed=1), actuator_noise=p_Q, **kw)


class StubRng:
    """Stands in for the mirror's numpy Generator: returns one experiment's fleet draws in the reference's call order."""

    def __init__(self):
        self.queue = []

    def load(self, sampling, raw, act):
        """raw [K, n_draws] of a solve period (None: an advance period), act the actuator uniform."""
        if raw is not None:
            if sampling in ("random_walk", "uniform"):
                self.queue += [("u" if sampling == "uniform" else "n", np.ascontiguousarray(raw[:, t])) for t in range(raw.shape[1])]
            else:
                self.queue.append(("n", raw))
        self.queue.append(("a", float(act)))

    def standard_normal(self, size, dtype=np.float64):
        kind, v = self.queue.pop(0)
        assert kind == "n" and v.size == int(np.prod(size)) and dtype == np.float32
        return v.reshape(size)

    def uniform(self, low=0.0, high=1.0, size=None):
        kind, v = self.queue.pop(0)
        assert (low, high) == (-1.0, 1.0)
        if size is None:
            assert kind == "a"
            return v
        assert kind == "u" and v.size == int(np.prod(size))
        return v.astype(np.float64)


def mirrors(fl, E, K, T, sampling, predictor, update_every, p_Q):
    from cartpolesimulation_b200.controller_mppi_cartpole_b200 import controller_mppi_cartpole_b200
    out = []
    for _ in range(E):
        c = controller_mppi_cartpole_b200(dict(num_rollouts=K, mpc_horizon=T, SAMPLING_TYPE=sampling, seed=1,
                                               predictor_specification=predictor, update_every=update_every),
                                          actuator_noise=p_Q)
        c.rng_mppi = StubRng()
        out.append(c)
    return out


BIT_CASES = [  # E, K, T, sampling, predictor, update_every, p_Q
    (1, 300, 35, "interpolated", "ODE", 1, 0.0),
    (3, 300, 35, "iid", "ODE_v0", 3, 0.1),
    (3, 100, 35, "random_walk", "ODE", 1, 0.1),
    (3, 300, 20, "uniform", "ODE_v0", 1, 0.0),
    (3, 300, 35, "repeated", "ODE", 3, 0.0),
    (37, 300, 35, "interpolated", "ODE_v0", 1, 0.1),
    (3, 3500, 35, "interpolated", "ODE", 1, 0.1),
    (3, 3500, 35, "iid", "ODE_v0", 3, 0.0),
]


@pytest.mark.parametrize("E,K,T,sampling,predictor,update_every,p_Q", BIT_CASES)
def test_legacy_fleet_is_bit_identical_to_the_single_controller(E, K, T, sampling, predictor, update_every, p_Q):
    """Each experiment equals its own controller_mppi_cartpole_b200 stepped on the fleet's recorded states with a stub
    generator that returns the fleet's draws: Q, u, u_prev every period for 12 periods, bit for bit (K = 300 and 100 have
    a partial last block).  The solve periods' costs equal Engine.legacy_step's on the same perturbations."""
    from cartpolesimulation_b200.core import Engine
    P = 12
    fl = make(E, K, T, sampling, predictor, update_every, p_Q, seed=7)
    fl.reset(random_states(E, 3))
    tp = np.random.default_rng(4).uniform(-0.1, 0.1, (P, E)).astype(np.float32)
    ctl = mirrors(fl, E, K, T, sampling, predictor, update_every, p_Q)
    eng = Engine(K, T, dt=0.02, substeps=10, integrator=predictor, cost="legacy_mppi", noise_mode="direct")
    eng.set_cost_params([ctl[0].dd_weight, ctl[0].ep_weight, ctl[0].ekp_weight, ctl[0].ekc_weight, ctl[0].ccrc_weight])
    eng.set_mppi_params(cc_weight=ctl[0].cc_weight, R=ctl[0].R, LBD=ctl[0].LBD, NU=ctl[0].NU)
    for j in range(P):
        solve = fl.solves(j)
        raw = fl.draws(j).cpu().numpy() if solve else None
        act = fl.act_draws(j).cpu().numpy()
        du = fl.perturbations(j) if solve else None
        u0, up0 = fl.inputs()
        rec, S = torch.zeros((1, E, 16), device="cuda"), torch.full((1, E, K), -1.0, device="cuda")
        fl.run(1, cuda(tp[j:j + 1]), None, None, None, rec, S)
        rec, S = rec.cpu().numpy()[0], S.cpu().numpy()[0]
        u1, up1 = fl.inputs()
        for e in range(E):
            ctl[e].rng_mppi.load(sampling, None if raw is None else raw[e], act[e])
            s = rec[e, [1, 2, 4, 5, 6, 7]]
            Q = ctl[e].step(s.copy(), updated_attributes={"target_position": float(tp[j, e])})
            assert not ctl[e].rng_mppi.queue, (j, e)
            assert np.float32(Q) == rec[e, 9] == rec[e, 10], (j, e, Q, rec[e, 9])
            u_m, up_m = ctl[e]._pull_inputs()
            np.testing.assert_array_equal(u1[e], u_m)
            np.testing.assert_array_equal(up1[e], up_m)
            if solve:
                np.testing.assert_array_equal(du[e].cpu().numpy(), ctl[e].delta_u.astype(np.float32))
                eng.set_variable_parameters(target_position=float(tp[j, e]))
                eng.legacy_set_inputs(u0[e], up0[e])
                S_ref = torch.empty(K, device="cuda")
                eng.legacy_step(cuda(s), du[e].contiguous(), S_out=S_ref)
                np.testing.assert_array_equal(S[e], S_ref.cpu().numpy())
            else:
                assert np.all(S[e] == -1.0)
    assert fl.period == P


@pytest.mark.parametrize("predictor", ["ODE", "ODE_v0"])
def test_legacy_fleet_matches_oracle_teacher_forced(predictor):
    """oracle/legacy.py iteration + oracle.plant_period from the fleet's own state, u, u_prev and perturbations each
    period: costs by cost_agreement, controls within 1e-4 (the updated sequence within 2e-4), the plant state as in the
    other fleet tests."""
    from tests.test_gpu_legacy import cost_agreement
    E, K, T, P, p_Q = 3, 500, 35, 8, 0.1
    fl = make(E, K, T, "interpolated", predictor, 1, p_Q, seed=2)
    fl.reset(random_states(E, 8))
    tp = np.full((P, E), 0.05, np.float32)
    for j in range(P):
        s = fl.states()
        u0, up0 = fl.inputs()
        du = fl.perturbations(j).cpu().numpy()
        act = fl.act_draws(j).cpu().numpy()
        rec, S = torch.zeros((1, E, 16), device="cuda"), torch.zeros((1, E, K), device="cuda")
        fl.run(1, cuda(tp[j:j + 1]), None, None, None, rec, S)
        rec, S = rec.cpu().numpy()[0], S.cpu().numpy()[0]
        s1 = fl.states()
        u1, up1 = fl.inputs()
        for e in range(E):
            o = OL.iteration(predictor, s[e], u0[e], up0[e], du[e], target_position=float(tp[j, e]))
            frac, worst = cost_agreement(S[e], o["S"])
            assert frac > 0.995, (j, e, frac, worst)
            # the control within 1e-4; the rest of the updated sequence within 2e-4 (its later steps average
            # perturbations over the same float32-rounded weights and reach 1.1e-4 from a fleet state after a few periods)
            assert abs(up1[e][0] - o["u_updated"][0]) < 1e-4
            assert np.max(np.abs(up1[e] - o["u_updated"])) < 2e-4
            Q_ref = np.clip(np.float32(float(o["Q_raw"]) * (1 + p_Q * float(act[e]))), -1.0, 1.0)
            assert abs(rec[e, 9] - Q_ref) < 1e-4
            s_ref, _, _ = O.plant_period(s[e], float(rec[e, 9]))
            assert state_err(s1[e], s_ref) < 1e-5


@pytest.mark.parametrize("sampling", SAMPLINGS)
def test_legacy_fleet_draws_match_restated_philox_and_supplied(sampling):
    """draws(period) equals the numpy Philox restatement, and a supplied fleet fed a Philox fleet's draws / act_draws
    gives bit-identical records, costs, inputs and states."""
    E, K, T, P = 3, 64, 23, 5
    a = make(E, K, T, sampling, update_every=2, p_Q=0.1, seed=SEED, experiment_offset=OFFSET)
    b = make(E, K, T, sampling, update_every=2, p_Q=0.1, noise="supplied")
    s0 = random_states(E, 5)
    a.reset(s0, period=1)
    b.reset(s0, period=1)
    k, e = np.arange(K)[None, :], OFFSET + np.arange(E)[:, None]
    n = a.n_draws
    for p in (1, 4):
        got = a.draws(p).cpu().numpy()
        if sampling == "uniform":
            words = []
            for g in range((n + 3) // 4):
                words += philox4x32_10(k, LEGACY_DRAWS + g, p, e, SEED)
            u = np.stack([(w >> np.uint64(8)).astype(np.float32) * np.float32(2.0 ** -24) for w in words[:n]], -1)
            np.testing.assert_array_equal(got, (np.float32(-1.0) + np.float32(2.0) * u).astype(np.float32))
        else:
            np.testing.assert_allclose(got, normals(k, LEGACY_DRAWS, p, e, n), rtol=1e-6, atol=1e-6)
        w = philox4x32_10(0, LEGACY_ACT, p, e[:, 0], SEED)[0]
        want = np.float32(-1.0) + np.float32(2.0) * ((w >> np.uint64(8)).astype(np.float32) * np.float32(2.0 ** -24))
        np.testing.assert_array_equal(a.act_draws(p).cpu().numpy(), want.astype(np.float32))
    draws = torch.stack([a.draws(1 + j) for j in range(P)]).contiguous()
    acts = torch.stack([a.act_draws(1 + j) for j in range(P)]).contiguous()
    ra, rb = torch.zeros((P, E, 16), device="cuda"), torch.zeros((P, E, 16), device="cuda")
    Sa, Sb = torch.zeros((P, E, K), device="cuda"), torch.zeros((P, E, K), device="cuda")
    a.run(P, None, None, None, None, ra, Sa)
    b.run(P, None, None, draws, acts, rb, Sb)
    assert torch.equal(ra, rb) and torch.equal(Sa, Sb)
    for x, y in zip(a.inputs() + a.states(with_u_prev=True), b.inputs() + b.states(with_u_prev=True)):
        np.testing.assert_array_equal(x, y)
    assert a.period == b.period == P + 1


def test_legacy_fleet_split_and_permutation():
    """One fleet equals two fleets split by experiment_offset (Philox); permuting the experiments of a supplied fleet
    permutes every output, bit for bit."""
    E, K, P = 6, 200, 6
    s0 = random_states(E, 8)
    tp = np.random.default_rng(9).uniform(-0.1, 0.1, (P, E)).astype(np.float32)
    whole = make(E, K, p_Q=0.1, seed=4)
    whole.reset(s0)
    r = torch.zeros((P, E, 16), device="cuda")
    whole.run(P, cuda(tp), None, record=r)
    parts = []
    for lo, hi in ((0, 2), (2, 6)):
        f = make(hi - lo, K, p_Q=0.1, seed=4, experiment_offset=lo)
        f.reset(s0[lo:hi])
        rp = torch.zeros((P, hi - lo, 16), device="cuda")
        f.run(P, cuda(tp[:, lo:hi]), None, record=rp)
        parts.append(rp)
    assert torch.equal(r, torch.cat(parts, dim=1))
    perm = np.array([3, 0, 5, 1, 4, 2])
    rng = np.random.default_rng(10)
    n_draws = whole.n_draws
    draws = rng.standard_normal((P, E, K, n_draws)).astype(np.float32)
    acts = rng.uniform(-1.0, 1.0, (P, E)).astype(np.float32)
    outs = []
    for p in (np.arange(E), perm):
        f = make(E, K, p_Q=0.1, noise="supplied")
        f.reset(s0[p])
        rec, S = torch.zeros((P, E, 16), device="cuda"), torch.zeros((P, E, K), device="cuda")
        f.run(P, cuda(tp[:, p]), None, cuda(draws[:, p]), cuda(acts[:, p]), rec, S)
        outs.append([x.cpu().numpy() for x in (rec, S)] + list(f.inputs()) + list(f.states(with_u_prev=True)))
    for x, y in zip(outs[0][:2], outs[1][:2]):
        np.testing.assert_array_equal(x[:, perm], y)
    for x, y in zip(outs[0][2:], outs[1][2:]):
        np.testing.assert_array_equal(x[perm], y)


def test_legacy_fleet_nan_target_stays_in_its_experiment():
    E, K, P = 4, 200, 5
    s0 = random_states(E, 41)
    tp = np.full((P, E), 0.02, np.float32)
    tp_nan = tp.copy()
    tp_nan[:, 1] = np.nan
    recs, fleets = [], []
    for table in (tp, tp_nan):
        fl = make(E, K, p_Q=0.1, seed=5)
        fl.reset(s0)
        r = torch.zeros((P, E, 16), device="cuda")
        fl.run(P, cuda(table), None, record=r)
        torch.cuda.synchronize()
        recs.append(r.cpu().numpy())
        fleets.append(fl)
    others = [0, 2, 3]
    np.testing.assert_array_equal(recs[1][:, others], recs[0][:, others])
    assert fleets[0].nonfinite_costs() == 0 and fleets[1].nonfinite_costs() >= K


def test_legacy_fleet_launches_per_period():
    """One launch per period, solve or advance, Philox or supplied, whatever E."""
    for E in (1, 300):
        for noise in ("philox", "supplied"):
            fl = make(E, 300, update_every=2, noise=noise)
            fl.reset(random_states(E, 1))
            kw = {}
            if noise == "supplied":
                kw = dict(draws=torch.zeros((3, E, 300, fl.n_draws), device="cuda"), act_draws=torch.zeros((3, E), device="cuda"))
            n0 = fl.engine.launch_count()
            fl.run(3, **kw)
            assert fl.engine.launch_count() - n0 == 3, (E, noise)


def test_legacy_fleet_advance_rows_and_csv(tmp_path):
    """With update_every = 3 the advance periods' rows follow the mirror's shift (Q = the previous solve's u[1], u[2]),
    and save_fleet_recordings writes the reference's CSV with `Controller: mppi-cartpole`."""
    from cartpolesimulation_b200.recording import save_fleet_recordings
    E, K, P = 3, 300, 7
    fl = make(E, K, update_every=3, seed=2)
    fl.reset(random_states(E, 2))
    rec = torch.zeros((P, E, 16), device="cuda")
    ups = []
    for j in range(P):
        fl.run(1, None, None, record=rec[j:j + 1])
        ups.append(fl.inputs()[1])
    r = rec.cpu().numpy()
    for j in (1, 2, 4, 5):   # Q = the last solve's u[j - solve]
        s = j - j % 3
        np.testing.assert_array_equal(r[j, :, 9], np.clip(ups[s][:, j - s], -1.0, 1.0))
    assert np.all(np.isfinite(r)) and np.all(np.abs(r[:, :, 9]) <= 1.0)
    paths = save_fleet_recordings(rec, str(tmp_path), controller_name="mppi-cartpole", optimizer_name=None,
                                  run_for_ML_Pipeline=False)
    assert len(paths) == E
    with open(paths[1]) as f:
        text = f.read()
    assert "Controller: mppi-cartpole" in text
    rows = [row for row in csv.reader(line for line in text.splitlines() if not line.startswith("#"))]
    assert rows[0][:15] == ["time", "angle", "angleD", "angleDD", "angle_cos", "angle_sin", "position", "positionD",
                            "positionDD", "Q_calculated", "Q_applied", "Q_ccrc", "u", "target_position", "target_equilibrium"]
    assert len(rows) == P + 1


def test_legacy_fleet_rejections():
    import ctypes as C
    from cartpolesimulation_b200 import _lib as L
    from cartpolesimulation_b200.core import Engine
    fl = make(2, 200)
    with pytest.raises(NotImplementedError):
        fl.set_plant_models(latency=0.01)
    with pytest.raises(RuntimeError):          # CPS_ERR_NOT_CONFIGURED before reset()
        fl.states()
    fl.reset(np.zeros((2, 6), np.float32))
    with pytest.raises(ValueError):            # a Philox fleet draws its own numbers
        fl.run(1, act_draws=torch.zeros((1, 2), device="cuda"))
    sup = make(2, 200, noise="supplied")
    sup.reset(np.zeros((2, 6), np.float32))
    with pytest.raises(ValueError):            # and a supplied one needs them
        sup.run(1)
    with pytest.raises(ValueError):            # a supplied fleet has no draws of its own
        sup.perturbations(0)

    def cfg(**kw):
        c = L.cps_legacy_fleet_config(C.sizeof(L.cps_legacy_fleet_config), 2, 10, L.FLEET_NOISE_PHILOX, 0.002, 0, 0, 4, 1,
                                      0.14, 0.0)
        for k, v in kw.items():
            setattr(c, k, v)
        return C.byref(c)
    eng = Engine(200, 35, cost="legacy_mppi", noise_mode="direct")
    assert eng.lib.cps_legacy_fleet_step(eng._h, 1, None, None, None, None, None, None) == 4   # no fleet
    for bad in (dict(sim_substeps=7), dict(n_experiments=65536), dict(struct_size=8), dict(draw_source=7),
                dict(sampling_type=5), dict(update_every=0)):
        assert eng.lib.cps_legacy_fleet_create(eng._h, cfg(**bad)) == 1, bad
    assert eng.lib.cps_legacy_fleet_create(eng._h, cfg()) == 0
    assert eng.lib.cps_legacy_fleet_step(eng._h, 1, None, None, None, None, None, None) == 4   # no states yet
    other = Engine(200, 35)
    assert other.lib.cps_legacy_fleet_create(other._h, cfg()) == 4   # not a legacy handle
