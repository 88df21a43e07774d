"""Random action, CEM and CEM-GMM on the neural predictor (cps_plan_random_action, cps_cem_step, cps_cem_gmm_step and
their fleets with CPS_PREDICTOR_NEURAL): the costs are those of cps_plan_cost on the sampled plans bit for bit and match
the float64 restatement oracle/net_grad.py; the selection and update, teacher-forced on the GPU's costs, are the
oracle's; fleets are bit-identical to the single solves; the stored hidden state is read and never written."""
import numpy as np
import pytest

from tests.test_gpu_net_grad import GRADMIN, J_BOUND, NETS, QBGRAD, _engine, _h_after, _spec, _state

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _oracle_J(sp, cost, s, Q, u_prev, tp, te, h0):
    from oracle import net_grad as NG
    from tests.test_gpu_net_grad import _cost_cfg
    return NG.plan_cost(sp, cost, s, torch.from_numpy(np.asarray(Q, np.float64)), u_prev, tp, te, _cost_cfg(cost, te),
                        None if h0 is None else torch.from_numpy(h0.astype(np.float64))).numpy()


def _rel(a, b):
    return float(np.abs(np.asarray(a, np.float64) - b).max() / max(np.abs(b).max(), 1e-30))


def _gpu_costs(monkeypatch, eng, s, u_prev):
    """oracle.plan_cost answered by the GPU's cps_plan_cost on the oracle's plans (teacher forcing)."""
    from cartpolesimulation_b200 import _lib as L
    from oracle import oracle as O

    def pc(integrator, cost_name, s_, Q, u_prev_=0.0, **kw):
        J, _ = eng.plan_cost(cuda(s), cuda(np.asarray(Q, np.float32)), L.ROLLOUT_MAJOR, u_prev)
        return J.cpu().numpy()
    monkeypatch.setattr(O, "plan_cost", pc)


CASES = [("gru32", None, GRADMIN, 1.0), ("gru32", "h", QBGRAD, -1.0), ("gru64", "h", GRADMIN, -1.0), ("dense32", None, QBGRAD, 1.0)]


@pytest.mark.parametrize("net,h,cost,te", CASES)
@pytest.mark.parametrize("K,T", [(64, 35), (200, 35), (300, 23)])
def test_random_action_neural(net, h, cost, te, K, T):
    from cartpolesimulation_b200 import _lib as L
    sp = _spec(net)
    h0 = _h_after(net) if h else None
    eng = _engine(sp, K, T, cost, 0.05, te, h0)
    hs = eng.net_get_state().copy()
    rng = np.random.default_rng(K + T)
    s = _state(K)
    Q = rng.uniform(-1, 1, (K, T)).astype(np.float32)
    J = torch.empty(K, device="cuda")
    u = float(eng.plan_random_action(cuda(s), cuda(Q), L.ROLLOUT_MAJOR, 0.3, J_out=J).cpu()[0])
    Jc, _ = eng.plan_cost(cuda(s), cuda(Q), L.ROLLOUT_MAJOR, 0.3)
    assert torch.equal(J, Jc)
    Jn = J.cpu().numpy()
    assert u == Q[int(np.argsort(Jn, kind="stable")[0]), 0]
    assert _rel(Jn, _oracle_J(sp, cost, s, Q, 0.3, 0.05, te, h0)) < J_BOUND
    # time-major plans and the host form give the same control
    assert float(eng.plan_random_action(cuda(s), cuda(Q.T), L.TIME_MAJOR, 0.3).cpu()[0]) == u
    assert eng.plan_random_action_host(s, cuda(Q), L.ROLLOUT_MAJOR, 0.3) == u
    np.testing.assert_array_equal(eng.net_get_state(), hs)


@pytest.mark.parametrize("net,h,cost,te", CASES)
@pytest.mark.parametrize("K,T,its,best_k", [(64, 35, 1, 8), (200, 35, 3, 40), (300, 17, 2, 150)])
def test_cem_neural(monkeypatch, net, h, cost, te, K, T, its, best_k):
    from cartpolesimulation_b200 import _lib as L
    from oracle import oracle as O
    sp = _spec(net)
    h0 = _h_after(net) if h else None
    eng = _engine(sp, K, T, cost, -0.1, te, h0)
    eng.cem_configure(best_k, 0.5, 0.01)
    hs = eng.net_get_state().copy()
    rng = np.random.default_rng(K * its)
    s, u_prev = _state(T), -0.2
    mu = rng.uniform(-0.3, 0.3, T).astype(np.float32)
    sd = rng.uniform(0.2, 0.6, T).astype(np.float32)
    eng.cem_set_distribution(mean=mu, stdev=sd)
    eps = rng.normal(0, 1, (its, K, T)).astype(np.float32)
    Qo, Jo = torch.empty((K, T), device="cuda"), torch.empty(K, device="cuda")
    u = float(eng.cem_step(cuda(s), cuda(eps), L.ROLLOUT_MAJOR, u_prev, Q_out=Qo, J_out=Jo).cpu()[0])
    mu_g, sd_g = eng.cem_get_distribution()
    # the last iteration's costs are cps_plan_cost's on its plans, and the network restatement's
    Jc, _ = eng.plan_cost(cuda(s), Qo, L.ROLLOUT_MAJOR, u_prev)
    assert torch.equal(Jo, Jc)
    assert _rel(Jo.cpu().numpy(), _oracle_J(sp, cost, s, Qo.cpu().numpy(), u_prev, -0.1, te, h0)) < J_BOUND
    np.testing.assert_array_equal(eng.net_get_state(), hs)
    # selection and update teacher-forced on the GPU's costs
    _gpu_costs(monkeypatch, eng, s, u_prev)
    ref = O.cem_step("neural", cost, s, eps, mu, sd, best_k, 0.01, 0.5, u_prev)
    if its == 1:
        np.testing.assert_array_equal(Qo.cpu().numpy(), ref["Q"])
    assert abs(u - ref["u"]) < 1e-6
    np.testing.assert_allclose(mu_g, ref["mean"], rtol=0, atol=2e-6)
    np.testing.assert_allclose(sd_g, ref["stdev"], rtol=0, atol=2e-6)


@pytest.mark.parametrize("net,h,cost,te", CASES[:3])
@pytest.mark.parametrize("K,T,its,best_k", [(64, 35, 1, 2), (200, 35, 3, 40), (300, 19, 2, 300)])
def test_cem_gmm_neural(monkeypatch, net, h, cost, te, K, T, its, best_k):
    from cartpolesimulation_b200 import _lib as L
    from oracle import oracle as O
    sp = _spec(net)
    h0 = _h_after(net) if h else None
    eng = _engine(sp, K, T, cost, 0.0, te, h0)
    eng.cem_gmm_configure(best_k, 0.5, 0.01)
    hs = eng.net_get_state().copy()
    rng = np.random.default_rng(K + best_k)
    s, u_prev = _state(best_k), 0.1
    eps = rng.normal(0, 1, (its, K, T, 2)).astype(np.float32)
    u01 = rng.uniform(0, 1, (its, K, T)).astype(np.float32)
    Qo, Jo = torch.empty((K, T), device="cuda"), torch.empty(K, device="cuda")
    u = float(eng.cem_gmm_step(cuda(s), cuda(eps), cuda(u01), L.ROLLOUT_MAJOR, u_prev, Q_out=Qo, J_out=Jo).cpu()[0])
    loc, scale, p1 = eng.cem_gmm_get_distribution()
    Jc, _ = eng.plan_cost(cuda(s), Qo, L.ROLLOUT_MAJOR, u_prev)
    assert torch.equal(Jo, Jc)
    assert _rel(Jo.cpu().numpy(), _oracle_J(sp, cost, s, Qo.cpu().numpy(), u_prev, 0.0, te, h0)) < J_BOUND
    np.testing.assert_array_equal(eng.net_get_state(), hs)
    _gpu_costs(monkeypatch, eng, s, u_prev)
    ref = O.cem_gmm_step("neural", cost, s, eps, u01, np.zeros((T, 2)), np.full((T, 2), 0.5), 0.5, best_k, 0.01, u_prev)
    if its == 1:
        np.testing.assert_array_equal(Qo.cpu().numpy(), ref["Q"])
    assert abs(u - ref["u"]) < 1e-6
    np.testing.assert_allclose(loc.T, ref["loc"], rtol=0, atol=2e-6)
    np.testing.assert_allclose(scale.T, ref["scale"], rtol=0, atol=2e-6)
    assert abs(p1 - ref["p1"]) < 1e-6


# ---- fleets ---------------------------------------------------------------------------------------------------------
KINDS = ("cem", "gmm", "ra")


def _fleet(kind, E, K, T, net="gru32", noise="supplied", integrator="neural", **kw):
    from cartpolesimulation_b200.fleet import CemFleet, CemGmmFleet, RandomActionFleet
    from tests.test_gpu_net_grad import _engine_spec
    cls = dict(cem=CemFleet, gmm=CemGmmFleet, ra=RandomActionFleet)[kind]
    if kind != "ra":
        kw.setdefault("cem_best_k", 12)
    network = _engine_spec(_spec(net)) if integrator == "neural" else None
    return cls(E, num_rollouts=K, mpc_horizon=T, integrator=integrator, noise=noise, network=network, device=0, **kw)


def _states(E, seed):
    from tests.test_gpu_fleet_random_action import random_states
    return random_states(E, seed)


def _draws(kind, fl, P, rng):
    E, K, T = fl.E, fl.K, fl.T
    if kind == "cem":
        return (cuda(rng.normal(0, 1, (P * fl.outer_its, E, T, K)).astype(np.float32)),)
    if kind == "gmm":
        return (cuda(rng.normal(0, 1, (P * fl.outer_its, E, 2, T, K)).astype(np.float32)),
                cuda(rng.uniform(0, 1, (P * fl.outer_its, E, T, K)).astype(np.float32)))
    return (cuda(rng.uniform(-1, 1, (P, E, T, K)).astype(np.float32)),)


def _run(kind, fl, P, tp, te, draws, rec, J, Q):
    if kind == "gmm":
        return fl.run(P, tp, te, draws[0], draws[1], rec, J, Q)
    return fl.run(P, tp, te, draws[0], rec, J, Q)


@pytest.mark.parametrize("kind,best_k", [("cem", 12), ("cem", 64), ("gmm", 12), ("ra", 0)])
@pytest.mark.parametrize("E,P", [(1, 12), (3, 12), (37, 12)])
def test_neural_fleet_is_bit_identical_to_the_single_solve(kind, best_k, E, P):
    """Per experiment and period the single solve from the fleet's state, distribution, u_prev, targets and draws gives
    the fleet's u, costs, plans and distribution bit for bit; the plant period then follows oracle.plant_period."""
    from cartpolesimulation_b200 import _lib as L
    from oracle import oracle as O
    from tests.test_gpu_fleet_random_action import targets
    K, T = 64, 35   # CEM best_k 64: best_k x T > 2048, the statistics in cem_update(_fleet)_kernel
    h = _h_after("gru32")   # a non-zero stored hidden state, shared by every rollout of fleet and single solve
    fl = _fleet(kind, E, K, T, cost=QBGRAD, **({"cem_best_k": best_k} if best_k else {}))
    fl.engine.net_set_state(h)
    fl.reset(_states(E, 3))
    rng = np.random.default_rng(4)
    draws = _draws(kind, fl, P, rng)
    tp, te = targets(P, E, 5, flip=1)
    from cartpolesimulation_b200.core import Engine
    from tests.test_gpu_net_grad import _engine_spec
    eng = Engine(K, T, integrator="neural", cost=QBGRAD, device=0)   # the fleet's default cost weights
    eng.net_load(_engine_spec(_spec("gru32")))
    eng.set_mppi_params(lo=-1.0, hi=1.0)
    eng.net_set_state(h)
    if kind == "cem":
        eng.cem_configure(best_k, 0.5, 0.01)
    if kind == "gmm":
        eng.cem_gmm_configure(best_k, 0.5, 0.01)
    n_it = 1 if kind == "ra" else fl.outer_its
    for j in range(P):
        s, u_prev = fl.states(with_u_prev=True)
        dist = fl.distribution() if kind != "ra" else None
        J, Q = torch.zeros((1, E, K), device="cuda"), torch.zeros((1, E, T, K), device="cuda")
        _run(kind, fl, 1, cuda(tp[j:j + 1]), cuda(te[j:j + 1]), [d[j * n_it:(j + 1) * n_it] for d in draws], None, J, Q)
        s_n, u_n = fl.states(with_u_prev=True)
        dist_n = fl.distribution() if kind != "ra" else None
        for e in range(E):
            eng.set_variable_parameters(target_position=float(tp[j, e]), target_equilibrium=float(te[j, e]))
            Je, Qe = torch.empty(K, device="cuda"), torch.empty((T, K), device="cuda")
            if kind == "ra":
                u = eng.plan_random_action(cuda(s[e]), draws[0][j, e].contiguous(), L.TIME_MAJOR, float(u_prev[e]), J_out=Je)
                Qe = draws[0][j, e]
            elif kind == "cem":
                eng.cem_set_distribution(mean=dist[0][e], stdev=dist[1][e])
                u = eng.cem_step(cuda(s[e]), draws[0][j * n_it:(j + 1) * n_it, e].contiguous(), L.TIME_MAJOR,
                                 float(u_prev[e]), Q_out=Qe, J_out=Je)
                np.testing.assert_array_equal(eng.cem_get_distribution()[0], dist_n[0][e])
                np.testing.assert_array_equal(eng.cem_get_distribution()[1], dist_n[1][e])
            else:
                eng.cem_gmm_set_distribution(dist[0][e], dist[1][e], dist[2][e])
                u = eng.cem_gmm_step(cuda(s[e]), draws[0][j * n_it:(j + 1) * n_it, e].contiguous(),
                                     draws[1][j * n_it:(j + 1) * n_it, e].contiguous(), L.TIME_MAJOR, float(u_prev[e]),
                                     Q_out=Qe, J_out=Je)
                for a, b in zip(eng.cem_gmm_get_distribution(), (dist_n[0][e], dist_n[1][e], dist_n[2][e])):
                    np.testing.assert_array_equal(a, b)
            assert float(u.cpu()[0]) == float(u_n[e]), (j, e)
            assert torch.equal(Je, J[0, e]), (j, e)
            assert torch.equal(Qe, Q[0, e]), (j, e)
            s_ref, _, _ = O.plant_period(s[e], float(u_n[e]))
            np.testing.assert_allclose(s_n[e], s_ref, rtol=0, atol=1e-5)
    np.testing.assert_array_equal(eng.net_get_state(), h)
    np.testing.assert_array_equal(fl.engine.net_get_state(), h)


@pytest.mark.parametrize("kind", KINDS)
def test_neural_fleet_philox_matches_supplied_split_and_permutation(kind):
    """A Philox fleet equals a supplied fleet fed its draws(period); those draws are the ODE fleet's; splitting the
    experiments by experiment_offset and permuting a supplied fleet's experiments change nothing; a NaN state stays in
    its experiment; launches per period do not depend on E."""
    E, K, T, P = 37, 64, 35, 12
    s0 = _states(E, 7)
    a = _fleet(kind, E, K, T, noise="philox", seed=11)
    b = _fleet(kind, E, K, T, noise="supplied")
    o = _fleet(kind, E, K, T, noise="philox", seed=11, integrator="ODE")
    for f in (a, b, o):
        f.reset(s0)
    n_it = 1 if kind == "ra" else a.outer_its

    def draws_of(f, j):   # as run() takes them: [iterations, E, ...] per draw array
        d = f.draws(j)
        return d if kind == "gmm" else (d if kind == "cem" else d[None],)
    ds = [draws_of(a, j) for j in range(P)]
    for j in (0, 5):
        for x, y in zip(ds[j], draws_of(o, j)):
            assert torch.equal(x, y)
    cat = [torch.cat([d[i] for d in ds]).contiguous() for i in range(len(ds[0]))]
    ra_, rb = torch.zeros((P, E, 16), device="cuda"), torch.zeros((P, E, 16), device="cuda")
    Ja, Jb = torch.zeros((P, E, K), device="cuda"), torch.zeros((P, E, K), device="cuda")
    l0 = a.engine.launch_count()
    _run(kind, a, P, None, None, [None, None], ra_, Ja, None)
    launches = a.engine.launch_count() - l0
    _run(kind, b, P, None, None, cat, rb, Jb, None)
    assert torch.equal(ra_, rb) and torch.equal(Ja, Jb)
    # split by experiment_offset
    c1 = _fleet(kind, 20, K, T, noise="philox", seed=11)
    c2 = _fleet(kind, E - 20, K, T, noise="philox", seed=11, experiment_offset=20)
    c1.reset(s0[:20])
    c2.reset(s0[20:])
    r1, r2 = torch.zeros((P, 20, 16), device="cuda"), torch.zeros((P, E - 20, 16), device="cuda")
    _run(kind, c1, P, None, None, [None, None], r1, None, None)
    _run(kind, c2, P, None, None, [None, None], r2, None, None)
    assert torch.equal(torch.cat([r1, r2], dim=1), ra_)
    assert c1.engine.launch_count() == launches
    # permutation of a supplied fleet's experiments
    perm = np.random.default_rng(1).permutation(E)
    pc = [d.index_select(1, torch.from_numpy(perm).cuda()).contiguous() for d in cat]   # experiments are dimension 1
    pf = _fleet(kind, E, K, T, noise="supplied")
    pf.reset(s0[perm])
    rp = torch.zeros((P, E, 16), device="cuda")
    _run(kind, pf, P, None, None, pc, rp, None, None)
    assert torch.equal(rp, ra_[:, torch.from_numpy(perm).cuda()])
    # NaN isolation
    s_nan = s0.copy()
    s_nan[4, 1] = np.nan
    nf = _fleet(kind, E, K, T, noise="philox", seed=11)
    nf.reset(s_nan)
    rn = torch.zeros((P, E, 16), device="cuda")
    _run(kind, nf, P, None, None, [None, None], rn, None, None)
    keep = torch.ones(E, dtype=torch.bool, device="cuda")
    keep[4] = False
    assert torch.equal(rn[:, keep], ra_[:, keep])
    assert nf.nonfinite_costs() > 0
    # 3 launches per iteration (sample, network, selection / update) and the plant: n_it x 3 + 1 per period
    assert launches == P * (3 * n_it + 1), launches


def test_neural_fleet_records_write_the_reference_csv(tmp_path):
    from cartpolesimulation_b200.recording import save_fleet_recordings
    E, K, T, P = 3, 64, 35, 4
    fl = _fleet("ra", E, K, T, noise="philox")
    fl.reset(_states(E, 9))
    rec = torch.zeros((P, E, 16), device="cuda")
    fl.run(P, None, None, None, rec)
    r = rec.cpu().numpy()
    assert np.all(np.isfinite(r)) and np.all(np.abs(r[:, :, 9]) <= 1.0)
    paths = save_fleet_recordings(rec, str(tmp_path), optimizer_name="random-action-b200", run_for_ML_Pipeline=False)
    assert len(paths) == E
    with open(paths[1]) as f:
        rows = [row for row in f if not row.startswith("#")]
    assert len(rows) == P + 1 and rows[0].startswith("time,angle,")


def test_neural_planner_refusals():
    """Outside the supported scope the calls raise NotImplementedError (differential networks, the MAX_COST plugins,
    the tensor-core kernel, K above 8192); without a network the engine raises RuntimeError and the fleets and drop-ins
    NotImplementedError."""
    from cartpolesimulation_b200.core import Engine
    from cartpolesimulation_b200.fleet import CemFleet
    from tests.test_gpu_net_grad import _engine_spec
    from tests.netutil import net_spec_from_golden
    from tests.parity import load_golden
    zd, _ = load_golden("net_diff_GRU_6IN_32H1_32H2_5OUT_1")
    spd = net_spec_from_golden(zd)
    d = _engine_spec(spd)
    f = spd["diff"]
    d.update(differential=True, diff_p1=f["p1"], diff_p2=f["p2"], out_norm_a=f["on_a"], out_norm_b=f["on_b"],
             out_to_in=f["out_to_in"])
    eng = Engine(64, 10, integrator="neural", cost=GRADMIN, device=0)
    eng.net_load(d)
    bad = [eng] + [_engine(_spec("gru32"), 64, 10, c) for c in ("default", "quadratic_boundary")] + \
          [_engine(_spec("gru32"), 64, 10, net_kernel="tensor"), _engine(_spec("gru32"), 8193, 10)]
    for e in bad:
        with pytest.raises(NotImplementedError):
            e.cem_configure(8, 0.5, 0.01)
        with pytest.raises(NotImplementedError):
            e.cem_gmm_configure(8, 0.5, 0.01)
        with pytest.raises(NotImplementedError):
            e.plan_random_action(cuda(_state(0)), torch.zeros((e.K, 10), device="cuda"))
    with pytest.raises(NotImplementedError):
        _fleet("cem", 2, 8193, 10)
    with pytest.raises(NotImplementedError):
        _fleet("gmm", 2, 64, 10, cost="default")
    bare = Engine(64, 10, integrator="neural", cost=GRADMIN, device=0)
    with pytest.raises(RuntimeError):
        bare.cem_configure(8, 0.5, 0.01)
    with pytest.raises(NotImplementedError):
        CemFleet(4, integrator="neural")
    with pytest.raises(NotImplementedError):
        _fleet("ra", 2, 64, 10).set_plant_models()
