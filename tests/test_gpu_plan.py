"""GPU parity of the forward-only planners (SURVEY 8f row f3): plan_kernel through cps_plan_cost /
cps_plan_random_action / cps_cem_step and the optimizer_random_action_b200 / optimizer_cem_b200 mirrors, against the
CPU oracle and the recordings of the reference's optimizer_random_action_tf / optimizer_cem_tf (tests/golden/plan_*)."""
import numpy as np
import pytest

from tests.parity import load_golden, traj_err, vec_err

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

COSTS = ["default", "quadratic_boundary", "quadratic_boundary_grad_minimal", "quadratic_boundary_grad"]
RA = ["plan_ra_ode_gradmin", "plan_ra_v0_qb", "plan_ra_ode_default"]
CEM = ["plan_cem_ode_gradmin", "plan_cem_v0_gradmin", "plan_cem_ode_qb", "plan_cem_ode_K1024"]
SHIFTED = ("default", "quadratic_boundary")  # MAX_COST plugins: order below the 6e9 shift is noise (DESIGN.md 6.3)


def _engine(K, T, integ, cost, tp=0.0, te=1.0):
    from cartpolesimulation_b200.core import Engine
    eng = Engine(K, T, integrator=integ, cost=cost, device=0)
    eng.set_variable_parameters(tp, te)
    return eng


def _hanging():
    a = np.pi - 1e-3
    return np.array([a, 0.0, np.cos(a), np.sin(a), 0.0, 0.0], dtype=np.float32)


@pytest.mark.parametrize("integ", ["ODE", "ODE_v0"])
@pytest.mark.parametrize("cost", COSTS)
def test_plan_cost_matches_oracle(integ, cost):
    from cartpolesimulation_b200 import _lib as L
    from oracle import oracle as O
    rng = np.random.default_rng(3)
    K, T = 333, 35
    Q = np.clip(rng.normal(0, 0.5, (K, T)), -1, 1).astype(np.float32)
    s = _hanging()
    eng = _engine(K, T, integ, cost, 0.03, 1.0)
    J_ref, traj_ref = O.plan_cost(integ, cost, s, Q, 0.2, target_position=0.03, target_equilibrium=1.0, want_traj=True)
    sd = torch.from_numpy(s).cuda()
    J, traj = eng.plan_cost(sd, torch.from_numpy(Q).cuda(), L.ROLLOUT_MAJOR, 0.2, want_traj=True)
    assert max(traj_err(traj.cpu().numpy(), traj_ref).values()) < 1e-5
    tol = 1e-6 if cost in SHIFTED else 3e-5
    assert vec_err(J.cpu().numpy(), J_ref) < tol
    # time-major plans and trajectories give the same bits
    J2, traj2 = eng.plan_cost(sd, torch.from_numpy(np.ascontiguousarray(Q.T)).cuda(), L.TIME_MAJOR, 0.2, want_traj=True,
                              traj_layout=L.TIME_MAJOR)
    assert torch.equal(J, J2)
    assert torch.equal(traj2.permute(2, 0, 1).contiguous(), traj)
    # any batch size and horizon up to the caller (the Brunton test evaluates test_len plans of its own horizon)
    J3, _ = eng.plan_cost(sd, torch.from_numpy(Q[:17, :9].copy()).cuda(), L.ROLLOUT_MAJOR, 0.2)
    J3_ref = O.plan_cost(integ, cost, s, Q[:17, :9], 0.2, target_position=0.03, target_equilibrium=1.0)
    assert vec_err(J3.cpu().numpy(), J3_ref) < tol


def test_plan_cost_is_the_two_call_path_fused():
    """predict_core followed by get_trajectory_cost (cps_rollout + cps_trajectory_cost) gives the same costs."""
    from cartpolesimulation_b200 import _lib as L
    rng = np.random.default_rng(4)
    K, T = 2000, 50
    Q = torch.from_numpy(rng.uniform(-1, 1, (K, T)).astype(np.float32)).cuda()
    eng = _engine(K, T, "ODE", "quadratic_boundary_grad_minimal")
    s = torch.from_numpy(_hanging()).cuda()
    J, _ = eng.plan_cost(s, Q, L.ROLLOUT_MAJOR, 0.1)
    traj, _ = eng.rollout(s, Q)
    J2 = eng.trajectory_cost(traj, Q, 0.1)
    assert vec_err(J.cpu().numpy(), J2.cpu().numpy()) < 2e-6


@pytest.mark.parametrize("name", RA)
def test_random_action_matches_reference(name):
    from cartpolesimulation_b200 import _lib as L
    z, m = load_golden(name)
    K, T = m["K"], m["T"]
    eng = _engine(K, T, m["predictor"], m["cost"], m["target_position"], m["target_equilibrium"])
    J = torch.empty(K, device="cuda")
    best = torch.zeros(1, dtype=torch.int32, device="cuda")
    for i in range(m["steps"]):
        Q = torch.from_numpy(z["Q"][i].copy()).cuda()
        u = eng.plan_random_action(torch.from_numpy(z["s"][i].copy()).cuda(), Q, L.ROLLOUT_MAJOR, float(z["u_prev"][i]),
                                   J_out=J, best_out=best)
        Jh = J.cpu().numpy()
        assert vec_err(Jh, z["J"][i]) < (1e-6 if m["cost"] in SHIFTED else 3e-5)
        # the selection itself: exactly the arg-min of the costs the kernel computed, lowest index first
        b = int(best.cpu()[0])
        assert b == int(np.argsort(Jh, kind="stable")[0])
        assert float(u.cpu()[0]) == float(z["Q"][i][b, 0])
        if m["cost"] not in SHIFTED:
            assert float(u.cpu()[0]) == float(z["u"][i])
        uh = eng.plan_random_action_host(z["s"][i], Q, L.ROLLOUT_MAJOR, float(z["u_prev"][i]))
        assert uh == float(u.cpu()[0])


def test_random_action_ties_go_to_the_lowest_index():
    from cartpolesimulation_b200 import _lib as L
    rng = np.random.default_rng(5)
    K, T = 512, 20
    Q = rng.uniform(-1, 1, (K, T)).astype(np.float32)
    Q[256:] = Q[:256]   # every plan twice: each cost occurs at k and k + 256
    eng = _engine(K, T, "ODE", "quadratic_boundary_grad_minimal")
    best = torch.zeros(1, dtype=torch.int32, device="cuda")
    J = torch.empty(K, device="cuda")
    eng.plan_random_action(torch.from_numpy(_hanging()).cuda(), torch.from_numpy(Q).cuda(), L.ROLLOUT_MAJOR, 0.0, J_out=J,
                           best_out=best)
    Jh = J.cpu().numpy()
    assert np.array_equal(Jh[:256], Jh[256:])
    assert int(best.cpu()[0]) == int(np.argmin(Jh[:256]))


def _cem_reference_update(Q, J, best_k):
    el = np.argsort(J, kind="stable")[:best_k]
    eq = Q[el].astype(np.float64)
    return el, eq.mean(0), eq.std(0)


@pytest.mark.parametrize("name", CEM)
def test_cem_matches_reference(name):
    from cartpolesimulation_b200 import _lib as L
    z, m = load_golden(name)
    K, T = m["K"], m["T"]
    eng = _engine(K, T, m["predictor"], m["cost"], m["target_position"], m["target_equilibrium"])
    eng.cem_configure(m["best_k"], m["initial_stdev"], m["stdev_min"])
    mu0, sd0 = eng.cem_get_distribution()
    assert np.array_equal(mu0, np.zeros(T, np.float32)) and np.array_equal(sd0, np.full(T, m["initial_stdev"], np.float32))
    Q = torch.empty((K, T), device="cuda")
    J = torch.empty(K, device="cuda")
    for i in range(m["steps"]):
        eps = torch.from_numpy(z["eps"][i].copy()).cuda()
        u = eng.cem_step(torch.from_numpy(z["s"][i].copy()).cuda(), eps, L.ROLLOUT_MAJOR, float(z["u_prev"][i]), Q_out=Q,
                         J_out=J)
        mu, sd = eng.cem_get_distribution()
        assert vec_err(J.cpu().numpy(), z["J"][i]) < (1e-6 if m["cost"] in SHIFTED else 3e-5)
        if m["cost"] in SHIFTED:
            eng.cem_set_distribution(z["mean"][i], z["stdev"][i])  # order below the shift is noise; restart from the reference
            continue
        np.testing.assert_allclose(Q.cpu().numpy(), z["Q"][i], rtol=0, atol=2e-6)
        np.testing.assert_allclose(mu, z["mean"][i], rtol=0, atol=3e-6)
        np.testing.assert_allclose(sd, z["stdev"][i], rtol=0, atol=3e-6)
        assert abs(float(u.cpu()[0]) - float(z["u"][i])) < 1e-4   # north_star's tolerance on the selected control
        assert mu[-1] == 0.0 and sd[-1] == np.float32(m["initial_stdev"]) and (sd >= np.float32(m["stdev_min"])).all()


def test_cem_time_major_and_host_entry_give_the_same_result():
    from cartpolesimulation_b200 import _lib as L
    z, m = load_golden("plan_cem_ode_gradmin")
    K, T = m["K"], m["T"]
    res = []
    for layout in (L.ROLLOUT_MAJOR, L.TIME_MAJOR, "host"):
        eng = _engine(K, T, m["predictor"], m["cost"])
        eng.cem_configure(m["best_k"], m["initial_stdev"], m["stdev_min"])
        e = z["eps"][0]
        if layout == L.TIME_MAJOR:
            e = np.ascontiguousarray(e.transpose(0, 2, 1))
        eps = torch.from_numpy(e.copy()).cuda()
        if layout == "host":
            u = eng.cem_step_host(z["s"][0], eps, L.ROLLOUT_MAJOR, 0.0)
        else:
            u = float(eng.cem_step(torch.from_numpy(z["s"][0].copy()).cuda(), eps, layout, 0.0).cpu()[0])
        res.append((u,) + eng.cem_get_distribution())
    for r in res[1:]:
        assert r[0] == res[0][0] and np.array_equal(r[1], res[0][1]) and np.array_equal(r[2], res[0][2])


@pytest.mark.parametrize("K,best_k", [(65536, 1000), (20000, 1), (4096, 4096), (777, 100)])
def test_cem_selection_at_scale(K, best_k):
    """One outer iteration at large K (every launch geometry): the elite statistics must equal those of a stable sort of
    the costs the kernel itself produced -- a size-independent property, no oracle rollouts needed."""
    from cartpolesimulation_b200 import _lib as L
    T = 30
    rng = np.random.default_rng(K)
    eng = _engine(K, T, "ODE", "quadratic_boundary_grad_minimal")
    eng.cem_configure(best_k, 0.5, 0.0)
    eps_h = rng.standard_normal((1, K, T)).astype(np.float32)
    eps_h[0, K // 2:] = eps_h[0, :K - K // 2]   # duplicated plans: ties straddle the elite boundary somewhere
    Q = torch.empty((K, T), device="cuda")
    J = torch.empty(K, device="cuda")
    u = eng.cem_step(torch.from_numpy(_hanging()).cuda(), torch.from_numpy(eps_h).cuda(), L.ROLLOUT_MAJOR, 0.0, Q_out=Q, J_out=J)
    Qh, Jh = Q.cpu().numpy(), J.cpu().numpy()
    assert np.array_equal(Qh, np.clip(np.float32(0.5) * eps_h[0], -1, 1))
    el, mean, std = _cem_reference_update(Qh, Jh, best_k)
    mu, sd = eng.cem_get_distribution()
    np.testing.assert_allclose(mu[:-1], mean[1:], rtol=0, atol=2e-6)
    np.testing.assert_allclose(sd[:-1], std[1:], rtol=0, atol=2e-6)
    assert float(u.cpu()[0]) == float(Qh[el[0], 0])


def test_planner_errors():
    from cartpolesimulation_b200 import _lib as L
    from cartpolesimulation_b200.core import Engine
    eng = _engine(64, 10, "ODE", "quadratic_boundary_grad_minimal")
    s = torch.from_numpy(_hanging()).cuda()
    with pytest.raises(RuntimeError):   # CPS_ERR_NOT_CONFIGURED
        eng.cem_step(s, torch.zeros((1, 64, 10), device="cuda"))
    with pytest.raises(ValueError):
        eng.cem_configure(65, 0.5, 0.01)   # best_k > K
    with pytest.raises(ValueError):
        eng.plan_random_action(s, torch.zeros((63, 10), device="cuda"))
    no_cost = Engine(64, 10, integrator="ODE", cost=None, device=0)
    with pytest.raises(RuntimeError):
        no_cost.plan_cost(s, torch.zeros((64, 10), device="cuda"))
    for flag in ("fast_div", "substep_sincos"):   # the planners' rotation substeps only: refused at configure, nothing launched
        gmm = Engine(64, 10, integrator="ODE", cost="quadratic_boundary_grad_minimal", device=0, **{flag: True})
        with pytest.raises(NotImplementedError):   # CPS_ERR_UNSUPPORTED
            gmm.cem_gmm_configure(8, 0.5, 0.01)
        assert gmm.launch_count() == 0


# ---- the optimizer mirrors ---------------------------------------------------------------------------------------------
class Injected:
    def __init__(self, draws):
        self.draws, self.i = list(draws), 0

    def _next(self, shape):
        d = self.draws[self.i]
        self.i += 1
        assert list(d.shape) == list(shape)
        return d

    def normal(self, shape, dtype=None):
        return self._next(shape)

    def uniform(self, shape, minval=None, maxval=None, dtype=None):
        return self._next(shape)


def _make(cls, m, logging=False, **params):
    import cartpolesimulation_b200 as cps
    vp = cps.VariableParameters(target_position=m["target_position"], target_equilibrium=m["target_equilibrium"],
                                L=0.395, m_pole=0.087)
    cost, predictor = cps.CostFunctionWrapper(), cps.PredictorWrapper()
    opt = cls(predictor=predictor, cost_function=cost,
              control_limits=(np.array([-1.0], np.float32), np.array([1.0], np.float32)), computation_library=None,
              seed=1, mpc_horizon=m["T"], num_rollouts=m["K"], optimizer_logging=logging,
              calculate_optimal_trajectory=False, **params)
    predictor.configure(batch_size=m["K"], horizon=m["T"], dt=0.02, variable_parameters=vp,
                        predictor_specification=m["predictor"])
    cost.configure(batch_size=m["K"], horizon=m["T"], variable_parameters=vp, environment_name="CartPole",
                   computation_library=None, cost_function_specification=m["cost"])
    opt.configure(num_states=6, num_control_inputs=1, dt=0.02, predictor_specification=m["predictor"])
    return opt, vp


@pytest.mark.parametrize("logging", [False, True])
def test_optimizer_cem_b200_step_sequence(logging):
    from cartpolesimulation_b200.optimizer_forward_b200 import optimizer_cem_b200
    z, m = load_golden("plan_cem_ode_gradmin")
    opt, _ = _make(optimizer_cem_b200, m, logging, cem_outer_it=m["iterations"], cem_initial_action_stdev=m["initial_stdev"],
                   cem_stdev_min=m["stdev_min"], cem_best_k=m["best_k"], warmup=False, warmup_iterations=250)
    opt.rng = Injected([torch.from_numpy(z["eps"][i, j][:, :, None].copy()) for i in range(m["steps"])
                        for j in range(m["iterations"])])
    for i in range(m["steps"]):
        u = opt.step(z["s"][i].copy())
        assert isinstance(u, np.ndarray) and u.dtype == np.float32 and u.shape == ()
        assert abs(float(u) - float(z["u"][i])) < 1e-4
        assert opt.dist_mue.shape == (1, m["T"], 1) and opt.stdev.shape == (1, m["T"], 1)
        np.testing.assert_allclose(opt.dist_mue.numpy().reshape(-1), z["mean"][i], rtol=0, atol=3e-6)
        np.testing.assert_allclose(opt.stdev.numpy().reshape(-1), z["stdev"][i], rtol=0, atol=3e-6)
        if logging:
            lv = opt.logging_values
            assert lv["Q_logged"].shape == (m["K"], m["T"], 1)
            assert lv["rollout_trajectories_logged"].shape == (m["K"], m["T"] + 1, 6)
            np.testing.assert_allclose(lv["Q_logged"][:, :, 0], z["Q"][i], rtol=0, atol=2e-6)
            assert vec_err(lv["J_logged"], z["J"][i]) < 3e-5
    assert opt.count == m["steps"] and opt.optimizer_name == "cem-b200"
    opt.optimizer_reset()
    assert opt.count == 0 and opt.u == 0.0
    np.testing.assert_array_equal(opt.stdev.numpy().reshape(-1), np.full(m["T"], m["initial_stdev"], np.float32))


def test_optimizer_cem_b200_own_rng_and_warmup():
    from cartpolesimulation_b200.optimizer_forward_b200 import optimizer_cem_b200
    z, m = load_golden("plan_cem_ode_gradmin")
    kw = dict(cem_outer_it=3, cem_initial_action_stdev=0.5, cem_stdev_min=0.01, cem_best_k=40)
    a, _ = _make(optimizer_cem_b200, m, **kw)
    b, _ = _make(optimizer_cem_b200, m, **kw)
    w, _ = _make(optimizer_cem_b200, m, warmup=True, warmup_iterations=12, **kw)
    s = z["s"][0]
    ua, ub = [float(a.step(s)) for _ in range(3)], [float(b.step(s)) for _ in range(3)]
    assert ua == ub and all(np.isfinite(ua)) and all(abs(v) <= 1.0 for v in ua)   # seeded, reproducible, clipped
    n0 = w.engine.launch_count()
    w.step(s)
    assert w.engine.launch_count() - n0 == 12   # the first solve runs warmup_iterations launches (:93)
    w.step(s)
    assert w.engine.launch_count() - n0 == 15


def test_optimizer_random_action_b200():
    from cartpolesimulation_b200.optimizer_forward_b200 import optimizer_random_action_b200
    z, m = load_golden("plan_ra_ode_gradmin")
    opt, vp = _make(optimizer_random_action_b200, m, logging=True)
    opt.rng = Injected([torch.from_numpy(q[:, :, None].copy()) for q in z["Q"]])
    for i in range(m["steps"]):
        u = opt.step(z["s"][i].copy())
        assert float(u) == float(z["u"][i])
        assert vec_err(opt.logging_values["J_logged"], z["J"][i]) < 3e-5
    assert opt.optimizer_name == "random-action-b200"
    own, _ = _make(optimizer_random_action_b200, m)
    us = [float(own.step(z["s"][0])) for _ in range(3)]
    assert all(-1.0 <= v <= 1.0 for v in us) and len(set(us)) > 1


@pytest.mark.parametrize("K", [200, 5000])
def test_cem_all_costs_equal(K):
    """Identical plans -> identical costs: the radix select has no varying bit, the elites are the first best_k plans,
    the elite spread is zero and the stdev floor applies."""
    from cartpolesimulation_b200 import _lib as L
    T, best_k = 25, 33
    eng = _engine(K, T, "ODE", "quadratic_boundary_grad_minimal")
    eng.cem_configure(best_k, 0.5, 0.02)
    J = torch.empty(K, device="cuda")
    best = None
    u = eng.cem_step(torch.from_numpy(_hanging()).cuda(), torch.zeros((2, K, T), device="cuda"), L.ROLLOUT_MAJOR, 0.0, J_out=J)
    Jh = J.cpu().numpy()
    assert (Jh == Jh[0]).all() and float(u.cpu()[0]) == 0.0
    mu, sd = eng.cem_get_distribution()
    assert (mu == 0.0).all()
    np.testing.assert_array_equal(sd, np.r_[np.full(T - 1, 0.02, np.float32), np.float32(0.5)])


def test_packed_planner_kernels_match_the_one_per_thread_kernels():
    """From 65536 time-major plans on, rollouts + costs run two plans per thread in packed FP32: every cost is
    bit-identical to the one-plan-per-thread kernel's (reached here through the rollout-major layout), for the plain
    evaluation and for a CEM solve (sampled plans, costs, distribution and control)."""
    from cartpolesimulation_b200 import _lib as L
    rng = np.random.default_rng(21)
    K, T = 65536, 40
    s = torch.from_numpy(_hanging()).cuda()
    for integ in ("ODE", "ODE_v0"):
        eng = _engine(K, T, integ, "quadratic_boundary", 0.02, 1.0)
        Q = torch.from_numpy(rng.uniform(-1, 1, (K, T)).astype(np.float32)).cuda()
        J_one, _ = eng.plan_cost(s, Q, L.ROLLOUT_MAJOR, 0.3)
        J_two, _ = eng.plan_cost(s, Q.t().contiguous(), L.TIME_MAJOR, 0.3)
        assert torch.equal(J_one, J_two)
    eps = rng.standard_normal((2, K, T)).astype(np.float32)
    res = []
    for layout in (L.ROLLOUT_MAJOR, L.TIME_MAJOR):
        eng = _engine(K, T, "ODE", "quadratic_boundary_grad_minimal")
        eng.cem_configure(500, 0.5, 0.01)
        e = eps if layout == L.ROLLOUT_MAJOR else np.ascontiguousarray(eps.transpose(0, 2, 1))
        Qo = torch.empty((K, T) if layout == L.ROLLOUT_MAJOR else (T, K), device="cuda")
        J = torch.empty(K, device="cuda")
        u = float(eng.cem_step(s, torch.from_numpy(e).cuda(), layout, 0.0, Q_out=Qo, J_out=J).cpu()[0])
        res.append((u, J.cpu().numpy(), (Qo if layout == L.ROLLOUT_MAJOR else Qo.t()).cpu().numpy()) + eng.cem_get_distribution())
    a, b = res
    assert a[0] == b[0] and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    np.testing.assert_array_equal(a[3], b[3])
    np.testing.assert_array_equal(a[4], b[4])


# ---- optimizer_cem_gmm_tf (cps_cem_gmm_*, optimizer_cem_gmm_b200) ---------------------------------------------------------
GMM = ["plan_gmm_ode_gradmin", "plan_gmm_v0_gradmin", "plan_gmm_ode_K512"]


@pytest.mark.parametrize("name", GMM)
def test_cem_gmm_matches_reference(name):
    from cartpolesimulation_b200 import _lib as L
    z, m = load_golden(name)
    K, T = m["K"], m["T"]
    eng = _engine(K, T, m["predictor"], m["cost"], m["target_position"], m["target_equilibrium"])
    eng.cem_gmm_configure(m["best_k"], m["initial_stdev"], m["stdev_min"])
    loc0, sc0, p0 = eng.cem_gmm_get_distribution()
    assert np.array_equal(loc0, np.zeros((2, T), np.float32)) and p0 == 0.5
    assert np.array_equal(sc0, np.full((2, T), m["initial_stdev"], np.float32))
    Q = torch.empty((K, T), device="cuda")
    J = torch.empty(K, device="cuda")
    for i in range(m["steps"]):
        eps = torch.from_numpy(z["eps"][i].copy()).cuda()        # [it, K, T, 2]: the reference's sample shape
        u01 = torch.from_numpy(z["u01"][i].copy()).cuda()
        u = eng.cem_gmm_step(torch.from_numpy(z["s"][i].copy()).cuda(), eps, u01, L.ROLLOUT_MAJOR, float(z["u_prev"][i]),
                             Q_out=Q, J_out=J)
        loc, sc, p1 = eng.cem_gmm_get_distribution()
        np.testing.assert_allclose(Q.cpu().numpy(), z["Q"][i], rtol=0, atol=2e-6)
        assert vec_err(J.cpu().numpy(), z["J"][i]) < 3e-5
        assert p1 == float(z["p1"][i])                           # same cluster sizes
        np.testing.assert_allclose(loc.T, z["loc"][i], rtol=0, atol=3e-6)
        np.testing.assert_allclose(sc.T, z["scale"][i], rtol=0, atol=3e-6)
        assert abs(float(u.cpu()[0]) - float(z["u"][i])) < 1e-4  # north_star's tolerance on the selected control
        assert (loc[:, -1] == loc[:, -2]).all() and (sc >= np.float32(m["stdev_min"])).all()


def test_cem_gmm_layouts_and_host_entry_give_the_same_result():
    from cartpolesimulation_b200 import _lib as L
    z, m = load_golden("plan_gmm_ode_gradmin")
    K, T = m["K"], m["T"]
    res = []
    for layout in (L.ROLLOUT_MAJOR, L.TIME_MAJOR, "host"):
        eng = _engine(K, T, m["predictor"], m["cost"])
        eng.cem_gmm_configure(m["best_k"], m["initial_stdev"], m["stdev_min"])
        e, w = z["eps"][0], z["u01"][0]
        if layout == L.TIME_MAJOR:
            e, w = np.ascontiguousarray(e.transpose(0, 3, 2, 1)), np.ascontiguousarray(w.transpose(0, 2, 1))
        eps, u01 = torch.from_numpy(e.copy()).cuda(), torch.from_numpy(w.copy()).cuda()
        if layout == "host":
            u = eng.cem_gmm_step_host(z["s"][0], eps, u01, L.ROLLOUT_MAJOR, 0.0)
        else:
            u = float(eng.cem_gmm_step(torch.from_numpy(z["s"][0].copy()).cuda(), eps, u01, layout, 0.0).cpu()[0])
        res.append((u,) + eng.cem_gmm_get_distribution())
    for r in res[1:]:
        assert r[0] == res[0][0] and np.array_equal(r[1], res[0][1]) and np.array_equal(r[2], res[0][2]) and r[3] == res[0][3]


@pytest.mark.parametrize("K,best_k", [(20000, 500), (3000, 2), (777, 777)])
def test_cem_gmm_vs_oracle_at_scale(K, best_k):
    """Selection, clustering and statistics over many plans against the numpy restatement (one iteration, T = 12)."""
    from cartpolesimulation_b200 import _lib as L
    from oracle import oracle as O
    T = 12
    rng = np.random.default_rng(K)
    eps = rng.standard_normal((1, K, T, 2)).astype(np.float32)
    u01 = rng.uniform(0, 1, (1, K, T)).astype(np.float32)
    s = _hanging()
    eng = _engine(K, T, "ODE", "quadratic_boundary_grad_minimal")
    eng.cem_gmm_configure(best_k, 0.5, 0.01)
    ref = O.cem_gmm_step("ODE", "quadratic_boundary_grad_minimal", s, eps, u01, np.zeros((T, 2), np.float32),
                         np.full((T, 2), 0.5, np.float32), 0.5, best_k, 0.01)
    J = torch.empty(K, device="cuda")
    u = eng.cem_gmm_step(torch.from_numpy(s).cuda(), torch.from_numpy(eps).cuda(), torch.from_numpy(u01).cuda(),
                         L.ROLLOUT_MAJOR, 0.0, J_out=J)
    loc, sc, p1 = eng.cem_gmm_get_distribution()
    # the elite set is decided by the cost order: compare on the GPU's own costs when a near-tie flips an elite
    Jg = J.cpu().numpy()
    if set(np.argsort(Jg, kind="stable")[:best_k]) == set(ref["elites"]):
        assert p1 == float(ref["p1"])
        np.testing.assert_allclose(loc.T, ref["loc"], rtol=0, atol=5e-6)
        np.testing.assert_allclose(sc.T, ref["scale"], rtol=0, atol=5e-6)
        assert abs(float(u.cpu()[0]) - float(ref["u"])) < 1e-6
    assert vec_err(Jg, ref["J"]) < 3e-5
    assert 0.0 < p1 < 1.0 and (sc >= np.float32(0.01)).all()


def test_optimizer_cem_gmm_b200_step_sequence():
    from cartpolesimulation_b200.optimizer_forward_b200 import optimizer_cem_gmm_b200
    z, m = load_golden("plan_gmm_ode_gradmin")
    opt, _ = _make(optimizer_cem_gmm_b200, m, True, cem_outer_it=m["iterations"], cem_initial_action_stdev=m["initial_stdev"],
                   cem_stdev_min=m["stdev_min"], cem_best_k=m["best_k"])
    draws = []
    for i in range(m["steps"]):
        for j in range(m["iterations"]):
            draws += [torch.from_numpy(z["eps"][i, j][:, :, None, :].copy()), torch.from_numpy(z["u01"][i, j][:, :, None].copy())]
    opt.rng = Injected(draws)
    for i in range(m["steps"]):
        u = opt.step(z["s"][i].copy())
        assert isinstance(u, np.ndarray) and u.dtype == np.float32 and u.shape == ()
        assert abs(float(u) - float(z["u"][i])) < 1e-4
        d = opt.sampling_dist
        assert d["loc"].shape == (m["T"], 1, 2) and d["scale"].shape == (m["T"], 1, 2)
        np.testing.assert_allclose(d["loc"].numpy().reshape(m["T"], 2), z["loc"][i], rtol=0, atol=3e-6)
        np.testing.assert_allclose(d["scale"].numpy().reshape(m["T"], 2), z["scale"][i], rtol=0, atol=3e-6)
        assert float(d["probs"][0]) == float(z["p1"][i])
        lv = opt.logging_values
        np.testing.assert_allclose(lv["Q_logged"][:, :, 0], z["Q"][i], rtol=0, atol=2e-6)
        assert vec_err(lv["J_logged"], z["J"][i]) < 3e-5
    assert opt.optimizer_name == "cem-gmm-b200"
    opt.optimizer_reset()
    assert float(opt.sampling_dist["probs"][0]) == 0.5
    own, _ = _make(optimizer_cem_gmm_b200, m, cem_outer_it=3, cem_best_k=40)
    own2, _ = _make(optimizer_cem_gmm_b200, m, cem_outer_it=3, cem_best_k=40)
    ua, ub = [float(own.step(z["s"][0])) for _ in range(3)], [float(own2.step(z["s"][0])) for _ in range(3)]
    assert ua == ub and all(abs(v) <= 1.0 for v in ua)   # seeded, reproducible, clipped
