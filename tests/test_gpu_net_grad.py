"""GPU parity of predict_and_cost with the neural predictor (cps_plan_cost, cps_plan_cost_grad, cps_rpgd_grad_step with
CPS_PREDICTOR_NEURAL; net_grad_kernel) and of optimizer_rpgd_b200 on a neural PredictorWrapper, against torch autograd
through the float64 restatement oracle/net_grad.py (pinned to the reference's recordings by tests/test_oracle_net_grad.py).
Networks: the weights and normalisation of tests/golden/net_*.npz; stored hidden states: zero and h_after of
tests/golden/mppi_net_*.npz.  Bounds: about twice the errors measured on a B200 (recorded with tests.parity.record)."""
import numpy as np
import pytest

from tests.netutil import net_spec_from_golden
from tests.parity import close_except_few, load_golden, record

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

NETS = {"gru32": "net_GRU_6IN_32H1_32H2_5OUT_0", "gru64": "net_GRU_6IN_64H1_64H2_5OUT_0",
        "dense32": "net_Dense_6IN_32H1_32H2_5OUT_0"}
H_AFTER = {"gru32": "mppi_net_gru32_grad", "gru64": "mppi_net_gru64_gradmin"}   # non-zero stored states
GRADMIN, QBGRAD = "quadratic_boundary_grad_minimal", "quadratic_boundary_grad"
QB_OVER = {1.0: {"dd_linear_weight_up": 25.0, "ccrc_weight_up": 1.5},
           -1.0: {"dd_linear_weight_down": 25.0, "ccrc_weight_down": 1.5}}

# bounds of max |a - b| / max |b| (J: costs, G: gradient); measured on a B200 over every case below, T up to 300:
# J <= 1.7e-6, G <= 2.0e-6 (the ODE adjoint's bar is 5e-5)
J_BOUND = 3.5e-6
G_BOUND = 4e-6


def _spec(net):
    z, _ = load_golden(NETS[net])
    return net_spec_from_golden(z)


def _engine_spec(sp):
    from oracle import oracle as O
    d = dict(sp)
    d["weights"] = O.pack_net_weights(sp["net_type"], sp["layers"], sp["out_layer"])
    return d


def _h_after(net):
    if net not in H_AFTER:
        return None
    z, _ = load_golden(H_AFTER[net])
    return z["h_after"][0].astype(np.float32)


def _cost_cfg(cost, te):
    if cost != QBGRAD:
        return None
    from oracle import oracle as O
    cfg = dict(O.DEFAULT_COST_CONFIG[cost])
    cfg.update(QB_OVER[te])
    return cfg


def _engine(sp, K, T, cost=GRADMIN, tp=0.0, te=1.0, h0=None, net_kernel=None):
    from cartpolesimulation_b200 import config as cfgmod
    from cartpolesimulation_b200.core import Engine
    eng = Engine(K, T, integrator="neural", cost=cost, device=0, net_kernel=net_kernel)
    eng.net_load(_engine_spec(sp))
    eng.set_variable_parameters(tp, te)
    cfg = _cost_cfg(cost, te)
    if cfg is not None:
        eng.set_cost_params(cfgmod.cost_vector(cost, cfg))
    if h0 is not None:
        eng.net_set_state(h0)
    return eng


def _state(seed):
    rng = np.random.default_rng(seed)
    a = rng.uniform(-np.pi, np.pi)
    return np.array([a, rng.normal(0, 1.0), np.cos(a), np.sin(a), rng.uniform(-0.1, 0.1), rng.normal(0, 0.3)], np.float32)


def _plans(K, T, seed):
    return np.clip(np.random.default_rng(seed).normal(0, 0.5, (K, T)), -1, 1).astype(np.float32)


def _rel(a, b):
    return float(np.abs(np.asarray(a, np.float64) - b).max() / max(np.abs(b).max(), 1e-12))


@pytest.mark.parametrize("net", list(NETS))
@pytest.mark.parametrize("cost", [GRADMIN, QBGRAD])
def test_plan_cost_neural(net, cost):
    """J against the oracle; the trajectory bit-identical to cps_net_rollout on a handle forced to the FP32 kernel (the
    forward is net_kernel's device code)."""
    from cartpolesimulation_b200 import _lib as L
    from oracle import net_grad as NG
    sp = _spec(net)
    K, T, h0 = 96, 50, _h_after(net)
    s, Q = _state(1), _plans(K, T, 2)
    eng = _engine(sp, K, T, cost, 0.03, 1.0, h0, net_kernel="fp32")
    sd, Qd = torch.from_numpy(s).cuda(), torch.from_numpy(Q).cuda()
    J, traj = eng.plan_cost(sd, Qd, L.ROLLOUT_MAJOR, -0.2, want_traj=True)
    traj_r, _ = eng.net_rollout(sd, Qd)
    assert torch.equal(traj, traj_r)
    Jr = NG.plan_cost(sp, cost, s, torch.from_numpy(Q.astype(np.float64)), -0.2, 0.03, 1.0, _cost_cfg(cost, 1.0), h0).numpy()
    eJ = _rel(J.cpu().numpy(), Jr)
    record("net_plan_cost_vs_oracle", f"{net}/{cost}", J=eJ)
    assert eJ < J_BOUND
    J2, traj2 = eng.plan_cost(sd, Qd.t().contiguous(), L.TIME_MAJOR, -0.2, want_traj=True, traj_layout=L.TIME_MAJOR)
    assert torch.equal(J2, J) and torch.equal(traj2.permute(2, 0, 1), traj)


SIZES = [(1, 1), (16, 35), (33, 7), (2000, 50), (5000, 20), (4, 300)]


@pytest.mark.parametrize("net", list(NETS))
@pytest.mark.parametrize("K,T", SIZES)
def test_plan_cost_grad_neural_vs_autograd(net, K, T):
    """cps_plan_cost_grad against torch autograd; the plugin, the stored state and the layout rotate over the sizes so that
    every network meets every combination."""
    from cartpolesimulation_b200 import _lib as L
    from oracle import net_grad as NG
    i = SIZES.index((K, T))
    cost = (GRADMIN, QBGRAD)[i % 2]
    te = (1.0, -1.0)[(i // 2) % 2] if cost == QBGRAD else 1.0
    h0 = _h_after(net) if (i // 2) % 2 == 0 else None
    time_major = (i % 3) == 1
    u_prev = -0.3 if cost == QBGRAD else 0.0
    sp = _spec(net)
    s, Q = _state(10 + i), _plans(K, T, 20 + i)
    eng = _engine(sp, K, T, cost, -0.02, te, h0)
    Qd = torch.from_numpy(np.ascontiguousarray(Q.T) if time_major else Q).cuda()
    J, G = eng.plan_cost_grad(torch.from_numpy(s).cuda(), Qd, L.TIME_MAJOR if time_major else L.ROLLOUT_MAJOR, u_prev)
    G = G.cpu().numpy().T if time_major else G.cpu().numpy()
    Jr, Gr = NG.plan_cost_grad(sp, cost, s, Q.astype(np.float64), u_prev, -0.02, te, _cost_cfg(cost, te), h0)
    eJ, eG = _rel(J.cpu().numpy(), Jr), _rel(G, Gr)
    record("net_plan_cost_grad_vs_autograd", f"{net}/K{K}_T{T}", J=eJ, G=eG, cost=cost, te=te, h0=h0 is not None,
           time_major=time_major)
    assert eJ < J_BOUND
    assert eG < G_BOUND
    assert eng.nonfinite_costs() == 0


@pytest.mark.parametrize("net", list(NETS))
@pytest.mark.parametrize("te", [1.0, -1.0])
@pytest.mark.parametrize("stored", [False, True])
def test_plan_cost_grad_quadratic_boundary_grad(net, te, stored):
    """quadratic_boundary_grad at both target equilibria with its linear-distance and control-change weights switched on,
    u_prev != 0, both plan layouts, at the shipped RPGD size."""
    from cartpolesimulation_b200 import _lib as L
    from oracle import net_grad as NG
    sp = _spec(net)
    K, T = 16, 35
    h0 = _h_after(net) if stored else None
    s, Q = _state(30), _plans(K, T, 31)
    eng = _engine(sp, K, T, QBGRAD, 0.05, te, h0)
    Jr, Gr = NG.plan_cost_grad(sp, QBGRAD, s, Q.astype(np.float64), 0.4, 0.05, te, _cost_cfg(QBGRAD, te), h0)
    sd = torch.from_numpy(s).cuda()
    J, G = eng.plan_cost_grad(sd, torch.from_numpy(Q).cuda(), L.ROLLOUT_MAJOR, 0.4)
    J2, G2 = eng.plan_cost_grad(sd, torch.from_numpy(np.ascontiguousarray(Q.T)).cuda(), L.TIME_MAJOR, 0.4)
    assert torch.equal(J, J2) and torch.equal(G, G2.t())
    eJ, eG = _rel(J.cpu().numpy(), Jr), _rel(G.cpu().numpy(), Gr)
    record("net_plan_cost_grad_qb_grad", f"{net}/te{te:+.0f}/stored{int(stored)}", J=eJ, G=eG)
    assert eJ < J_BOUND and eG < G_BOUND


@pytest.mark.parametrize("net", list(NETS))
@pytest.mark.parametrize("K", [16, 3000])
def test_gradient_and_plan_cost_share_J_and_leave_the_state(net, K):
    """J of cps_plan_cost_grad is bit-identical to cps_plan_cost's (one code path); neither call, nor an RPGD step, writes
    the stored hidden state."""
    from cartpolesimulation_b200 import _lib as L
    sp = _spec(net)
    T = 20
    eng = _engine(sp, K, T, GRADMIN, 0.0, 1.0, _h_after(net))
    h_before = eng.net_get_state().copy()
    sd, Qd = torch.from_numpy(_state(5)).cuda(), torch.from_numpy(_plans(K, T, 6)).cuda()
    Jp, _ = eng.plan_cost(sd, Qd, L.ROLLOUT_MAJOR, 0.0)
    Jg, _ = eng.plan_cost_grad(sd, Qd, L.ROLLOUT_MAJOR, 0.0)
    assert torch.equal(Jp, Jg)
    eng.rpgd_reset()
    eng.rpgd_grad_step(sd, Qd, 0.0)
    assert np.array_equal(eng.net_get_state(), h_before)


def test_rpgd_grad_step_neural_is_clip_adam_clip():
    """grad_step (optimizer_rpgd_tf.py:166-180) with the neural predictor: three steps against a numpy clip_by_norm -> Adam
    -> clip fed with the autograd gradients."""
    from oracle import net_grad as NG
    sp = _spec("gru32")
    K, T = 64, 20
    s, Q0 = _state(40), _plans(K, T, 41)
    h0 = _h_after("gru32")
    eng = _engine(sp, K, T, GRADMIN, 0.0, 1.0, h0)
    eng.rpgd_reset()
    lr, b1, b2, eps, clip = 0.05, 0.9, 0.999, 1e-8, 5.0
    Q, sd = torch.from_numpy(Q0.copy()).cuda(), torch.from_numpy(s).cuda()
    Qr = Q0.astype(np.float64)
    mm, vv = np.zeros_like(Qr), np.zeros_like(Qr)
    for it in range(1, 4):
        Jd = torch.empty(K, device="cuda")
        eng.rpgd_grad_step(sd, Q, 0.0, lr, b1, b2, eps, clip, J_out=Jd)
        Jr, G = NG.plan_cost_grad(sp, GRADMIN, s, Qr, 0.0, h0=h0)
        G = G * clip / np.maximum(np.sqrt((G ** 2).sum(axis=1, keepdims=True)), clip)
        mm = b1 * mm + (1 - b1) * G
        vv = b2 * vv + (1 - b2) * G * G
        Qr = np.clip(Qr - lr * np.sqrt(1 - b2 ** it) / (1 - b1 ** it) * mm / (np.sqrt(vv) + eps), -1.0, 1.0)
        eQ, eJ = float(np.abs(Q.cpu().numpy() - Qr).max()), _rel(Jd.cpu().numpy(), Jr)
        record("net_rpgd_grad_step", f"it{it}", Q=eQ, J=eJ)
        assert eQ < 9e-6 and eJ < J_BOUND   # measured Q <= 4.5e-6
    m_dev, _, iters = eng.rpgd_adam_state()
    assert iters == 3
    np.testing.assert_allclose(m_dev.cpu().numpy(), mm, rtol=0, atol=1e-4 * np.abs(mm).max())


class _Draws:
    def __init__(self, draws):
        self.draws, self.i = list(draws), 0

    def normal(self, shape, mean=0.0, stddev=1.0, dtype=None):
        d = self.draws[self.i]
        self.i += 1
        assert list(d.shape) == list(shape)
        return d * stddev + mean


def test_optimizer_rpgd_b200_neural_predictor_wrapper(tmp_path, monkeypatch):
    """optimizer_rpgd_b200 on a PredictorWrapper configured with a GRU 2 x 32 model directory, at the shipped size: four
    solves (the first and the fourth resample) against oracle.rpgd_step driven by the autograd gradient; each solve starts
    from the oracle's state.  The optimizer's stored hidden state stays zero (step() does not advance it)."""
    import cartpolesimulation_b200 as cps
    from cartpolesimulation_b200.optimizer_forward_b200 import optimizer_rpgd_b200
    from oracle import net_grad as NG
    from oracle import oracle as O
    from tests.netutil import write_model_dir
    z, _ = load_golden(NETS["gru32"])
    sp = net_spec_from_golden(z)
    K, T, outer, resamp, keep_ratio, p = 16, 35, 4, 3, 0.75, 4
    keep = int(K * keep_ratio)
    n_ind = O.num_inducing(T, p)
    rng = np.random.default_rng(50)
    draws = [rng.normal(0, 1, (K, n_ind, 1)).astype(np.float32)] + \
            [rng.normal(0, 1, (K - keep, n_ind, 1)).astype(np.float32) for _ in range(2)]
    vp = cps.VariableParameters(target_position=0.02, target_equilibrium=1.0, L=0.395, m_pole=0.087)
    cost, predictor = cps.CostFunctionWrapper(), cps.PredictorWrapper()
    predictor.configure(batch_size=K, horizon=T, dt=0.02, variable_parameters=vp,
                        predictor_specification=write_model_dir(str(tmp_path), z))
    cost.configure(batch_size=K, horizon=T, variable_parameters=vp, environment_name="CartPole", computation_library=None,
                   cost_function_specification=GRADMIN)
    opt = optimizer_rpgd_b200(predictor=predictor, cost_function=cost,
                              control_limits=(np.array([-1.0], np.float32), np.array([1.0], np.float32)), seed=1,
                              mpc_horizon=T, num_rollouts=K, outer_its=outer, resamp_per=resamp, opt_keep_k_ratio=keep_ratio,
                              period_interpolation_inducing_points=p, optimizer_logging=True)
    opt.configure(num_states=6, num_control_inputs=1, default_configure=False, dt=0.02, predictor_specification="neural")
    assert opt.predictor_type == "neural"
    opt.rng = _Draws([torch.from_numpy(d) for d in draws])
    opt.optimizer_reset()
    W = opt._W.cpu().numpy()
    np.testing.assert_allclose(opt.Q_tf.cpu().numpy(), np.clip(draws[0][:, :, 0] * 0.5, -1, 1) @ W, rtol=0, atol=1e-6)
    monkeypatch.setattr(O, "plan_cost_grad", lambda cost_name, s, Q, u_prev, **kw: NG.plan_cost_grad(sp, cost_name, s, Q, u_prev, **kw))
    Q, (m, v), it = opt.Q_tf.cpu().numpy().astype(np.float64), (np.zeros((K, T)), np.zeros((K, T))), 0
    for i in range(4):
        s = _state(60 + i)
        u_prev = float(np.asarray(opt.u).reshape(-1)[0])
        ref = O.rpgd_step(GRADMIN, s, Q, m, v, it, i, u_prev, resamp_draw=draws[1 + (i // resamp)][:, :, 0] if i % resamp == 0 else None,
                          outer_its=outer, resamp_per=resamp, opt_keep_k=keep, period=p, target_position=0.02)
        u = opt.step(s.copy())
        Q_opt = opt.logging_values["Q_logged"][:, :, 0]
        eQ, eu = float(np.abs(Q_opt - ref["Q_opt"]).max()), abs(float(u) - ref["u"])
        record("optimizer_rpgd_neural", f"solve{i}", Q=eQ, u=eu)
        assert close_except_few(Q_opt, ref["Q_opt"], 1.6e-5), eQ   # measured Q <= 8.1e-6, u <= 1.1e-6
        assert eu < 2.2e-6
        assert close_except_few(opt.Q_tf.cpu().numpy(), ref["Q_next"], 1.6e-5)
        mm, vv, iters = opt.engine.rpgd_adam_state()
        assert iters == ref["iterations"]
        np.testing.assert_allclose(mm.cpu().numpy(), ref["m"], rtol=0, atol=2e-4 * max(1.0, np.abs(ref["m"]).max()))
        np.testing.assert_allclose(vv.cpu().numpy(), ref["v"], rtol=0, atol=2e-4 * max(1.0, np.abs(ref["v"]).max()))
        assert not np.any(opt.engine.net_get_state())
        # the next solve starts from the oracle's state
        Q, m, v, it = ref["Q_next"], ref["m"], ref["v"], ref["iterations"]
        opt.Q_tf.copy_(torch.from_numpy(Q.astype(np.float32)).cuda())
        mm.copy_(torch.from_numpy(m.astype(np.float32)).cuda())
        vv.copy_(torch.from_numpy(v.astype(np.float32)).cuda())
        opt.u = np.array(ref["u"], dtype=np.float32)


def test_neural_gradient_rejections():
    """Each configuration outside the scope raises NotImplementedError; a neural engine without a network raises what
    net_rollout raises there; the forward-only planners CEM and random action still refuse the neural predictor."""
    from cartpolesimulation_b200 import _lib as L
    from cartpolesimulation_b200.core import Engine
    from cartpolesimulation_b200.optimizer_forward_b200 import optimizer_cem_b200, optimizer_random_action_b200
    K, T = 8, 5
    s, Q = torch.from_numpy(_state(0)).cuda(), torch.from_numpy(_plans(K, T, 0)).cuda()

    def both_raise(eng, exc):
        with pytest.raises(exc):
            eng.plan_cost(s, Q, L.ROLLOUT_MAJOR, 0.0)
        with pytest.raises(exc):
            eng.plan_cost_grad(s, Q, L.ROLLOUT_MAJOR, 0.0)
        with pytest.raises(exc):
            eng.rpgd_grad_step(s, Q.clone(), 0.0)

    # differential (D_*) network
    zd, _ = load_golden("net_diff_GRU_6IN_32H1_32H2_5OUT_1")
    spd = net_spec_from_golden(zd)
    d = _engine_spec(spd)
    f = spd["diff"]
    d.update(differential=True, diff_p1=f["p1"], diff_p2=f["p2"], out_norm_a=f["on_a"], out_norm_b=f["on_b"],
             out_to_in=f["out_to_in"])
    eng = Engine(K, T, integrator="neural", cost=GRADMIN, device=0)
    eng.net_load(d)
    both_raise(eng, NotImplementedError)
    # cost plugins other than the two gradient ones
    for cost in ("default", "quadratic_boundary"):
        both_raise(_engine(_spec("gru32"), K, T, cost), NotImplementedError)
    # the tensor-core flag
    both_raise(_engine(_spec("gru64"), K, T, net_kernel="tensor"), NotImplementedError)
    # a network that loads but whose image with the gradient's buffers exceeds 227 KB of shared memory (GRU 2 x 72)
    sp = dict(_spec("gru32"))
    rng = np.random.default_rng(0)
    H, n_in = 72, len(sp["in_idx"]) + 1
    sp["hsz"] = [H, H]
    sp["layers"] = [tuple(rng.normal(0, 0.1, shp).astype(np.float32) for shp in ((3 * H, i), (3 * H, H), (3 * H,), (3 * H,)))
                    for i in (n_in, H)]
    sp["out_layer"] = (rng.normal(0, 0.1, (len(sp["out_idx"]), H)).astype(np.float32),
                       np.zeros(len(sp["out_idx"]), np.float32))
    eng = _engine(sp, K, T)
    J, _ = eng.plan_cost(s, Q, L.ROLLOUT_MAJOR, 0.0)   # the forward-only instantiation fits
    assert torch.isfinite(J).all()
    with pytest.raises(NotImplementedError):
        eng.plan_cost_grad(s, Q, L.ROLLOUT_MAJOR, 0.0)
    # no network loaded: what net_rollout raises
    eng = Engine(K, T, integrator="neural", cost=GRADMIN, device=0)
    with pytest.raises(RuntimeError):
        eng.net_rollout(s, Q)
    both_raise(eng, RuntimeError)
    # CEM and random action keep their gate
    for cls in (optimizer_cem_b200, optimizer_random_action_b200):
        opt = cls(predictor="neural", cost_function=GRADMIN,
                  control_limits=(np.array([-1.0], np.float32), np.array([1.0], np.float32)), num_rollouts=K, mpc_horizon=T)
        with pytest.raises(NotImplementedError):
            opt.configure(num_states=6, num_control_inputs=1, dt=0.02)
