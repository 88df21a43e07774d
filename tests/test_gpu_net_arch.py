"""GPU parity of the neural predictor on every architecture of the catalogue in tests/netutil.py -- the specialisations of
net_kernel, net_grad_kernel and net_tc_kernel that the three shipped networks never reach: generic widths (HT = 0), 1, 3
and 4 layers, a first layer wider than 64 units, `angle` outputs, permuted / partial / extended input-output layouts,
tensor cores on non-shipped layouts, the widest networks the shared-memory checks admit, RPGD fleets and differential
networks at generic widths.  References: oracle/net_grad.py (float64, run on the GPU; pinned to the reference's torch
modules on the same catalogue by tests/test_oracle_net_arch.py) and the C oracle (oracle.net_rollout, mppi_step_net).
Bounds: about twice the errors measured on a B200 (recorded with tests.parity.record; profiles/parity_net_arch.json)."""
import numpy as np
import pytest

from tests.netutil import ARCHS, SHIPPED_IN, SHIPPED_OUT, ANGLE_IN, ANGLE_OUT, arch, arch_net
from tests.parity import record, traj_err, vec_err

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

GRADMIN, QBGRAD = "quadratic_boundary_grad_minimal", "quadratic_boundary_grad"
QB_OVER = {1.0: {"dd_linear_weight_up": 25.0, "ccrc_weight_up": 1.5},
           -1.0: {"dd_linear_weight_down": 25.0, "ccrc_weight_down": 1.5}}
# plain 2-layer GRUs of <= 64 units: the tensor-core kernel by default
TC_ARCHS = [k for k, (t, hsz, _, _) in ARCHS.items() if t == "GRU" and len(hsz) == 2 and max(hsz) <= 64]

# Bounds: about twice the largest error measured on a B200 (1000 W) over the cases of each test.  Trajectories are
# range-relative, the angle channel apart; J and G are relative to the largest |J| / |G|; controls and hidden states absolute.
TRAJ_BOUND, ANGLE_BOUND = 2e-6, 5e-7        # measured 9.2e-7 (angle_cos), 2.4e-7
DIFF_TRAJ_BOUND, DIFF_ANGLE_BOUND = 4e-6, 6e-6   # differential networks: measured 1.9e-6, 2.8e-6
H_BOUND = 6.5e-7                             # measured 3.1e-7 (differential GRU), else <= 2.4e-7
J_MPPI_BOUND, U_BOUND = 1.1e-6, 6e-8         # MPPI solves: J measured 5.3e-7, u and u_nom 3.0e-8
# plan_cost_grad: J measured 5.5e-6 (T = 1: the float32 cost of the initial state alone), G 3.4e-6.  Where the float32
# problem itself is ill-conditioned, the float32 restatement (oracle/net_grad.py run in float32) departs from the float64
# one by as much as the kernel does; the bound is then twice that spread (see _grad_case).
J_BOUND, G_BOUND = 1e-5, 7e-6


def _engine(spec, K, T, cost=None, net_kernel=None, te=1.0, h0=None, **kw):
    from cartpolesimulation_b200 import config as cfgmod
    from cartpolesimulation_b200.core import Engine
    eng = Engine(K, T, integrator="neural", cost=cost, device=0, net_kernel=net_kernel, **kw)
    eng.net_load(spec)
    if cost is not None:
        eng.set_variable_parameters(-0.02, te)
    if cost == QBGRAD:
        eng.set_cost_params(cfgmod.cost_vector(cost, _cost_cfg(cost, te)))
    if h0 is not None and eng.net_htot:
        eng.net_set_state(h0)
    return eng


def _cost_cfg(cost, te):
    if cost != QBGRAD:
        return None
    from oracle import oracle as O
    cfg = dict(O.DEFAULT_COST_CONFIG[cost])
    cfg.update(QB_OVER[te])
    return cfg


def _states(B, rng):
    ang = rng.uniform(-np.pi, np.pi, B)
    return np.stack([ang, rng.uniform(-3, 3, B), np.cos(ang), np.sin(ang), rng.uniform(-0.15, 0.15, B),
                     rng.uniform(-0.5, 0.5, B)], 1).astype(np.float32)


def _oracle_args(osp):
    from oracle import oracle as O
    return (osp["net_type"], osp["hsz"], O.pack_net_weights(osp["net_type"], osp["layers"], osp["out_layer"]),
            osp["in_idx"], osp["out_idx"], osp["norm_a"], osp["norm_b"], osp["denorm_A"], osp["denorm_B"])


def _check_traj(e, what, traj_bound=TRAJ_BOUND, angle_bound=ANGLE_BOUND):
    ea = e.pop("angle")
    assert ea < angle_bound and max(e.values()) < traj_bound, (what, ea, e)


# ---- rollouts ---------------------------------------------------------------------------------------------------
ROLLOUT_SIZES = [(1, 1), (17, 2), (3000, 37), (1, 37), (17, 1), (3000, 2)]


def _rollout_case(spec, osp, B, T, i, net_kernel):
    """One rollout against oracle/net_grad.predict (float64) and the final hidden state against the C oracle; shared h0
    and the time-major layouts on odd i, per-rollout h0 and rollout-major on even i."""
    from cartpolesimulation_b200 import _lib as L
    from oracle import net_grad as NG
    from oracle import oracle as O
    rng = np.random.default_rng(1000 * B + 10 * T + i)
    s0, Q = _states(B, rng), rng.uniform(-1, 1, (B, T)).astype(np.float32)
    Ht = sum(osp["hsz"])
    shared = i % 2 == 1
    h0 = rng.uniform(-0.5, 0.5, Ht if shared else (B, Ht)).astype(np.float32)
    eng = _engine(spec, B, T, net_kernel=net_kernel)
    dev = eng.device
    gru = osp["net_type"] == "GRU"
    Qd = torch.from_numpy(np.ascontiguousarray(Q.T) if shared else Q).to(dev)
    lay = L.TIME_MAJOR if shared else L.ROLLOUT_MAJOR
    traj, hf = eng.net_rollout(torch.from_numpy(s0).to(dev), Qd, q_layout=lay, traj_layout=lay,
                               h0=torch.from_numpy(h0).to(dev) if gru else None, want_h=gru)
    traj = traj.permute(2, 0, 1) if shared else traj
    ref = NG.predict(osp, s0, torch.from_numpy(Q).to(dev).double(), h0 if gru else None).cpu().numpy()
    e = traj_err(traj.cpu().numpy(), ref)
    eh = 0.0
    if gru:
        _, href = O.net_rollout(*_oracle_args(osp), s0, Q, h0=np.broadcast_to(h0, (B, Ht)).copy(), want_h=True)
        eh = float(np.abs(hf.cpu().numpy() - href).max())
    kern = eng.net_last_kernel()
    eng.close()
    return e, eh, kern


@pytest.mark.parametrize("name", list(ARCHS))
@pytest.mark.parametrize("kernel", ["fp32", "default"])
def test_arch_rollout_vs_oracle(name, kernel):
    spec, osp = arch(name)
    for i, (B, T) in enumerate(ROLLOUT_SIZES):
        e, eh, kern = _rollout_case(spec, osp, B, T, i, "fp32" if kernel == "fp32" else None)
        record("net_arch_rollout", f"{name}/{kernel}/B{B}_T{T}", **e, h=eh, kernel=kern)
        assert kern == ("tensor" if kernel == "default" and name in TC_ARCHS else "fp32"), kern
        _check_traj(e, (B, T))
        assert eh < H_BOUND, eh


# ---- MPPI solve -------------------------------------------------------------------------------------------------
def _mppi(spec, K, T, s, u_nom, eps, h, net_kernel):
    from cartpolesimulation_b200 import _lib as L
    eng = _engine(spec, K, T, GRADMIN, net_kernel=net_kernel, h0=h)
    eng.set_variable_parameters(0.0, 1.0)
    eng.set_u_nom(u_nom)
    J = torch.empty(K, device=eng.device)
    u = eng.mppi_step(torch.from_numpy(s).to(eng.device), torch.from_numpy(eps).to(eng.device), L.ROLLOUT_MAJOR, 0.1, None, J)
    torch.cuda.synchronize()
    out = dict(u=float(u.cpu()[0]), J=J.cpu().numpy(), u_nom=eng.get_u_nom(), h=eng.net_get_state() if eng.net_htot else None,
               kernel=eng.net_last_kernel(), nonfinite=eng.nonfinite_costs())
    eng.close()
    return out


def _mppi_inputs(osp, K, T, seed):
    from oracle import oracle as O
    rng = np.random.default_rng(seed)
    eps = rng.standard_normal((K, O.num_inducing(T, 10))).astype(np.float32)
    u_nom = rng.uniform(-0.3, 0.3, T).astype(np.float32)
    h = rng.uniform(-0.3, 0.3, sum(osp["hsz"])).astype(np.float32)
    a = np.pi - 0.4
    s = np.array([a, 0.5, np.cos(a), np.sin(a), 0.03, -0.1], np.float32)
    return s, u_nom, eps, h


def _mppi_vs_oracle(spec, osp, K, T, seed, net_kernel):
    from oracle import oracle as O
    s, u_nom, eps, h = _mppi_inputs(osp, K, T, seed)
    gru = osp["net_type"] == "GRU"
    ref = O.mppi_step_net(GRADMIN, *_oracle_args(osp), s, u_nom, eps, h0=h if gru else None, u_prev=0.1)
    got = _mppi(spec, K, T, s, u_nom, eps, h, net_kernel)
    assert got["nonfinite"] == 0
    err = dict(J=vec_err(got["J"], ref["J"]), u=abs(got["u"] - float(ref["u"])),
               u_nom=float(np.abs(got["u_nom"] - ref["u_nom"]).max()), h=0.0)
    if gru:   # the solve advanced the stored state by one step on (u, s)
        _, hf = O.net_rollout(*_oracle_args(osp), s, np.array([[ref["u"]]], np.float32), h0=h, want_h=True)
        err["h"] = float(np.abs(got["h"] - hf[0]).max())
    return err, got["kernel"]


@pytest.mark.parametrize("name", list(ARCHS))
@pytest.mark.parametrize("K", [500, 3000])
def test_arch_mppi_vs_oracle(name, K):
    spec, osp = arch(name)
    err, kern = _mppi_vs_oracle(spec, osp, K, 30, K, "fp32")
    record("net_arch_mppi", f"{name}/K{K}", **err, kernel=kern)
    assert kern == "fp32"
    assert err["J"] < J_MPPI_BOUND and err["u"] < U_BOUND and err["u_nom"] < U_BOUND and err["h"] < H_BOUND, err


# ---- cost and gradient of predict_and_cost ----------------------------------------------------------------------------
GRAD_SIZES = [(1, 1), (16, 35), (33, 2), (3000, 100), (16, 100), (33, 1), (1, 35), (3000, 2)]


def _grad_case(spec, osp, K, T, i):
    """plan_cost_grad against autograd through oracle/net_grad (float64 on the GPU); plan_cost's J bit-identical to
    plan_cost_grad's, its trajectory to net_rollout's on the FP32 kernel.  The plugin, target equilibrium, stored state and
    plan layout rotate with i."""
    from cartpolesimulation_b200 import _lib as L
    from oracle import net_grad as NG
    cost = (GRADMIN, QBGRAD)[i % 2]
    te = (1.0, -1.0)[(i // 2) % 2] if cost == QBGRAD else 1.0
    gru = osp["net_type"] == "GRU"
    rng = np.random.default_rng(7 * K + T + i)
    h0 = rng.uniform(-0.3, 0.3, sum(osp["hsz"])).astype(np.float32) if (gru and (i // 2) % 2 == 0) else None
    time_major = i % 3 == 1
    u_prev = -0.3 if cost == QBGRAD else 0.1
    a = rng.uniform(-np.pi, np.pi)
    s = np.array([a, rng.normal(0, 1.0), np.cos(a), np.sin(a), rng.uniform(-0.1, 0.1), rng.normal(0, 0.3)], np.float32)
    Q = np.clip(rng.normal(0, 0.5, (K, T)), -1, 1).astype(np.float32)
    eng = _engine(spec, K, T, cost, net_kernel="fp32", te=te, h0=h0)
    dev = eng.device
    sd = torch.from_numpy(s).to(dev)
    Qd = torch.from_numpy(np.ascontiguousarray(Q.T) if time_major else Q).to(dev)
    lay = L.TIME_MAJOR if time_major else L.ROLLOUT_MAJOR
    J, G = eng.plan_cost_grad(sd, Qd, lay, u_prev)
    Jp, traj = eng.plan_cost(sd, Qd, lay, u_prev, want_traj=True)
    assert torch.equal(J, Jp)
    traj_r, _ = eng.net_rollout(sd, Qd, q_layout=lay)
    # plan_cost takes the gradient's tile (16 plans per CTA where the gradient's buffers leave no room for 32), net_rollout
    # its own: the output layer's sum is split differently, so above 148 x 16 rollouts they may differ in rounding
    same = bool(torch.equal(traj, traj_r))
    assert same or K > 148 * 16
    e_fwd = max(traj_err(traj.cpu().numpy(), traj_r.cpu().numpy()).values())
    assert e_fwd < 1e-6
    G = G.cpu().numpy().T if time_major else G.cpu().numpy()
    ref = {}
    for dt in (torch.float64, torch.float32):
        Qt = torch.from_numpy(Q).to(dev).to(dt).requires_grad_(True)
        Jr = NG.plan_cost(osp, cost, s, Qt, u_prev, -0.02, te, _cost_cfg(cost, te), h0, dtype=dt)
        (Gr,) = torch.autograd.grad(Jr.sum(), Qt)
        ref[dt] = (Jr.detach().double().cpu().numpy(), Gr.double().cpu().numpy())
    (Jr, Gr), (J32, G32) = ref[torch.float64], ref[torch.float32]
    nonfinite = eng.nonfinite_costs()
    eng.close()
    return dict(J=vec_err(J.cpu().numpy(), Jr), G=vec_err(G, Gr), J_f32_oracle=vec_err(J32, Jr), G_f32_oracle=vec_err(G32, Gr),
                traj_same=same, cost=cost, te=te, h0=h0 is not None, time_major=time_major, nonfinite=nonfinite)


def _check_grad(r, what):
    """Against the bounds, or where the float32 restatement itself departs further (an ill-conditioned float32 problem:
    e.g. 100 steps of an untrained network whose trajectory amplifies rounding), against twice its spread."""
    assert r["nonfinite"] == 0
    assert r["J"] < max(J_BOUND, 2 * r["J_f32_oracle"]) and r["G"] < max(G_BOUND, 2 * r["G_f32_oracle"]), (what, r)


@pytest.mark.parametrize("name", list(ARCHS))
def test_arch_plan_cost_grad_vs_autograd(name):
    spec, osp = arch(name)
    for i, (K, T) in enumerate(GRAD_SIZES):
        r = _grad_case(spec, osp, K, T, i)
        record("net_arch_plan_cost_grad", f"{name}/K{K}_T{T}", **r)
        _check_grad(r, (K, T))


@pytest.mark.parametrize("name", ["g_mixed", "d_angle", "g_perm", "g_noin"])
@pytest.mark.parametrize("te", [1.0, -1.0])
def test_arch_quadratic_boundary_grad_both_layouts(name, te):
    """quadratic_boundary_grad with its linear and control-change weights on, at both target equilibria, non-zero stored
    state: both plan layouts give bit-identical J and G, which match autograd."""
    from cartpolesimulation_b200 import _lib as L
    from oracle import net_grad as NG
    spec, osp = arch(name)
    K, T = 16, 35
    rng = np.random.default_rng(30)
    h0 = rng.uniform(-0.3, 0.3, sum(osp["hsz"])).astype(np.float32) if osp["net_type"] == "GRU" else None
    a = 2.5
    s = np.array([a, 0.7, np.cos(a), np.sin(a), 0.05, 0.2], np.float32)
    Q = np.clip(rng.normal(0, 0.5, (K, T)), -1, 1).astype(np.float32)
    eng = _engine(spec, K, T, QBGRAD, te=te, h0=h0)
    sd = torch.from_numpy(s).cuda()
    J, G = eng.plan_cost_grad(sd, torch.from_numpy(Q).cuda(), L.ROLLOUT_MAJOR, 0.4)
    J2, G2 = eng.plan_cost_grad(sd, torch.from_numpy(np.ascontiguousarray(Q.T)).cuda(), L.TIME_MAJOR, 0.4)
    assert torch.equal(J, J2) and torch.equal(G, G2.t())
    Jr, Gr = NG.plan_cost_grad(osp, QBGRAD, s, Q.astype(np.float64), 0.4, -0.02, te, _cost_cfg(QBGRAD, te), h0)
    r = dict(J=vec_err(J.cpu().numpy(), Jr), G=vec_err(G.cpu().numpy(), Gr))
    record("net_arch_qb_grad", f"{name}/te{te:+.0f}", **r)
    assert r["J"] < J_BOUND and r["G"] < G_BOUND, r


# ---- tensor-core kernel on non-shipped layouts ----------------------------------------------------------------------
@pytest.mark.parametrize("name", TC_ARCHS)
@pytest.mark.parametrize("K", [500, 6000, 12000])   # 32 / 64 / 128 live rollouts per CTA
def test_arch_tc_mppi_matches_fp32_kernel(name, K):
    spec, osp = arch(name)
    T = 12
    s, u_nom, eps, h = _mppi_inputs(osp, K, T, K + 1)
    f = _mppi(spec, K, T, s, u_nom, eps, h, "fp32")
    t = _mppi(spec, K, T, s, u_nom, eps, h, None)
    assert t["kernel"] == "tensor" and f["kernel"] == "fp32" and t["nonfinite"] == 0
    err = dict(J=vec_err(t["J"], f["J"]), u=abs(t["u"] - f["u"]), u_nom=float(np.abs(t["u_nom"] - f["u_nom"]).max()),
               h=float(np.abs(t["h"] - f["h"]).max()))
    record("net_arch_tc_vs_fp32", f"{name}/K{K}", **err)
    assert err["J"] < J_MPPI_BOUND and err["u"] < U_BOUND and err["u_nom"] < U_BOUND and err["h"] < H_BOUND, err


# ---- the widest networks the shared-memory checks admit ------------------------------------------------------------------
def _gru2(H):
    return arch_net("GRU", (H, H), SHIPPED_IN, SHIPPED_OUT, seed=H)


def _grad_rejected(H):
    from cartpolesimulation_b200 import _lib as L
    spec, _ = _gru2(H)
    eng = _engine(spec, 16, 35, GRADMIN)
    s, Q = torch.zeros(6, device="cuda"), torch.zeros((16, 35), device="cuda")
    try:
        eng.plan_cost_grad(s, Q, L.ROLLOUT_MAJOR, 0.0)
        return False
    except NotImplementedError:
        J, _ = eng.plan_cost(s, Q, L.ROLLOUT_MAJOR, 0.0)   # the forward-only instantiation still fits
        assert torch.isfinite(J).all()
        return True
    finally:
        eng.close()


def test_grad_max_width_vs_autograd():
    """GRU 2 x H with H the widest the gradient accepts (found from 72 down): wider than 64 units, so layer 0 runs without
    the split under the gradient's largest shared-memory carve-up; one unit more is refused while plan_cost still works."""
    H = 72
    while _grad_rejected(H):
        H -= 1
    assert H > 64 and _grad_rejected(H + 1)
    spec, osp = _gru2(H)
    for i, (K, T) in enumerate([(16, 35), (3000, 20)]):
        r = _grad_case(spec, osp, K, T, i)
        record("net_arch_grad_max", f"2x{H}/K{K}_T{T}", **r)
        _check_grad(r, (H, K, T))


def _load_refused(H, T):
    from cartpolesimulation_b200.core import Engine
    spec, _ = _gru2(H)
    eng = Engine(16, T, integrator="neural", cost=GRADMIN, device=0)
    try:
        eng.net_load(spec)
        return False
    except NotImplementedError:
        return True
    finally:
        eng.close()


def test_load_max_width_vs_oracle():
    """GRU 2 x H with H the widest cps_net_load accepts at the horizon used (found from 80 down): rollout and MPPI solve
    against the oracles; one unit more is refused."""
    T = 37
    H = 80
    while _load_refused(H, T):
        H -= 1
    assert H > 64 and _load_refused(H + 1, T)
    spec, osp = _gru2(H)
    e, eh, kern = _rollout_case(spec, osp, 3000, T, 0, None)
    record("net_arch_load_max_rollout", f"2x{H}/B3000_T{T}", **e, h=eh, kernel=kern)
    _check_traj(e, H)
    assert eh < H_BOUND
    err, kern = _mppi_vs_oracle(spec, osp, 3000, T, 5, None)
    record("net_arch_load_max_mppi", f"2x{H}/K3000_T{T}", **err, kernel=kern)
    assert err["J"] < J_MPPI_BOUND and err["u"] < U_BOUND and err["u_nom"] < U_BOUND and err["h"] < H_BOUND, err


# ---- RPGD fleets (net_grad_kernel<R, 0, GRAD, FLEET = true>) -----------------------------------------------------------
@pytest.mark.parametrize("name", ["g_mixed", "d_angle"])
@pytest.mark.parametrize("K", [16, 40])   # 40: a partial tile
def test_arch_rpgd_fleet_is_bit_identical_to_the_single_experiment_kernels(name, K):
    from cartpolesimulation_b200.core import Engine
    from cartpolesimulation_b200.fleet import RpgdFleet
    from tests.test_gpu_fleet_rpgd_neural import cuda, random_states, targets
    E, P, T, P_IND = 3, 2, 35, 4
    spec, osp = arch(name)
    h0 = np.random.default_rng(4).uniform(-0.3, 0.3, sum(osp["hsz"])).astype(np.float32) if osp["net_type"] == "GRU" else None
    fl = RpgdFleet(E, num_rollouts=K, mpc_horizon=T, cost=GRADMIN, noise="supplied", period_interpolation_inducing_points=P_IND,
                   integrator="neural", network=spec)
    if h0 is not None:
        fl.engine.net_set_state(h0)
    keep, n_ind = fl.opt_keep_k, fl.n_ind
    rng = np.random.default_rng(21)
    fl.reset(random_states(E, 22), init_draws=cuda(rng.standard_normal((E, K, n_ind))))
    draws = cuda(rng.standard_normal((P, E, K - keep, n_ind)))
    tp, te = targets(P, E, 23, flip=0)
    eng = Engine(K, T, integrator="neural", cost=GRADMIN, interp_period=P_IND)
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


# ---- differential (D_*) networks at generic widths: forward only -----------------------------------------------------
DIFF_ARCHS = {"diff_g_mixed": ("GRU", (40, 24), SHIPPED_IN, ["D_" + o for o in SHIPPED_OUT]),
              "diff_d_3layer": ("Dense", (16, 24, 8), ANGLE_IN, ["D_" + o for o in ANGLE_OUT])}


@pytest.mark.parametrize("name", list(DIFF_ARCHS))
def test_arch_differential_rollout_vs_oracle(name):
    from cartpolesimulation_b200 import _lib as L
    from oracle import oracle as O
    t, hsz, i, o = DIFF_ARCHS[name]
    spec, osp = arch_net(t, hsz, i, o, seed=11, dt=0.02)
    assert spec["differential"]
    for B, T in [(17, 1), (17, 37), (3000, 37)]:
        rng = np.random.default_rng(B + T)
        s0, Q = _states(B, rng), rng.uniform(-1, 1, (B, T)).astype(np.float32)
        h0 = rng.uniform(-0.5, 0.5, (B, sum(hsz))).astype(np.float32)
        gru = t == "GRU"
        eng = _engine(spec, B, T)
        traj, hf = eng.net_rollout(torch.from_numpy(s0).cuda(), torch.from_numpy(Q).cuda(),
                                   h0=torch.from_numpy(h0).cuda() if gru else None, want_h=gru)
        with O.net_differential(osp["diff"]):
            ref, href = O.net_rollout(*_oracle_args(osp), s0, Q, h0=h0, want_h=True)
        e = traj_err(traj.cpu().numpy(), ref)
        eh = float(np.abs(hf.cpu().numpy() - href).max()) if gru else 0.0
        record("net_arch_differential", f"{name}/B{B}_T{T}", **e, h=eh)
        _check_traj(e, (B, T), DIFF_TRAJ_BOUND, DIFF_ANGLE_BOUND)
        assert eh < H_BOUND
        eng.close()
    # the gradient of differential networks is not implemented: an error, not a wrong answer
    eng = _engine(spec, 16, 10, GRADMIN)
    with pytest.raises(NotImplementedError):
        eng.plan_cost_grad(torch.zeros(6, device="cuda"), torch.zeros((16, 10), device="cuda"), L.ROLLOUT_MAJOR, 0.0)
