"""MPPI fleets on the neural predictor (cps_fleet_* on a CPS_PREDICTOR_NEURAL handle, fleet.Fleet(integrator="neural",
network=...)): E closed-loop experiments whose controller solves with a GRU / Dense network, each with its own hidden state,
while the plant stays the CartPole ODE.  Against the oracle (oracle.mppi_step_net, oracle.net_rollout, oracle.plant_period),
against Engine.mppi_step per experiment (bit for bit), against its own Philox draws, a split over two fleets, a
permutation of the experiments, an ODE fleet's plant and optimizer_mppi_b200 on a neural PredictorWrapper.
Networks: the weights and normalisation of tests/golden/net_*.npz."""
import csv
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import oracle as O
from tests.netutil import net_spec_from_golden
from tests.parity import load_golden, record, shifted_cost_ok, vec_err

pytestmark = pytest.mark.gpu

GRADMIN, GRAD, QB = "quadratic_boundary_grad_minimal", "quadratic_boundary_grad", "quadratic_boundary"
ERR_INVALID, ERR_UNSUPPORTED, ERR_NOT_CONFIGURED = 1, 3, 4
NETS = {"gru32": "net_GRU_6IN_32H1_32H2_5OUT_0", "gru64": "net_GRU_6IN_64H1_64H2_5OUT_0",
        "dense32": "net_Dense_6IN_32H1_32H2_5OUT_0", "diff32": "net_diff_GRU_6IN_32H1_32H2_5OUT_1"}
RANGES = np.array([np.pi, 18.38, 1.0, 1.0, 0.198, 1.125], dtype=np.float64)  # the reference's normalisation ranges


def _spec(net):
    z, _ = load_golden(NETS[net])
    return net_spec_from_golden(z)


def engine_spec(sp):
    d = dict(sp)
    d["weights"] = O.pack_net_weights(sp["net_type"], sp["layers"], sp["out_layer"])
    if sp.get("diff") is not None:
        f = sp["diff"]
        d.update(differential=True, diff_p1=f["p1"], diff_p2=f["p2"], out_norm_a=f["on_a"], out_norm_b=f["on_b"],
                 out_to_in=f["out_to_in"])
    return d


def oracle_args(sp):
    return (sp["net_type"], sp["hsz"], O.pack_net_weights(sp["net_type"], sp["layers"], sp["out_layer"]), sp["in_idx"],
            sp["out_idx"], sp["norm_a"], sp["norm_b"], sp["denorm_A"], sp["denorm_B"])


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


def make(E, K, T, cost, net="gru32", noise="supplied", net_kernel=None, **kw):
    from cartpolesimulation_b200.fleet import Fleet
    return Fleet(E, K, T, cost=cost, noise=noise, integrator="neural", network=engine_spec(_spec(net)),
                 net_kernel=net_kernel, **kw)


def tc_rows(n_rows):
    """The tensor-core kernel's live rollouts per CTA for a launch of n_rows rollouts (cps_net_tc_rows)."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return 32 if n_rows <= 32 * sms else 64 if n_rows <= 64 * sms else 128


def run_periods(fl, P, tp, te, noise=None, h0=None, s0=None, seed=11):
    """reset, optional hidden states, P periods in one call; returns records [P, E, 16], costs and the final states
    (hidden states of a neural fleet included)."""
    fl.reset(random_states(fl.E, seed) if s0 is None else s0)
    if h0 is not None:
        fl.set_net_states(h0)
    rec = torch.zeros((P, fl.E, 16), device="cuda")
    J = torch.zeros((P, fl.E, fl.K), device="cuda")
    fl.run(P, cuda(tp), cuda(te), None if noise is None else cuda(noise), rec, J)
    s, u_nom, u_prev = fl.states(with_u_nom=True)
    out = dict(rec=rec.cpu().numpy(), J=J.cpu().numpy(), s=s, u_nom=u_nom, u_prev=u_prev)
    if getattr(fl, "neural", False):   # an ODE fleet (the plant comparison) has no hidden states
        out["h"] = fl.net_states()
    return out


# net, net_kernel, expected kernel, cost, E, K, T
ORACLE_CASES = [("gru32", None, "tensor", GRADMIN, 1, 200, 20),
                ("gru64", None, "tensor", GRAD, 3, 200, 20),
                ("gru32", "fp32", "fp32", QB, 3, 70, 20),
                ("dense32", None, "fp32", GRADMIN, 9, 40, 20),
                ("diff32", None, "fp32", GRAD, 3, 50, 20)]


@pytest.mark.parametrize("net,net_kernel,kernel,cost,E,K,T", ORACLE_CASES)
def test_neural_fleet_matches_oracle_teacher_forced(net, net_kernel, kernel, cost, E, K, T):
    """Every period starts oracle.mppi_step_net from the fleet's own state, warm start, last control and hidden state;
    the hidden state after the period is oracle.net_rollout's on (u, s), the next state oracle.plant_period's from the
    recorded state and Q.  10 periods, target equilibrium flipped to -1 at period 5 in the odd experiments, non-zero
    starting hidden states."""
    P = 10
    sp = _spec(net)
    fl = make(E, K, T, cost, net=net, net_kernel=net_kernel)
    htot = fl.engine.net_htot
    rng = np.random.default_rng(5)
    noise = rng.standard_normal((P, E, fl.n_ind, K)).astype(np.float32)
    tp, te = targets(P, E, 3, flip=5)
    fl.reset(random_states(E, 11))
    fl.set_net_states(rng.uniform(-0.3, 0.3, (E, htot)).astype(np.float32))
    d_noise, d_tp, d_te = cuda(noise), cuda(tp), cuda(te)
    worst = dict(J=0.0, u=0.0, u_nom=0.0, h=0.0, state=0.0)
    for j in range(P):
        s, u_nom, u_prev = fl.states(with_u_nom=True)
        H = fl.net_states()
        rec, J = torch.zeros((1, E, 16), device="cuda"), torch.zeros((1, E, K), device="cuda")
        fl.run(1, d_tp[j:j + 1].contiguous(), d_te[j:j + 1].contiguous(), d_noise[j:j + 1].contiguous(), rec, J)
        assert fl.engine.net_last_kernel() == kernel
        s2, u_nom2, u2 = fl.states(with_u_nom=True)
        H2 = fl.net_states()
        rec, J = rec.cpu().numpy()[0], J.cpu().numpy()[0]
        for e in range(E):
            kw = dict(h0=H[e], u_prev=float(u_prev[e]), target_position=float(tp[j, e]),
                      target_equilibrium=float(te[j, e]))
            with O.net_differential(sp["diff"]):   # None: a plain network
                ref = O.mppi_step_net(cost, *oracle_args(sp), s[e], u_nom[e], noise[j, e].T.copy(), **kw)
            if cost in ("default", QB):
                assert shifted_cost_ok(J[e], ref["J"]), (j, e)
            else:
                eJ = vec_err(J[e], ref["J"])
                worst["J"] = max(worst["J"], eJ)
                assert eJ < 1e-5, (j, e, eJ)
            eu, en = abs(float(u2[e]) - float(ref["u"])), float(np.abs(u_nom2[e] - ref["u_nom"]).max())
            worst["u"], worst["u_nom"] = max(worst["u"], eu), max(worst["u_nom"], en)
            assert eu < 1e-4 and en < 1e-4, (j, e, eu, en)
            if sp["net_type"] == "GRU":   # advanced on (u, s), u the fleet's own
                with O.net_differential(sp["diff"]):
                    _, hf = O.net_rollout(*oracle_args(sp), s[e], np.array([[u2[e]]], np.float32), h0=H[e], want_h=True)
                eh = float(np.abs(H2[e] - hf[0]).max())
                worst["h"] = max(worst["h"], eh)
                assert eh < 5e-6, (j, e, eh)
            else:                           # Dense: nothing to advance
                np.testing.assert_array_equal(H2[e], H[e])
            np.testing.assert_array_equal(rec[e, [1, 2, 4, 5, 6, 7]], s[e][[0, 1, 2, 3, 4, 5]])
            assert rec[e, 9] == u2[e] and rec[e, 10] == u2[e] and rec[e, 12] == tp[j, e] and rec[e, 13] == te[j, e]
            ps, _, _ = O.plant_period(rec[e, [1, 2, 4, 5, 6, 7]], float(rec[e, 9]))
            es = state_err(s2[e], ps)
            worst["state"] = max(worst["state"], es)
            assert es < 3e-7, (j, e, es)
    record("fleet_neural_vs_oracle", f"{net}_{net_kernel or 'auto'}_{cost}_E{E}_K{K}", **worst)
    assert fl.engine.nonfinite_costs() == 0


# net, net_kernel, E, K: the tensor-core kernel at its three occupancies (E x K on each side of 32 and 64 x SMs), the FP32
# kernel for a forced GRU and a Dense network; every K leaves a partial tile
BIT_CASES = [("gru32", None, 2, 1000), ("gru64", None, 3, 2000), ("gru32", None, 5, 2000),
             ("gru32", "fp32", 3, 200), ("dense32", None, 4, 100)]


@pytest.mark.parametrize("net,net_kernel,E,K", BIT_CASES)
def test_neural_fleet_is_bit_identical_to_engine_mppi_step(monkeypatch, net, net_kernel, E, K):
    """Two periods; each experiment's solve re-run by Engine.mppi_step on the same kernel at the same tile occupancy, fed
    the fleet's state, warm start, last control, hidden state, targets and draws: u, u_nom, J and the advanced hidden
    state agree bit for bit."""
    from cartpolesimulation_b200 import _lib as L
    from cartpolesimulation_b200.core import Engine
    T, P = 50, 2
    cost = GRADMIN
    fl = make(E, K, T, cost, net=net, net_kernel=net_kernel)
    eng = Engine(K, T, integrator="neural", cost=cost, device=0, net_kernel=net_kernel)
    eng.net_load(engine_spec(_spec(net)))
    if net_kernel is None and net != "dense32":
        monkeypatch.setenv("CPS_TC_ROWS", str(tc_rows(E * K)))
    rng = np.random.default_rng(E * K)
    noise = rng.standard_normal((P, E, fl.n_ind, K)).astype(np.float32)
    tp, te = targets(P, E, 9, flip=1)
    fl.reset(random_states(E, 21))
    fl.set_net_states(rng.uniform(-0.3, 0.3, (E, fl.engine.net_htot)).astype(np.float32))
    for j in range(P):
        s, u_nom, u_prev = fl.states(with_u_nom=True)
        H = fl.net_states()
        J = torch.zeros((1, E, K), device="cuda")
        fl.run(1, cuda(tp[j:j + 1]), cuda(te[j:j + 1]), cuda(noise[j:j + 1]), None, J)
        _, u_nom2, u2 = fl.states(with_u_nom=True)
        H2, J = fl.net_states(), J.cpu().numpy()[0]
        for e in range(E):
            eng.set_variable_parameters(float(tp[j, e]), float(te[j, e]))
            eng.set_u_nom(u_nom[e])
            eng.net_set_state(H[e])
            Je = torch.empty(K, device="cuda")
            u = eng.mppi_step(cuda(s[e]), cuda(noise[j, e]), L.TIME_MAJOR, float(u_prev[e]), None, Je)
            torch.cuda.synchronize()
            assert eng.net_last_kernel() == fl.engine.net_last_kernel()
            assert float(u.cpu()[0]) == float(u2[e]), (j, e)
            np.testing.assert_array_equal(eng.get_u_nom(), u_nom2[e])
            np.testing.assert_array_equal(Je.cpu().numpy(), J[e])
            np.testing.assert_array_equal(eng.net_get_state(), H2[e])


def test_neural_fleet_philox_and_split():
    """A Philox fleet equals a supplied fleet fed Fleet.noise(j); one fleet equals two fleets split by experiment_offset."""
    from cartpolesimulation_b200.fleet import Fleet
    E, K, T, P = 6, 300, 30, 3
    tp, te = targets(P, E, 2, flip=1)
    a = make(E, K, T, GRAD, noise="philox", seed=7)
    ra = run_periods(a, P, tp, te)
    noise = np.stack([a.noise(j).cpu().numpy() for j in range(P)])
    b = make(E, K, T, GRAD, noise="supplied")
    rb = run_periods(b, P, tp, te, noise=noise)
    for k in ra:
        np.testing.assert_array_equal(ra[k], rb[k], err_msg=k)
    s0 = random_states(E, 11)
    parts = []
    for off in (0, 3):
        f = make(3, K, T, GRAD, noise="philox", seed=7, experiment_offset=off)
        parts.append(run_periods(f, P, tp[:, off:off + 3], te[:, off:off + 3], s0=s0[off:off + 3]))
    for k in ("rec", "J"):
        np.testing.assert_array_equal(np.concatenate([p[k] for p in parts], axis=1), ra[k], err_msg=k)
    for k in ("s", "u_nom", "u_prev", "h"):
        np.testing.assert_array_equal(np.concatenate([p[k] for p in parts], axis=0), ra[k], err_msg=k)


def test_neural_fleet_experiments_are_independent():
    """Permuting the experiments permutes every output bit for bit; a NaN target stays inside its experiment and is counted;
    the handle's stored hidden state is read at reset() and never written."""
    E, K, T, P = 5, 200, 25, 4
    perm = np.array([3, 0, 4, 1, 2])
    rng = np.random.default_rng(1)
    tp, te = targets(P, E, 5, flip=2)
    fl = make(E, K, T, GRADMIN)
    noise = rng.standard_normal((P, E, fl.n_ind, K)).astype(np.float32)
    h0 = rng.uniform(-0.3, 0.3, (E, fl.engine.net_htot)).astype(np.float32)
    s0 = random_states(E, 4)
    stored = rng.uniform(-0.2, 0.2, fl.engine.net_htot).astype(np.float32)
    fl.engine.net_set_state(stored)
    fl.reset(s0)
    np.testing.assert_array_equal(fl.net_states(), np.broadcast_to(stored, (E, stored.size)))
    r1 = run_periods(fl, P, tp, te, noise=noise, h0=h0, s0=s0)
    rp = run_periods(fl, P, tp[:, perm], te[:, perm], noise=noise[:, perm], h0=h0[perm], s0=s0[perm])
    for k in ("rec", "J"):
        np.testing.assert_array_equal(rp[k], r1[k][:, perm], err_msg=k)
    for k in ("s", "u_nom", "u_prev", "h"):
        np.testing.assert_array_equal(rp[k], r1[k][perm], err_msg=k)
    assert fl.engine.nonfinite_costs() == 0
    tp_nan = tp.copy()
    tp_nan[1:, 2] = np.nan
    rn = run_periods(fl, P, tp_nan, te, noise=noise, h0=h0, s0=s0)
    others = [0, 1, 3, 4]
    np.testing.assert_array_equal(rn["rec"][:, others], r1["rec"][:, others])
    np.testing.assert_array_equal(rn["h"][others], r1["h"][others])
    assert fl.engine.nonfinite_costs() > 0
    np.testing.assert_array_equal(fl.engine.net_get_state(), stored)


def test_neural_fleet_plant_matches_the_ode_fleet():
    """With lo = hi = q every solve returns q: the record rows (states, derivatives, controls, targets) of a neural fleet
    and of an ODE Fleet from the same initial states agree bit for bit."""
    from cartpolesimulation_b200.fleet import Fleet
    E, K, T, P = 7, 64, 10, 25
    tp, te = targets(P, E, 6, flip=9)
    s0 = random_states(E, 8)
    recs = []
    for fl in (make(E, K, T, GRADMIN, noise="philox"), Fleet(E, K, T, cost=GRADMIN, noise="philox")):
        fl.engine.set_mppi_params(lo=0.3, hi=0.3)
        recs.append(run_periods(fl, P, tp, te, s0=s0))
    np.testing.assert_array_equal(recs[0]["rec"], recs[1]["rec"])
    np.testing.assert_array_equal(recs[0]["s"], recs[1]["s"])
    assert np.all(recs[0]["rec"][:, :, 9] == np.float32(0.3))


class _Draws:
    def __init__(self, draws):
        self.draws, self.i = list(draws), 0

    def normal(self, shape, mean=0.0, stddev=1.0, dtype=None):
        d = self.draws[self.i]
        self.i += 1
        assert list(d.shape) == list(shape)
        return d * stddev + mean


def test_neural_fleet_agrees_with_optimizer_mppi_b200(tmp_path):
    """optimizer_mppi_b200 on a PredictorWrapper configured with a GRU 2 x 32 model directory, driven with the same draws
    and the fleet's plant states (oracle.plant_period between the solves is the fleet's own plant), closed loop."""
    import cartpolesimulation_b200 as cps
    from cartpolesimulation_b200.fleet import Fleet
    from cartpolesimulation_b200.optimizer_mppi_b200 import _extract_net_spec, optimizer_mppi_b200
    from tests.netutil import write_model_dir
    z, _ = load_golden(NETS["gru32"])
    K, T, P, tp = 2000, 50, 8, 0.03
    vp = cps.VariableParameters(target_position=tp, target_equilibrium=1.0, L=0.395, m_pole=0.087)
    cost, predictor = cps.CostFunctionWrapper(), cps.PredictorWrapper()
    predictor.configure(batch_size=K, horizon=T, dt=0.02, variable_parameters=vp,
                        predictor_specification=write_model_dir(str(tmp_path), z))
    cost.configure(batch_size=K, horizon=T, variable_parameters=vp, environment_name="CartPole", computation_library=None,
                   cost_function_specification=GRADMIN)
    opt = optimizer_mppi_b200(predictor=predictor, cost_function=cost,
                              control_limits=(np.array([-1.0], np.float32), np.array([1.0], np.float32)), seed=1,
                              mpc_horizon=T, num_rollouts=K)
    opt.configure(num_states=6, num_control_inputs=1, default_configure=False, dt=0.02, predictor_specification="neural")
    assert opt.predictor_type == "neural"
    fl = Fleet(1, K, T, cost=GRADMIN, noise="supplied", integrator="neural", network=_extract_net_spec(predictor))
    rng = np.random.default_rng(41)
    noise = rng.standard_normal((P, 1, fl.n_ind, K)).astype(np.float32)
    opt.rng = _Draws([torch.from_numpy(noise[j, 0].T[:, :, None].copy()) for j in range(P)])
    fl.reset(random_states(1, 42))
    eu = en = 0.0
    s = fl.states()[0]
    for j in range(P):
        u_opt = float(opt.step(s.copy()))
        rec = torch.zeros((1, 1, 16), device="cuda")
        fl.run(1, cuda(np.full((1, 1), tp)), None, cuda(noise[j:j + 1]), rec)
        _, u_nom, u = fl.states(with_u_nom=True)
        eu = max(eu, abs(float(u[0]) - u_opt))
        en = max(en, float(np.abs(u_nom[0] - opt.optimal_control_sequence.reshape(-1)).max()))
        assert eu < 1e-6 and en < 1e-6, (j, eu, en)
        r = rec.cpu().numpy()[0, 0]
        s_next, _, _ = O.plant_period(r[[1, 2, 4, 5, 6, 7]], float(r[9]))
        assert state_err(fl.states()[0], s_next) < 3e-7
        s = fl.states()[0]
    record("fleet_neural_optimizer", "gru32_gradmin_K2000", u=eu, u_nom=en)


def test_neural_fleet_bookkeeping_and_rejections(tmp_path):
    """Launches per period (2 supplied, 3 Philox, whatever E), the kernel each network runs on, every rejection, and the
    reference's CSV from a neural fleet's records."""
    from cartpolesimulation_b200 import _lib as L
    from cartpolesimulation_b200.core import Engine
    from cartpolesimulation_b200.fleet import make_experiments
    from cartpolesimulation_b200.recording import save_fleet_recordings
    K, T = 64, 10
    for E in (1, 37):
        for noise, per in (("supplied", 2), ("philox", 3)):
            fl = make(E, K, T, GRADMIN, noise=noise)
            tp, te = targets(2, E, 1)
            fl.reset(random_states(E, 3))
            n0 = fl.engine.launch_count()
            fl.run(2, cuda(tp), cuda(te), cuda(np.zeros((2, E, fl.n_ind, K))) if noise == "supplied" else None)
            assert fl.engine.launch_count() - n0 == 2 * per
    for net, nk, kernel in (("gru32", None, "tensor"), ("gru64", None, "tensor"), ("gru32", "fp32", "fp32"),
                            ("dense32", None, "fp32"), ("diff32", None, "fp32")):
        fl = make(3, K, T, GRADMIN, net=net, net_kernel=nk, noise="philox")
        fl.reset(random_states(3, 3))
        fl.run(1)
        assert fl.engine.net_last_kernel() == kernel, net
    # rejections on a neural fleet
    fl = make(2, K, T, GRADMIN, noise="philox")
    fl.reset(random_states(2, 3))
    eng, h = fl.engine, fl.engine._h
    with pytest.raises(NotImplementedError):
        fl.set_plant_models(control_noise_mode="additive", control_noise=0.1)
    m = L.cps_fleet_plant_models(C.sizeof(L.cps_fleet_plant_models), 1, 0.1, 0.0, 0, 0.0, 0.0, 0.0, 0.0, 0.0)
    assert eng.lib.cps_fleet_set_plant_models(h, C.byref(m)) == ERR_UNSUPPORTED
    assert eng.lib.cps_fleet_step_noisy(h, 1, None, None, None, None, None, None, None) == ERR_UNSUPPORTED
    st, q = torch.zeros((1, 2, 6), device="cuda"), torch.zeros((1, 2), device="cuda")
    assert eng.lib.cps_fleet_relabel(h, 1, C.c_void_p(st.data_ptr()), None, None, None, None, None,
                                     C.c_void_p(q.data_ptr()), None) == ERR_UNSUPPORTED
    assert eng.lib.cps_fleet_relabel_masked(h, 1, C.c_void_p(st.data_ptr()), None, None, None, None, None,
                                            C.c_void_p(q.data_ptr()), None, None) == ERR_UNSUPPORTED
    # a network of another hidden size loaded after create: recreate the fleet
    eng.net_load(engine_spec(_spec("gru64")))
    with pytest.raises(ValueError, match="recreate"):
        fl.run(1)
    # a neural handle without a network; the tensor-core flag with a network it cannot take; an ODE fleet's hidden states
    c = L.cps_fleet_config(C.sizeof(L.cps_fleet_config), 2, 10, L.FLEET_NOISE_PHILOX, 0.002, 0, 0)
    e2 = Engine(K, T, integrator="neural", cost=GRADMIN, device=0)
    assert e2.lib.cps_fleet_create(e2._h, C.byref(c)) == ERR_NOT_CONFIGURED
    e3 = Engine(K, T, integrator="neural", cost=GRADMIN, device=0, net_kernel="tensor")
    e3.net_load(engine_spec(_spec("dense32")))
    assert e3.lib.cps_fleet_create(e3._h, C.byref(c)) == ERR_UNSUPPORTED
    from cartpolesimulation_b200.fleet import Fleet
    ode = Fleet(2, K, T, cost=GRADMIN)
    out = np.zeros(4, np.float32)
    assert ode.engine.lib.cps_fleet_get_net_states(ode.engine._h, out.ctypes.data_as(L._FP)) == ERR_NOT_CONFIGURED
    assert ode.engine.lib.cps_fleet_set_net_states(ode.engine._h, out.ctypes.data_as(L._FP)) == ERR_NOT_CONFIGURED
    # CSV
    E, P = 3, 20
    s0, tp, te = make_experiments(E, P, seed=2)
    fl = make(E, K, T, GRADMIN, net="dense32", noise="philox", seed=2)
    fl.reset(s0)
    rec = torch.zeros((P, E, 16), device="cuda")
    fl.run(P, cuda(tp), cuda(te), None, rec)
    r = rec.cpu().numpy()
    assert np.all(np.isfinite(r)) and np.all(np.abs(r[:, :, 9]) <= 1.0)
    paths = save_fleet_recordings(rec, str(tmp_path), optimizer_name="mppi-b200", run_for_ML_Pipeline=False)
    assert len(paths) == E
    with open(paths[1]) as f:
        rows = [row for row in csv.reader(line for line in f if not line.startswith("#"))]
    assert rows[0][:15] == ["time", "angle", "angleD", "angleDD", "angle_cos", "angle_sin", "position", "positionD",
                            "positionDD", "Q_calculated", "Q_applied", "Q_ccrc", "u", "target_position", "target_equilibrium"]
    assert len(rows) == P + 1
    np.testing.assert_allclose(np.array([float(x[1]) for x in rows[1:]]), r[:, 1, 1], rtol=1e-6, atol=1e-6)
