"""GPU parity of the autoregressive neural predictor (cps_net_*; net_kernel) and of the MPPI solve that drives it,
against goldens from the unmodified reference (tests/golden/net_*.npz, mppi_net_*.npz) and against the CPU oracle.
Tolerances: trajectories 1e-5 range-relative (north_star; measured ~1e-6), J 1e-5, controls 1e-4."""
import numpy as np
import pytest

from tests.netutil import net_spec_from_golden
from tests.parity import load_golden, record, shifted_cost_ok, traj_err, vec_err

pytestmark = pytest.mark.gpu

NET_GOLDENS = ["net_GRU_6IN_64H1_64H2_5OUT_0", "net_GRU_6IN_32H1_32H2_5OUT_0", "net_Dense_6IN_32H1_32H2_5OUT_0"]
MPPI_NET_RUNS = ["gru64_gradmin", "gru32_grad", "dense32_gradmin",
                 "diff_gru32_gradmin",   # differential network (SURVEY 8a row a15) under the optimizer
                 "gru32_qb"]             # MAX_COST plugin with the neural predictor (backend-ordered cost mean)
NET_DIFF_GOLDENS = ["net_diff_GRU_6IN_32H1_32H2_5OUT_1", "net_diff_Dense_5IN_32H1_32H2_4OUT_1",
                    "net_diff_GRU_6IN_64H1_64H2_5OUT_1"]


def engine_spec(sp):
    from oracle import oracle as O
    d = dict(sp)
    d["weights"] = O.pack_net_weights(sp["net_type"], sp["layers"], sp["out_layer"])
    if sp.get("diff") is not None:   # differential network: cps_net_desc fields (include/cps.h)
        f = sp["diff"]
        d.update(differential=True, diff_p1=f["p1"], diff_p2=f["p2"], out_norm_a=f["on_a"], out_norm_b=f["on_b"],
                 out_to_in=f["out_to_in"])
    return d


def oracle_args(sp):
    from oracle import oracle as O
    return (sp["net_type"], sp["hsz"], O.pack_net_weights(sp["net_type"], sp["layers"], sp["out_layer"]), sp["in_idx"],
            sp["out_idx"], sp["norm_a"], sp["norm_b"], sp["denorm_A"], sp["denorm_B"])


def make_engine(sp, K, T, cost=None, net_kernel=None):
    from cartpolesimulation_b200.core import Engine
    eng = Engine(K, T, integrator="neural", cost=cost, device=0, net_kernel=net_kernel)
    eng.net_load(engine_spec(sp))
    return eng


def fp32_unless_gru64(sp):
    """The generic tests below pin the FP32 kernel for every network except the plain 2 x 64 GRU (their tolerances were
    measured there); the tensor-core kernel, which narrower plain GRUs now run on by default (zero-padded to 64 units), has
    its own tests further down."""
    return None if (sp["net_type"] == "GRU" and list(sp["hsz"]) == [64, 64] and sp.get("diff") is None) else "fp32"


@pytest.mark.parametrize("name", NET_GOLDENS)
def test_net_rollout_vs_reference_golden(name):
    import torch
    z, m = load_golden(name)
    sp = net_spec_from_golden(z)
    K, T = z["Q"].shape
    eng = make_engine(sp, K, T, net_kernel=fp32_unless_gru64(sp))
    dev = eng.device
    Q = torch.from_numpy(z["Q"]).to(dev)
    traj, _ = eng.net_rollout(torch.from_numpy(z["s0"]).to(dev), Q)
    assert max(traj_err(traj.cpu().numpy(), z["traj_zero_h"]).values()) < 1e-5
    e1 = max(traj_err(traj.cpu().numpy()[:, :2], z["traj_zero_h"][:, :2]).values())
    assert e1 < 2e-6, e1
    for s, q in zip(z["upd_s"], z["upd_q"]):
        eng.net_update(torch.from_numpy(s).to(dev), torch.tensor([q], device=dev))
    if sp["net_type"] == "GRU":
        assert np.abs(eng.net_get_state() - z["h_after_updates"].reshape(-1)).max() < 2e-6
    else:
        assert eng.net_htot == 0 or sp["net_type"] == "Dense"
    traj2, _ = eng.net_rollout(torch.from_numpy(z["s_after"]).to(dev), Q)
    assert max(traj_err(traj2.cpu().numpy(), z["traj_after_updates"]).values()) < 1e-5
    # per-rollout initial states, time-major layouts, explicit shared h0, hidden state out
    h0 = torch.from_numpy(eng.net_get_state()).to(dev) if eng.net_htot else None
    traj3, hf = eng.net_rollout(torch.from_numpy(z["s_rand"]).to(dev), Q.t().contiguous(), q_layout=1, traj_layout=1,
                                h0=h0, want_h=True)
    t3 = traj3.permute(2, 0, 1).cpu().numpy()
    assert max(traj_err(t3, z["traj_rand"]).values()) < 1e-5
    # the stored state is untouched by rollouts
    if sp["net_type"] == "GRU":
        assert np.abs(eng.net_get_state() - z["h_after_updates"].reshape(-1)).max() < 2e-6
        eng.net_reset_state()
        assert np.abs(eng.net_get_state()).max() == 0.0


@pytest.mark.parametrize("name", NET_GOLDENS[:2])
@pytest.mark.parametrize("B,T", [(1, 1), (17, 3), (2000, 50), (4099, 20)])
def test_net_rollout_vs_oracle_sizes(name, B, T):
    """ragged tiles (B not a multiple of 16), per-rollout hidden states, B = 1."""
    import torch
    from oracle import oracle as O
    z, m = load_golden(name)
    sp = net_spec_from_golden(z)
    eng = make_engine(sp, B, T, net_kernel=fp32_unless_gru64(sp))
    dev = eng.device
    rng = np.random.default_rng(B * 100 + T)
    ang = rng.uniform(-np.pi, np.pi, B)
    s0 = np.stack([ang, rng.uniform(-3, 3, B), np.cos(ang), np.sin(ang), rng.uniform(-0.15, 0.15, B),
                   rng.uniform(-0.5, 0.5, B)], 1).astype(np.float32)
    Q = rng.uniform(-1, 1, (B, T)).astype(np.float32)
    h0 = rng.uniform(-0.5, 0.5, (B, sum(sp["hsz"]))).astype(np.float32)
    ref, href = O.net_rollout(*oracle_args(sp), s0, Q, h0=h0, want_h=True)
    traj, hf = eng.net_rollout(torch.from_numpy(s0).to(dev), torch.from_numpy(Q).to(dev), h0=torch.from_numpy(h0).to(dev),
                               want_h=True)
    e = traj_err(traj.cpu().numpy(), ref)
    # angle = atan2(sin, cos) of un-normalised network outputs: ill-conditioned where |(sin, cos)| is small, so the
    # angle channel amplifies the 1e-7 differences of the other channels by 1/|(sin, cos)|
    assert e.pop("angle") < 1e-4
    assert max(e.values()) < 2e-6, e
    assert np.abs(hf.cpu().numpy() - href).max() < 5e-6


@pytest.mark.parametrize("name", NET_DIFF_GOLDENS)
def test_net_diff_rollout_vs_reference_golden(name):
    """SURVEY 8a row a15: differential networks (outputs D_*; autoregression.py:118-158, Normalising.py:111-186) on
    net_kernel against the unmodified reference predictor: permuted inputs (output -> input gather), an `angle` output
    with sin / cos augmentation, the hidden state after updates, per-rollout initial states, horizon 1 (raw network
    output: the reference's loop routes around the helper).  The network description comes from the PRODUCT's
    build_net_spec and must equal the test's independent derivation."""
    import torch
    from cartpolesimulation_b200.neural import build_net_spec
    from oracle import oracle as O
    z, m = load_golden(name)
    sp = net_spec_from_golden(z)
    w = O.pack_net_weights(sp["net_type"], sp["layers"], sp["out_layer"])
    spec = build_net_spec(m["type"], m["inputs"], m["outputs"], sp["hsz"], w,
                          ([str(c) for c in z["norm_cols"]], z["norm_table"]), dt=m["dt"])
    assert spec["differential"]
    ref_spec = engine_spec(sp)
    for k in ("in_idx", "out_idx", "out_to_in"):
        assert list(spec[k]) == list(ref_spec[k]), k
    for k in ("norm_a", "norm_b", "denorm_A", "denorm_B", "diff_p1", "diff_p2", "out_norm_a", "out_norm_b"):
        np.testing.assert_array_equal(np.asarray(spec[k], np.float32), np.asarray(ref_spec[k], np.float32), err_msg=k)
    from cartpolesimulation_b200.core import Engine
    K, T = z["Q"].shape
    eng = Engine(K, T, integrator="neural", cost=None, device=0)
    eng.net_load(spec)
    dev = eng.device
    Q = torch.from_numpy(z["Q"]).to(dev)
    traj, _ = eng.net_rollout(torch.from_numpy(z["s0"]).to(dev), Q)
    e0 = max(traj_err(traj.cpu().numpy(), z["traj_zero_h"]).values())
    for s_, q_ in zip(z["upd_s"], z["upd_q"]):
        eng.net_update(torch.from_numpy(s_).to(dev), torch.tensor([q_], device=dev))
    eh = 0.0
    if sp["net_type"] == "GRU":
        eh = float(np.abs(eng.net_get_state() - z["h_after_updates"].reshape(-1)).max())
    traj3, _ = eng.net_rollout(torch.from_numpy(z["s_rand"]).to(dev), Q.t().contiguous(), q_layout=1, traj_layout=1)
    e3 = max(traj_err(traj3.permute(2, 0, 1).cpu().numpy(), z["traj_rand"]).values())
    # horizon 1 on a fresh handle (the generator used a fresh predictor: zero hidden state)
    eng1 = Engine(K, 1, integrator="neural", cost=None, device=0)
    eng1.net_load(spec)
    t1, _ = eng1.net_rollout(torch.from_numpy(z["s_rand"]).to(dev), Q[:, :1].contiguous())
    e1 = max(traj_err(t1.cpu().numpy(), z["traj_rand_T1"]).values())
    record("net_diff_rollout_vs_reference_golden", name, zero_h=e0, h_after_updates=eh, per_rollout_states=e3, horizon1=e1)
    assert e0 < 1e-5 and e3 < 1e-5 and e1 < 2e-6 and eh < 2e-6, (e0, e3, e1, eh)
    # the tensor-core kernel does not implement the differential feedback: asking for it is an error, not a wrong answer
    if name.endswith("64H1_64H2_5OUT_1"):
        eng_tc = Engine(K, T, integrator="neural", cost=None, device=0, net_kernel="tensor")
        eng_tc.net_load(spec)
        with pytest.raises(NotImplementedError):
            eng_tc.net_rollout(torch.from_numpy(z["s0"]).to(dev), Q)


@pytest.mark.parametrize("B,T", [(1, 2), (17, 3), (2000, 50)])
def test_net_diff_rollout_vs_oracle_sizes(B, T):
    import torch
    from oracle import oracle as O
    z, m = load_golden(NET_DIFF_GOLDENS[0])
    sp = net_spec_from_golden(z)
    eng = make_engine(sp, B, T)
    dev = eng.device
    rng = np.random.default_rng(B * 100 + T)
    ang = rng.uniform(-np.pi, np.pi, B)
    s0 = np.stack([ang, rng.uniform(-3, 3, B), np.cos(ang), np.sin(ang), rng.uniform(-0.15, 0.15, B),
                   rng.uniform(-0.5, 0.5, B)], 1).astype(np.float32)
    Q = rng.uniform(-1, 1, (B, T)).astype(np.float32)
    h0 = rng.uniform(-0.5, 0.5, (B, sum(sp["hsz"]))).astype(np.float32)
    with O.net_differential(sp["diff"]):
        ref, href = O.net_rollout(*oracle_args(sp), s0, Q, h0=h0, want_h=True)
    traj, hf = eng.net_rollout(torch.from_numpy(s0).to(dev), torch.from_numpy(Q).to(dev), h0=torch.from_numpy(h0).to(dev),
                               want_h=True)
    e = traj_err(traj.cpu().numpy(), ref)
    record("net_diff_rollout_vs_oracle_sizes", f"B{B}_T{T}", **e, h=float(np.abs(hf.cpu().numpy() - href).max()))
    assert e.pop("angle") < 1e-4
    assert max(e.values()) < 5e-6, e
    assert np.abs(hf.cpu().numpy() - href).max() < 5e-6


@pytest.mark.parametrize("run", MPPI_NET_RUNS)
def test_net_mppi_vs_reference_golden(run):
    import torch
    from cartpolesimulation_b200 import _lib as L
    z, m = load_golden("mppi_net_" + run)
    sp = net_spec_from_golden(z)
    K, T = m["K"], m["T"]
    eng = make_engine(sp, K, T, cost=m["cost"], net_kernel=fp32_unless_gru64(sp))
    eng.set_variable_parameters(m["target_position"], m["target_equilibrium"])
    dev = eng.device
    J = torch.empty(K, device=dev)
    traj = torch.empty((K, T + 1, 6), device=dev)
    u_run = torch.empty((K, T), device=dev)
    u_nom = np.zeros(T, dtype=np.float32)
    h = np.zeros(sum(sp["hsz"]), np.float32)
    for i in range(m["steps"]):
        eng.set_u_nom(u_nom)
        eng.net_set_state(h)
        eps = torch.from_numpy(z["eps"][i]).to(dev)  # [K, n_ind], the reference's layout
        u = eng.mppi_step(torch.from_numpy(z["s"][i]).to(dev), eps, L.ROLLOUT_MAJOR, float(z["u_prev"][i]), None, J, traj,
                          L.ROLLOUT_MAJOR, u_run)
        torch.cuda.synchronize()
        if i == 0:
            np.testing.assert_allclose(u_run.cpu().numpy(), z["u_run0"], rtol=0, atol=2e-7)
            assert max(traj_err(traj.cpu().numpy()[:32], z["traj0"]).values()) < 1e-5
        Jg = J.cpu().numpy()
        du, dn = abs(float(u.cpu()[0]) - float(z["u"][i])), float(np.abs(eng.get_u_nom() - z["u_nom"][i]).max())
        record("net_mppi_vs_reference_golden", f"{run}/{i}", J=vec_err(Jg, z["J"][i]), u=du, u_nom=dn)
        if m["cost"] in ("default", "quadratic_boundary"):
            assert shifted_cost_ok(Jg, z["J"][i])
        else:
            assert vec_err(Jg, z["J"][i]) < 1e-5
        assert du < 2e-5      # measured <= 9.1e-6 (gru32_grad); north_star: 1e-4
        np.testing.assert_allclose(eng.get_u_nom(), z["u_nom"][i], rtol=0, atol=2e-5)
        if sp["net_type"] == "GRU":  # the solve advanced the stored hidden state on (u, s) (optimizer_mppi.py:191)
            assert np.abs(eng.net_get_state() - z["h_after"][i]).max() < 5e-6
            h = z["h_after"][i].copy()
        u_nom = z["u_nom"][i].copy()
    assert eng.nonfinite_costs() == 0


def test_net_mppi_K2000_vs_oracle_and_time_major_noise():
    import torch
    from oracle import oracle as O
    from cartpolesimulation_b200 import _lib as L
    z, m = load_golden("mppi_net_gru64_gradmin")
    sp = net_spec_from_golden(z)
    K, T = 2000, 50
    eng = make_engine(sp, K, T, cost="quadratic_boundary_grad_minimal")
    dev = eng.device
    rng = np.random.default_rng(5)
    eps = rng.standard_normal((K, eng.n_ind)).astype(np.float32)
    u_nom = rng.uniform(-0.3, 0.3, T).astype(np.float32)
    h = rng.uniform(-0.3, 0.3, sum(sp["hsz"])).astype(np.float32)
    s = z["s"][1]
    ref = O.mppi_step_net("quadratic_boundary_grad_minimal", *oracle_args(sp), s, u_nom, eps, h0=h, u_prev=0.1)
    eng.set_u_nom(u_nom)
    eng.net_set_state(h)
    J = torch.empty(K, device=dev)
    u = eng.mppi_step(torch.from_numpy(s).to(dev), torch.from_numpy(np.ascontiguousarray(eps.T)).to(dev), L.TIME_MAJOR, 0.1,
                      None, J)
    assert vec_err(J.cpu().numpy(), ref["J"]) < 1e-5
    assert abs(float(u.cpu()[0]) - float(ref["u"])) < 1e-4
    np.testing.assert_allclose(eng.get_u_nom(), ref["u_nom"], rtol=0, atol=1e-4)
    _, hf = O.net_rollout(*oracle_args(sp), s, np.array([[ref["u"]]], np.float32), h0=h, want_h=True)
    assert np.abs(eng.net_get_state() - hf[0]).max() < 5e-6


def test_net_errors():
    from cartpolesimulation_b200.core import Engine
    import torch
    eng = Engine(64, 10, integrator="neural", cost=None, device=0)
    with pytest.raises(RuntimeError):  # CPS_ERR_NOT_CONFIGURED: no network loaded
        eng.net_htot = 0
        eng.net_rollout(torch.zeros(6, device=eng.device), torch.zeros((4, 10), device=eng.device))
    z, m = load_golden(NET_GOLDENS[0])
    sp = engine_spec(net_spec_from_golden(z))
    bad = dict(sp)
    bad["weights"] = sp["weights"][:-1]
    with pytest.raises(ValueError):
        eng.net_load(bad)
    bad = dict(sp)
    bad["net_type"] = "LSTM"
    with pytest.raises(NotImplementedError):
        eng.net_load(bad)


# ------------------------------------------------------------------------------------------------------------
# tensor-core kernel (tcgen05, fp16 hi/lo split operands, fp32 accumulation in tensor memory): same tolerances
# ------------------------------------------------------------------------------------------------------------
TC_NET = "net_GRU_6IN_64H1_64H2_5OUT_0"


TC_NETS = [TC_NET, "net_GRU_6IN_32H1_32H2_5OUT_0"]   # the second: 32-unit layers zero-padded to the kernel's 64


@pytest.mark.parametrize("net", TC_NETS)
def test_tc_rollout_vs_reference_golden(net):
    import torch
    z, m = load_golden(net)
    sp = net_spec_from_golden(z)
    K, T = z["Q"].shape
    eng = make_engine(sp, K, T, net_kernel="tensor")
    dev = eng.device
    Q = torch.from_numpy(z["Q"]).to(dev)
    traj, _ = eng.net_rollout(torch.from_numpy(z["s0"]).to(dev), Q)
    e = traj_err(traj.cpu().numpy(), z["traj_zero_h"])
    assert max(e.values()) < 1e-5, e
    e1 = max(traj_err(traj.cpu().numpy()[:, :2], z["traj_zero_h"][:, :2]).values())
    assert e1 < 2e-6, e1
    for s, q in zip(z["upd_s"], z["upd_q"]):
        eng.net_update(torch.from_numpy(s).to(dev), torch.tensor([q], device=dev))
    assert np.abs(eng.net_get_state() - z["h_after_updates"].reshape(-1)).max() < 2e-6
    traj2, _ = eng.net_rollout(torch.from_numpy(z["s_after"]).to(dev), Q)
    assert max(traj_err(traj2.cpu().numpy(), z["traj_after_updates"]).values()) < 1e-5
    traj3, hf = eng.net_rollout(torch.from_numpy(z["s_rand"]).to(dev), Q.t().contiguous(), q_layout=1, traj_layout=1,
                                want_h=True)
    assert max(traj_err(traj3.permute(2, 0, 1).cpu().numpy(), z["traj_rand"]).values()) < 1e-5


@pytest.mark.parametrize("B,T", [(1, 1), (129, 3), (2000, 50), (4736, 4), (4737, 4), (6000, 10), (20000, 10)])
def test_tc_rollout_vs_oracle_sizes(B, T):
    import torch
    from oracle import oracle as O
    z, m = load_golden(TC_NET)
    sp = net_spec_from_golden(z)
    eng = make_engine(sp, B, T, net_kernel="tensor")
    dev = eng.device
    rng = np.random.default_rng(B * 100 + T)
    ang = rng.uniform(-np.pi, np.pi, B)
    s0 = np.stack([ang, rng.uniform(-3, 3, B), np.cos(ang), np.sin(ang), rng.uniform(-0.15, 0.15, B),
                   rng.uniform(-0.5, 0.5, B)], 1).astype(np.float32)
    Q = rng.uniform(-1, 1, (B, T)).astype(np.float32)
    h0 = rng.uniform(-0.5, 0.5, (B, sum(sp["hsz"]))).astype(np.float32)
    ref, href = O.net_rollout(*oracle_args(sp), s0, Q, h0=h0, want_h=True)
    traj, hf = eng.net_rollout(torch.from_numpy(s0).to(dev), torch.from_numpy(Q).to(dev), h0=torch.from_numpy(h0).to(dev),
                               want_h=True)
    e = traj_err(traj.cpu().numpy(), ref)
    assert e.pop("angle") < 1e-4     # atan2 of small-norm outputs, see test_net_rollout_vs_oracle_sizes
    assert max(e.values()) < 3e-6, e
    assert np.abs(hf.cpu().numpy() - href).max() < 5e-6


def test_tc_live_rollouts_per_cta_modes(monkeypatch):
    """the three tile occupancies of net_tc_kernel (32 / 64 / 128 live rollouts per CTA; chosen by batch size, forced here).
    64 and 128: every rollout's arithmetic is the same -> bit-identical trajectories and costs, the control differs only by
    the order of the block partials.  32: the hi / lo operand parts are stacked in two tensor-memory rows (two MMA passes,
    lo * lo term included) -> equal to rounding."""
    import torch
    from cartpolesimulation_b200 import _lib as L
    z, m = load_golden("mppi_net_gru64_gradmin")
    sp = net_spec_from_golden(z)
    K, T = 1000, 20
    rng = np.random.default_rng(5)
    noise_np = rng.standard_normal((K, 16)).astype(np.float32)
    out = {}
    for r in (32, 64, 128):
        monkeypatch.setenv("CPS_TC_ROWS", str(r))
        eng = make_engine(sp, K, T, cost="quadratic_boundary_grad_minimal", net_kernel="tensor")
        noise = torch.from_numpy(noise_np[:, :eng.n_ind].copy()).to(eng.device)
        J = torch.empty(K, device=eng.device)
        traj = torch.empty((K, T + 1, 6), device=eng.device)
        u = eng.mppi_step(torch.from_numpy(z["s"][1]).to(eng.device), noise, L.ROLLOUT_MAJOR, 0.0, None, J, traj, L.ROLLOUT_MAJOR)
        torch.cuda.synchronize()
        out[r] = (float(u.cpu()[0]), J.cpu().numpy(), traj.cpu().numpy(), eng.get_u_nom(), eng.net_get_state())
        assert eng.nonfinite_costs() == 0
    a, b, c = out[64], out[128], out[32]
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    for x in (b, c):
        assert abs(a[0] - x[0]) < 1e-6
        np.testing.assert_allclose(a[3], x[3], rtol=0, atol=1e-6)
        np.testing.assert_allclose(a[4], x[4], rtol=0, atol=1e-6)
    assert vec_err(c[1], a[1]) < 2e-6
    e = traj_err(c[2], a[2])
    record("tc_stacked_vs_three_pass", "K1000_T20", J=vec_err(c[1], a[1]), **e)
    assert max(e.values()) < 1e-5, e


def test_tc_mppi_vs_reference_golden():
    import torch
    from cartpolesimulation_b200 import _lib as L
    z, m = load_golden("mppi_net_gru64_gradmin")
    sp = net_spec_from_golden(z)
    K, T = m["K"], m["T"]
    eng = make_engine(sp, K, T, cost=m["cost"], net_kernel="tensor")
    dev = eng.device
    J = torch.empty(K, device=dev)
    traj = torch.empty((K, T + 1, 6), device=dev)
    u_run = torch.empty((K, T), device=dev)
    u_nom = np.zeros(T, dtype=np.float32)
    h = np.zeros(sum(sp["hsz"]), np.float32)
    for i in range(m["steps"]):
        eng.set_u_nom(u_nom)
        eng.net_set_state(h)
        eps = torch.from_numpy(z["eps"][i]).to(dev)
        u = eng.mppi_step(torch.from_numpy(z["s"][i]).to(dev), eps, L.ROLLOUT_MAJOR, float(z["u_prev"][i]), None, J, traj,
                          L.ROLLOUT_MAJOR, u_run)
        torch.cuda.synchronize()
        if i == 0:
            np.testing.assert_allclose(u_run.cpu().numpy(), z["u_run0"], rtol=0, atol=2e-7)
            assert max(traj_err(traj.cpu().numpy()[:32], z["traj0"]).values()) < 1e-5
        assert vec_err(J.cpu().numpy(), z["J"][i]) < 1e-5
        assert abs(float(u.cpu()[0]) - float(z["u"][i])) < 1e-4
        np.testing.assert_allclose(eng.get_u_nom(), z["u_nom"][i], rtol=0, atol=1e-4)
        assert np.abs(eng.net_get_state() - z["h_after"][i]).max() < 5e-6
        h = z["h_after"][i].copy()
        u_nom = z["u_nom"][i].copy()
    assert eng.nonfinite_costs() == 0


def test_tc_matches_fp32_kernel_K65536():
    """full-size property: both kernels, same inputs -> same costs and control (K = 65536, T = 50)."""
    import torch
    from cartpolesimulation_b200 import _lib as L
    z, m = load_golden("mppi_net_gru64_gradmin")
    sp = net_spec_from_golden(z)
    K, T = 65536, 50
    out = {}
    rng = np.random.default_rng(1)
    for kern in ("fp32", "tensor"):
        eng = make_engine(sp, K, T, cost="quadratic_boundary_grad_minimal", net_kernel=kern)
        if kern == "fp32":
            noise = torch.from_numpy(rng.standard_normal((eng.n_ind, K)).astype(np.float32)).to(eng.device)
        J = torch.empty(K, device=eng.device)
        u = eng.mppi_step(torch.from_numpy(z["s"][1]).to(eng.device), noise, L.TIME_MAJOR, 0.0, None, J)
        out[kern] = (float(u.cpu()[0]), J.cpu().numpy(), eng.get_u_nom(), eng.net_get_state())
        assert eng.nonfinite_costs() == 0
    assert vec_err(out["tensor"][1], out["fp32"][1]) < 1e-5
    assert abs(out["tensor"][0] - out["fp32"][0]) < 1e-5
    np.testing.assert_allclose(out["tensor"][2], out["fp32"][2], rtol=0, atol=1e-5)
    np.testing.assert_allclose(out["tensor"][3], out["fp32"][3], rtol=0, atol=5e-6)


@pytest.mark.parametrize("cost", ["quadratic_boundary", "default"])
def test_tc_matches_fp32_kernel_shifted_costs(cost):
    """MAX_COST plugins on the tensor-core kernel (backend-ordered row sum of the T+1 cost entries): same costs and control
    as the FP32 kernel, which is pinned against the reference (mppi_net_gru32_qb)."""
    import torch
    from cartpolesimulation_b200 import _lib as L
    z, m = load_golden("mppi_net_gru64_gradmin")
    sp = net_spec_from_golden(z)
    K, T = 4096, 50
    out = {}
    rng = np.random.default_rng(7)
    noise_np = rng.standard_normal((K, 16)).astype(np.float32)
    for kern in ("fp32", "tensor"):
        eng = make_engine(sp, K, T, cost=cost, net_kernel=kern)
        noise = torch.from_numpy(noise_np[:, :eng.n_ind].copy()).to(eng.device)
        J = torch.empty(K, device=eng.device)
        u = eng.mppi_step(torch.from_numpy(z["s"][1]).to(eng.device), noise, L.ROLLOUT_MAJOR, 0.0, None, J)
        out[kern] = (float(u.cpu()[0]), J.cpu().numpy(), eng.get_u_nom())
        assert eng.net_last_kernel() == kern
        assert eng.nonfinite_costs() == 0
    assert shifted_cost_ok(out["tensor"][1], out["fp32"][1])
    record("tc_vs_fp32_shifted", cost, u=abs(out["tensor"][0] - out["fp32"][0]),
           u_nom=float(np.abs(out["tensor"][2] - out["fp32"][2]).max()))
    assert abs(out["tensor"][0] - out["fp32"][0]) < 2e-5
    np.testing.assert_allclose(out["tensor"][2], out["fp32"][2], rtol=0, atol=2e-5)


def test_default_kernel_choice():
    """plain two-layer GRUs of up to 64 units -> tensor cores at every batch size (BASELINE.json configs[2]: K = 2000; the
    reference's shipped GRU-6IN-32H1-32H2-5OUT too); anything else -> FP32."""
    import torch
    for net, K, want in ((TC_NET, 2000, "tensor"), (TC_NET, 16, "tensor"), ("net_GRU_6IN_32H1_32H2_5OUT_0", 2000, "tensor"),
                         ("net_Dense_6IN_32H1_32H2_5OUT_0", 2000, "fp32"),
                         ("net_diff_GRU_6IN_64H1_64H2_5OUT_1", 2000, "fp32")):
        z, m = load_golden(net)
        eng = make_engine(net_spec_from_golden(z), K, 5)
        eng.net_rollout(torch.zeros(6, device=eng.device), torch.zeros((K, 5), device=eng.device))
        assert eng.net_last_kernel() == want, (net, K)


def test_tc_flag_rejected_for_other_networks():
    z, m = load_golden("net_Dense_6IN_32H1_32H2_5OUT_0")
    sp = net_spec_from_golden(z)
    import torch
    eng = make_engine(sp, 256, 10, net_kernel="tensor")
    with pytest.raises(NotImplementedError):
        eng.net_rollout(torch.zeros(6, device=eng.device), torch.zeros((256, 10), device=eng.device))


@pytest.mark.parametrize("run", ["gru32_grad", "gru32_qb"])
def test_tc_padded_gru32_mppi_vs_reference_golden(run):
    """the reference's shipped network size (GRU 2 x 32) on the tensor-core kernel (layers zero-padded to 64 units): the
    recorded solves of the unmodified optimizer_mppi + torch Sequence, as test_net_mppi_vs_reference_golden checks them on
    the FP32 kernel."""
    import torch
    from cartpolesimulation_b200 import _lib as L
    z, m = load_golden("mppi_net_" + run)
    sp = net_spec_from_golden(z)
    K, T = m["K"], m["T"]
    shifted = m["cost"] in ("default", "quadratic_boundary")
    eng = make_engine(sp, K, T, cost=m["cost"], net_kernel="tensor")
    eng.set_variable_parameters(m["target_position"], m["target_equilibrium"])
    dev = eng.device
    J = torch.empty(K, device=dev)
    u_nom = np.zeros(T, dtype=np.float32)
    h = np.zeros(sum(sp["hsz"]), np.float32)
    for i in range(m["steps"]):
        eng.set_u_nom(u_nom)
        eng.net_set_state(h)
        eps = torch.from_numpy(z["eps"][i]).to(dev)
        u = eng.mppi_step(torch.from_numpy(z["s"][i]).to(dev), eps, L.ROLLOUT_MAJOR, float(z["u_prev"][i]), None, J)
        torch.cuda.synchronize()
        assert eng.net_last_kernel() == "tensor"
        if shifted:
            assert shifted_cost_ok(J.cpu().numpy(), z["J"][i])
        else:
            assert vec_err(J.cpu().numpy(), z["J"][i]) < 1e-5
        eu = abs(float(u.cpu()[0]) - float(z["u"][i]))
        eh = float(np.abs(eng.net_get_state() - z["h_after"][i]).max())
        record("tc_padded_gru32_mppi", f"{run}/{i}", u=eu, u_nom=float(np.abs(eng.get_u_nom() - z["u_nom"][i]).max()), h=eh)
        assert eu < 1e-4      # north_star; measured <= 3.7e-5 (gru32_grad solve 2, whose control is the sensitive one on the FP32
        np.testing.assert_allclose(eng.get_u_nom(), z["u_nom"][i], rtol=0, atol=1e-4)   # kernel too: 9.1e-6 there)
        assert eh < max(5e-6, eu)   # the stored state is advanced on the selected control: its error carries the control's
        h = z["h_after"][i].copy()
        u_nom = z["u_nom"][i].copy()
    assert eng.nonfinite_costs() == 0


@pytest.mark.parametrize("hsz", [(32, 32), (48, 40), (16, 64), (64, 24), (8, 8)])
@pytest.mark.parametrize("K", [500, 6000, 12000])   # 32 / 64 / 128 live rollouts per CTA
def test_tc_padded_widths_match_fp32_kernel(hsz, K):
    """two-layer GRUs narrower than the tensor-core kernel's 64 units (zero-padded image; k-steps and half-layer jobs that hold
    only padding are skipped): same costs, control, nominal inputs and stored hidden state as the FP32 kernel, which
    tests/test_gpu_net_arch.py pins against the oracle for arbitrary widths."""
    import torch
    from cartpolesimulation_b200 import _lib as L
    from cartpolesimulation_b200.core import Engine
    from cartpolesimulation_b200.neural import synthetic_net_spec
    spec = synthetic_net_spec(hsz, "GRU", seed=sum(hsz))
    T = 12
    a = np.pi - 0.3
    s = torch.tensor([a, 0.2, np.cos(a), np.sin(a), 0.03, -0.1], dtype=torch.float32)
    rng = np.random.default_rng(K + hsz[0])
    out = {}
    for kern in ("fp32", "tensor"):
        eng = Engine(K, T, integrator="neural", cost="quadratic_boundary_grad_minimal", device=0, net_kernel=kern)
        eng.net_load(spec)
        if kern == "fp32":
            noise = torch.from_numpy(rng.standard_normal((eng.n_ind, K)).astype(np.float32)).to(eng.device)
            h0 = rng.uniform(-0.5, 0.5, sum(hsz)).astype(np.float32)
        eng.net_set_state(h0)
        J = torch.empty(K, device=eng.device)
        u = eng.mppi_step(s.to(eng.device), noise, L.TIME_MAJOR, 0.0, None, J)
        torch.cuda.synchronize()
        assert eng.net_last_kernel() == kern and eng.nonfinite_costs() == 0
        out[kern] = (float(u.cpu()[0]), J.cpu().numpy(), eng.get_u_nom(), eng.net_get_state())
        eng.close()
    t, f = out["tensor"], out["fp32"]
    eJ = vec_err(t[1], f[1])
    record("tc_padded_widths_vs_fp32", f"{hsz[0]}x{hsz[1]}_K{K}", J=eJ, u=abs(t[0] - f[0]))
    assert eJ < 2.5e-5    # measured <= 1.24e-5 (16 x 64, K = 500: rollouts on the boundary term's steep flank), else < 1e-5
    assert abs(t[0] - f[0]) < 1e-5
    np.testing.assert_allclose(t[2], f[2], rtol=0, atol=1e-5)
    np.testing.assert_allclose(t[3], f[3], rtol=0, atol=5e-6)
