"""Accuracy of the headline integrator (predictor_ODE_v0: explicit Euler, rotation substeps) against an fp64
integration of the same scheme (oracle rollout_f64), as test_gpu_parity.test_fp32_noise_floor checks for predictor_ODE.

The fp32 yardstick differs from that test's: predictor_ODE_v0 integrates a control step in float64 and rounds to
float32 only at its end, so the reference's output (and the oracle's port of it) is closer to fp64 than any float32
integration can be -- the rotation kernels sit ~2e-6 .. 9e-6 from fp64 on the near-upright and random cases, the
reference 3e-7 .. 2.4e-6.  The yardstick here is the float32 realisation of the reference's formulas: the
substep_sincos kernel variant (sincosf every substep, the arithmetic of the reference text, no rotation).  The rotation
kernels must be no further from fp64 than it is (x2 + 3e-6 slack for a different realisation of the rounding noise).
Cases: the reference's recorded batches, and a sample of the benchmark's inputs (bench.make_inputs) at a batch size
that runs the packed two-cartpoles-per-thread kernel."""
import numpy as np
import pytest

from tests.parity import load_golden, record, traj_err

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def cuda(x):
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).cuda()


def _check(case, got, fp32, truth, ref=None):
    e_fp32 = traj_err(fp32, truth)
    e_got = traj_err(got, truth)
    e_ref = traj_err(ref, truth) if ref is not None else {}
    print("\nnoise floor ODE_v0", case, "substep_sincos-vs-fp64:", {k: f"{v:.1e}" for k, v in e_fp32.items()},
          "rotation-vs-fp64:", {k: f"{v:.1e}" for k, v in e_got.items()},
          "reference-vs-fp64:", {k: f"{v:.1e}" for k, v in e_ref.items()})
    record("rollout_v0_noise_floor", case, substep_sincos=e_fp32, rotation=e_got, reference=e_ref)
    for ch in e_fp32:
        assert e_got[ch] <= 2.0 * e_fp32[ch] + 3e-6, (ch, e_got, e_fp32)


def _rollout(B, T, s0, Q, n=10, dt=0.02, var=None, **kw):
    from cartpolesimulation_b200.core import Engine
    eng = Engine(B, T, dt=dt, substeps=n, integrator="ODE_v0", cost=None, **kw)
    if var is not None:
        eng.set_variable_parameters(L=var[0], m_pole=var[1])
    got, _ = eng.rollout(cuda(s0), cuda(Q))
    return got.cpu().numpy(), eng


@pytest.mark.parametrize("case", ["tiled", "upright", "random"])
def test_rollout_v0_noise_floor_golden(case):
    from oracle import oracle as O
    z, meta = load_golden("rollout_ode_v0")
    s0, Q, ref = z[f"{case}__s0"], z[f"{case}__Q"], z[f"{case}__traj"]
    Lv, m_pole, n = z[f"{case}__var"]
    B, T = Q.shape
    s_in = s0[0] if s0.shape[0] == 1 else s0
    truth = O.rollout_f64("ODE_v0", s0, Q, n=int(n), dt=meta["dt"], L=Lv)
    got, _ = _rollout(B, T, s_in, Q, int(n), meta["dt"], (Lv, m_pole))
    fp32, _ = _rollout(B, T, s_in, Q, int(n), meta["dt"], (Lv, m_pole), substep_sincos=True)
    _check(case, got, fp32, truth, ref)


def test_rollout_v0_noise_floor_bench_inputs():
    import bench
    from cartpolesimulation_b200 import _lib as L
    from cartpolesimulation_b200.core import Engine
    from oracle import oracle as O
    B, T, n = L.PAIR_MIN_BATCH, 50, 10
    s0, Q = bench.make_inputs(B, T, seed=7)                 # Q time-major [T, B]
    eng = Engine(B, T, integrator="ODE_v0", cost=None)
    traj, _ = eng.rollout(cuda(s0), cuda(Q), q_layout=L.TIME_MAJOR, traj_layout=L.TIME_MAJOR)
    assert eng.rollout_last_kernel() == "rollout_pair_kernel"
    idx = np.sort(np.random.default_rng(7).choice(B, n, replace=False))
    got = np.transpose(traj[:, :, torch.from_numpy(idx).cuda()].cpu().numpy(), (2, 0, 1))   # [n, T+1, 6]
    Qs = np.ascontiguousarray(Q[:, idx].T)
    truth = O.rollout_f64("ODE_v0", s0[idx], Qs)
    fp32, _ = _rollout(n, T, s0[idx], Qs, substep_sincos=True)
    _check("bench_inputs", got, fp32, truth, O.rollout("ODE_v0", s0[idx], Qs))
