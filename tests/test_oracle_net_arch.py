"""The references of the neural predictor pinned without a GPU on every architecture of the catalogue in tests/netutil.py
(layer counts 1 to 4, widths 1 to 128, mixed widths, Dense and GRU, permuted / partial / extended input-output layouts):
oracle/net_grad.predict against an independent float64 run of the reference's own modules (torch.nn.GRUCell /
torch.nn.Linear + tanh, the autoregressive loop of Predictors/autoregression.py:94-98, de-normalisation and augmentation
of predictors_customization.py:120-139), and against the C oracle's oracle.net_rollout; its autograd gradient against
central finite differences on the layouts whose angle routes differ from the shipped one."""
import numpy as np
import pytest

from tests.netutil import ARCHS, arch, atan2_layout
from tests.parity import record, traj_err
from tests.test_oracle_net_grad import fd_gradient_error

torch = pytest.importorskip("torch")

IDX = {"angle": 0, "angleD": 1, "angle_cos": 2, "angle_sin": 3, "position": 4, "positionD": 5}


def reference_modules_rollout(osp, s0, Q, h0):
    """float64 trajectories [B, T+1, 6] of the reference's torch modules on plans Q [B, T], s0 [B, 6], h0 [B, Htot]."""
    gru = osp["net_type"] == "GRU"
    mods, off, hs = [], 0, []
    n_in = len(osp["in_idx"]) + 1
    for lay, H in zip(osp["layers"], osp["hsz"]):
        if gru:
            m = torch.nn.GRUCell(n_in, H).double()
            m.weight_ih.data, m.weight_hh.data = (torch.from_numpy(a.astype(np.float64)) for a in lay[:2])
            m.bias_ih.data, m.bias_hh.data = (torch.from_numpy(a.astype(np.float64)) for a in lay[2:])
            hs.append(torch.from_numpy(h0[:, off:off + H].astype(np.float64)))
        else:
            m = torch.nn.Linear(n_in, H).double()
            m.weight.data, m.bias.data = (torch.from_numpy(a.astype(np.float64)) for a in lay)
        mods.append(m)
        off += H
        n_in = H
    out = torch.nn.Linear(n_in, len(osp["out_idx"])).double()
    out.weight.data, out.bias.data = (torch.from_numpy(a.astype(np.float64)) for a in osp["out_layer"])
    f64 = lambda a: torch.from_numpy(np.asarray(a, np.float64))
    na, nb, A, B = f64(osp["norm_a"]), f64(osp["norm_b"]), f64(osp["denorm_A"]), f64(osp["denorm_B"])
    s0, Qt = f64(s0), f64(Q)
    names = {v: k for k, v in IDX.items()}
    outs = [names[c] for c in osp["out_idx"]]
    x_state = na[1:] * s0[:, list(osp["in_idx"])] + nb[1:]
    states = [s0]
    with torch.no_grad():
        for t in range(Qt.shape[1]):
            x = torch.cat([(na[0] * Qt[:, t] + nb[0])[:, None], x_state], dim=1)
            for l, m in enumerate(mods):
                if gru:
                    hs[l] = m(x, hs[l])
                    x = hs[l]
                else:
                    x = torch.tanh(m(x))
            y = out(x)
            x_state = y[:, :len(osp["in_idx"])]   # the normalised output is the next normalised input
            v = {n: A[o] * y[:, o] + B[o] for o, n in enumerate(outs)}
            if "angle" not in v:
                v["angle"] = torch.atan2(v["angle_sin"], v["angle_cos"])
            v.setdefault("angle_sin", torch.sin(v["angle"]))
            v.setdefault("angle_cos", torch.cos(v["angle"]))
            st = torch.zeros_like(s0)
            for n, c in IDX.items():
                if n in v:
                    st[:, c] = v[n]
            states.append(st)
    return torch.stack(states, dim=1).numpy()


def _inputs(osp, B, T, seed):
    rng = np.random.default_rng(seed)
    ang = rng.uniform(-np.pi, np.pi, B)
    s0 = np.stack([ang, rng.uniform(-3, 3, B), np.cos(ang), np.sin(ang), rng.uniform(-0.15, 0.15, B),
                   rng.uniform(-0.5, 0.5, B)], 1).astype(np.float32)
    Q = rng.uniform(-1, 1, (B, T)).astype(np.float32)
    h0 = rng.uniform(-0.5, 0.5, (B, sum(osp["hsz"]))).astype(np.float32)
    return s0, Q, h0


@pytest.mark.parametrize("name", list(ARCHS))
def test_restatement_matches_reference_modules_and_c_oracle(name):
    from oracle import net_grad as NG
    from oracle import oracle as O
    _, osp = arch(name)
    B, T = 64, 40
    s0, Q, h0 = _inputs(osp, B, T, 7)
    ref = reference_modules_rollout(osp, s0, Q, h0)
    got = NG.predict(osp, s0, torch.from_numpy(Q.astype(np.float64)), h0).numpy()
    e_mod = traj_err(got, ref)
    # the C oracle (float32)
    c_traj = O.net_rollout(osp["net_type"], osp["hsz"], O.pack_net_weights(osp["net_type"], osp["layers"], osp["out_layer"]),
                           osp["in_idx"], osp["out_idx"], osp["norm_a"], osp["norm_b"], osp["denorm_A"], osp["denorm_B"],
                           s0, Q, h0=h0)
    e_c = traj_err(c_traj, got)
    norm = None
    if atan2_layout(osp):   # the catalogue keeps |(sin, cos)| near 1 (tests/netutil.arch_net): checked, not assumed
        norm = float(np.hypot(got[:, 1:, 2], got[:, 1:, 3]).min())
        assert 0.5 < norm < 1.5, norm
    record("net_arch_oracle_vs_reference_modules", name, modules=max(e_mod.values()), c_oracle=max(e_c.values()),
           sincos_norm_min=norm if norm is not None else -1.0)
    assert max(e_mod.values()) < 1e-12, e_mod
    assert max(e_c.values()) < 2e-6, e_c


@pytest.mark.parametrize("name", ["d_angle", "g_perm", "g_noin"])
@pytest.mark.parametrize("cost", ["quadratic_boundary_grad_minimal", "quadratic_boundary_grad"])
def test_autograd_gradient_matches_finite_differences(name, cost):
    _, osp = arch(name)
    a = 0.4
    s0 = np.array([a, 0.3, np.cos(a), np.sin(a), 0.02, -0.1], np.float32)
    h0 = np.random.default_rng(1).uniform(-0.3, 0.3, sum(osp["hsz"])) if osp["net_type"] == "GRU" else None
    e = fd_gradient_error(osp, cost, s0, h0)
    record("net_arch_oracle_vs_finite_differences", f"{name}/{cost}", G=e)
    assert e < 1e-6
