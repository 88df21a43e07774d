"""Torch restatement of predict_and_cost with the autoregressive neural predictor and the two gradient cost plugins, and
its gradient by torch autograd -- the gradient oracle of cps_plan_cost_grad for CPS_PREDICTOR_NEURAL.

What it restates (plain networks; differential D_* networks are not covered):
  predictor_autoregressive_neural._predict_core (SI_Toolkit/Predictors/predictor_autoregressive_neural.py:266-313): the torch
    Sequence's GRUCell / tanh Linear stack and linear output layer (Functions/Pytorch/Network.py:239-287), the normalised
    output fed back as the next normalised input (Predictors/autoregression.py:94-98), de-normalisation, the scatter into
    the 6-vector state and the angle augmentation (predictors_customization.py:120-139);
  quadratic_boundary_grad_minimal / quadratic_boundary_grad stage costs, written as oracle.plan_cost_grad writes them (the
    kinetic term's target under stop_gradient), mean over the T + 1 entries (terminal cost zero).
Driven by a tests.netutil.net_spec_from_golden spec.  Test infrastructure: the package does not import it."""
from __future__ import annotations

import numpy as np
import torch

from . import oracle as O

IDX_ANGLE, IDX_ANGLED, IDX_COS, IDX_SIN, IDX_POS = 0, 1, 2, 3, 4


def _t(a, dtype, device=None):
    if isinstance(a, torch.Tensor):
        return a.to(dtype=dtype, device=device)
    return torch.as_tensor(np.asarray(a), dtype=dtype, device=device)


def predict(spec, s0, Q, h0=None, dtype=torch.float64):
    """Trajectories [K, T+1, 6] of the network on plans Q [K, T] (tensor; may require grad) from s0 ([6] or [K, 6]) and
    the initial hidden state h0 ([Htot] shared or [K, Htot], concatenated over the layers; None = zeros).  Runs on Q's
    device."""
    K, T = Q.shape
    dev = Q.device
    s0 = _t(s0, dtype, dev)
    s0 = s0.reshape(1, 6).expand(K, 6) if s0.numel() == 6 else s0.reshape(K, 6)
    gru = spec["net_type"] == "GRU"
    layers = [tuple(_t(a, dtype, dev) for a in lay) for lay in spec["layers"]]
    Wo, bo = (_t(a, dtype, dev) for a in spec["out_layer"])
    na, nb = _t(spec["norm_a"], dtype, dev), _t(spec["norm_b"], dtype, dev)
    A, B = _t(spec["denorm_A"], dtype, dev), _t(spec["denorm_B"], dtype, dev)
    in_idx, out_idx = list(spec["in_idx"]), list(spec["out_idx"])
    ns = len(in_idx)
    h = []
    if gru:
        Ht = int(sum(spec["hsz"]))
        hv = torch.zeros(Ht, dtype=dtype, device=dev) if h0 is None else _t(h0, dtype, dev)
        hv = hv.reshape(-1, Ht).expand(K, Ht)
        off = 0
        for H in spec["hsz"]:
            h.append(hv[:, off:off + H])
            off += H
    has = set(out_idx)

    def compose(y):
        v = A * y + B
        cols = [torch.zeros(K, dtype=dtype, device=dev) for _ in range(6)]
        for o, c in enumerate(out_idx):
            cols[c] = v[:, o]
        if IDX_ANGLE not in has and IDX_SIN in has and IDX_COS in has:
            cols[IDX_ANGLE] = torch.atan2(cols[IDX_SIN], cols[IDX_COS])
        if IDX_ANGLE in has and IDX_SIN not in has:
            cols[IDX_SIN] = torch.sin(cols[IDX_ANGLE])
        if IDX_ANGLE in has and IDX_COS not in has:
            cols[IDX_COS] = torch.cos(cols[IDX_ANGLE])
        return torch.stack(cols, dim=1)

    feat = na[1:] * s0[:, in_idx] + nb[1:]
    states = [s0]
    for t in range(T):
        x = torch.cat([(na[0] * Q[:, t] + nb[0]).reshape(K, 1), feat], dim=1)
        for l, lay in enumerate(layers):
            if gru:
                w_ih, w_hh, b_ih, b_hh = lay
                gi, gh = x @ w_ih.T + b_ih, h[l] @ w_hh.T + b_hh
                H = w_hh.shape[1]
                r = torch.sigmoid(gi[:, :H] + gh[:, :H])
                z = torch.sigmoid(gi[:, H:2 * H] + gh[:, H:2 * H])
                n = torch.tanh(gi[:, 2 * H:] + r * gh[:, 2 * H:])
                h[l] = (1.0 - z) * n + z * h[l]
                x = h[l]
            else:
                x = torch.tanh(x @ lay[0].T + lay[1])
        y = x @ Wo.T + bo
        feat = y[:, :ns]
        states.append(compose(y))
    return torch.stack(states, dim=1)


def stage_costs(cost_name, traj, Q, u_prev=0.0, target_position=0.0, target_equilibrium=1.0, cost_cfg=None, thl=None):
    """[K, T] stage costs of the gradient plugins on traj [K, T+1, 6] (rows 0..T-1) -- oracle.plan_cost_grad's `stage`."""
    if cost_name not in ("quadratic_boundary_grad_minimal", "quadratic_boundary_grad"):
        raise NotImplementedError("restated for quadratic_boundary_grad_minimal and quadratic_boundary_grad only")
    full = cost_name == "quadratic_boundary_grad"
    cfg = dict(O.DEFAULT_COST_CONFIG[cost_name]) if cost_cfg is None else cost_cfg
    thl = float(O.physics_vector()[8]) if thl is None else float(thl)
    tp, te = float(target_position), float(target_equilibrium)
    sfx = "_up" if (not full or te == 1.0) else "_down"
    w_dd, w_db, w_ep, w_ekp = (cfg[k + sfx] for k in ("dd_quadratic_weight", "db_weight", "ep_weight", "ekp_weight"))
    w_cc, pf = cfg["cc_weight" + sfx] * cfg["R"], cfg["permissible_track_fraction"]
    th, w, x = traj[:, :-1, IDX_ANGLE], traj[:, :-1, IDX_ANGLED], traj[:, :-1, IDX_POS]
    up = torch.cat([torch.full_like(Q[:, :1], float(u_prev)), Q[:, :-1]], dim=1)
    dist = (x - tp) / (2 * thl)
    over = torch.where(torch.abs(x) > pf * thl, (torch.abs(x) - pf * thl) / ((1 - pf) * thl), torch.zeros_like(x))
    if not full:
        return w_dd * dist ** 2 + w_db * over ** 2 + w_ep * (1 - te * torch.cos(th)) ** 2 + w_ekp * w ** 2 + w_cc * Q ** 2
    w_lin, w_ccrc = cfg["dd_linear_weight" + sfx], cfg["ccrc_weight" + sfx]
    tmax = abs(120.0 * (1.0 + te) / 2.0 + cfg["target_angular_speed_sqr_max_correction" + sfx])
    cos_adm = np.cos(np.pi * cfg["admissible_angle"] / 180.0)
    ca = torch.cos(th).detach()   # _E_kin_cost's target carries no gradient (stop_gradient)
    scaling = torch.where(te * (ca - cos_adm) > 0, torch.zeros_like(ca), (1.0 - te * ca) / 2.0)
    return (w_dd * dist ** 2 + w_lin * torch.abs(dist) + w_db * over ** 2 + w_ep * ((2 - te * torch.cos(th)) ** 2 - 1)
            + w_ekp * torch.abs(w * w - tmax * scaling) + w_cc * Q ** 2 + w_ccrc * (Q - up) ** 2)


def plan_cost(spec, cost_name, s, Q, u_prev=0.0, target_position=0.0, target_equilibrium=1.0, cost_cfg=None, h0=None,
              dtype=torch.float64):
    """J [K] (tensor) of predict_and_cost; Q a [K, T] tensor."""
    traj = predict(spec, s, Q, h0, dtype)
    st = stage_costs(cost_name, traj, Q, u_prev, target_position, target_equilibrium, cost_cfg)
    return st.sum(dim=1) / (Q.shape[1] + 1)


def plan_cost_grad(spec, cost_name, s, Q, u_prev=0.0, target_position=0.0, target_equilibrium=1.0, cost_cfg=None, h0=None,
                   dtype=torch.float64):
    """(J [K], dJ/dQ [K, T]) as numpy arrays, by torch autograd through the restatement (the plans are independent, so
    the gradient of the sum is every plan's own gradient)."""
    Qt = _t(Q, dtype).reshape(np.asarray(Q).shape[0], -1).clone().requires_grad_(True)
    J = plan_cost(spec, cost_name, s, Qt, u_prev, target_position, target_equilibrium, cost_cfg, h0, dtype)
    (G,) = torch.autograd.grad(J.sum(), Qt)
    return J.detach().numpy(), G.numpy()
