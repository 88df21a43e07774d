"""Builds the flat network description (cps_net_load / cps_oracle_net_rollout arguments) from a net golden file.

Follows the reference's bookkeeping: SI_Toolkit/src/SI_Toolkit/Predictors/predictor_autoregressive_neural.py:163-199
(input/output index maps), Functions/General/Normalising.py:15-108 (minmax_sym coefficients, computed in float32 as
the torch library does)."""
import json

import numpy as np

STATE_VARIABLES = ["angle", "angleD", "angle_cos", "angle_sin", "position", "positionD"]


def minmax_sym_coeffs(table, cols, names):
    """(a, b, A, B) float32 vectors for `names`; table rows: mean, std, max, min (Normalising.py:1-9)."""
    t = np.asarray(table, dtype=np.float32)
    idx = [list(cols).index(n) for n in names]
    mx, mn = t[2, idx], t[3, idx]
    a = np.float32(2.0) / (mx - mn)
    b = np.float32(-1.0) + np.float32(2.0) * (-mn / (mx - mn))
    A = (mx - mn) / np.float32(2.0)
    B = (mx - mn) / np.float32(2.0) + mn
    return a.astype(np.float32), b.astype(np.float32), A.astype(np.float32), B.astype(np.float32)


def net_spec_from_golden(z):
    meta = json.loads(str(z["meta"]))
    inputs, outputs, ntype = meta["inputs"], meta["outputs"], meta["type"]
    keys = [str(k) for k in z["state_dict_keys"]]
    n_lay = max(int(k.split(".")[1]) for k in keys)  # index of the output layer
    layers, hsz = [], []
    for l in range(n_lay):
        if ntype == "GRU":
            lay = tuple(z[f"w__layers.{l}.{n}"] for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"))
            hsz.append(lay[1].shape[1])
        else:
            lay = (z[f"w__layers.{l}.weight"], z[f"w__layers.{l}.bias"])
            hsz.append(lay[0].shape[0])
        layers.append(lay)
    out_layer = (z[f"w__layers.{n_lay}.weight"], z[f"w__layers.{n_lay}.bias"])
    cols = [str(c) for c in z["norm_cols"]]
    a, b, _, _ = minmax_sym_coeffs(z["norm_table"], cols, inputs)
    # differential networks (outputs D_*): the integrated variables carry the output names without the prefix
    # (predictor_autoregressive_neural.py:184-190)
    out_names = [(o[2:] if o[:2] == "D_" else o) for o in outputs]
    _, _, A, B = minmax_sym_coeffs(z["norm_table"], cols, out_names)
    diff = None
    if any("D_" in o for o in outputs):
        # Normalising.py:111-186: p1 = a * C * dt, p2 = a * D * dt with a of the integrated variables and C, D of the
        # derivatives; autoregression.py:137-146: state -> output and output -> input index maps
        on_a, on_b, _, _ = minmax_sym_coeffs(z["norm_table"], cols, out_names)
        _, _, Cd, Dd = minmax_sym_coeffs(z["norm_table"], cols, outputs)
        dt = np.float32(meta["dt"])
        diff = dict(p1=(on_a * Cd * dt).astype(np.float32), p2=(on_a * Dd * dt).astype(np.float32), on_a=on_a, on_b=on_b,
                    out_to_in=[out_names.index(n) for n in inputs[1:]])
    return dict(net_type=ntype, hsz=hsz, layers=layers, out_layer=out_layer,
                in_idx=[STATE_VARIABLES.index(n) for n in inputs[1:]],
                out_idx=[STATE_VARIABLES.index(n) for n in out_names],
                norm_a=a, norm_b=b, denorm_A=A, denorm_B=B, diff=diff, meta=meta)


def write_model_dir(root, z):
    """Writes <root>/<net full name>/{<name>.txt, ckpt.pt, NI.csv} from a net golden file, in the reference's formats
    (Functions/General/Initialization.py:35-104; torch state_dict of Functions/Pytorch/Network.py Sequence).
    Returns the model path to use as `predictor_specification` / `model_name`."""
    import os
    import torch
    meta = json.loads(str(z["meta"]))
    full = meta["net"]
    d = os.path.join(root, full)
    os.makedirs(d, exist_ok=True)
    short = "-".join(p for p in full.split("-") if not (p.endswith("IN") or p.endswith("OUT")))[:-2]
    cols = [str(c) for c in z["norm_cols"]]
    ni = os.path.join(d, "NI.csv")
    with open(ni, "w") as f:
        f.write("," + ",".join(cols) + "\n")
        for r, rowname in enumerate(["mean", "std", "max", "min"]):
            f.write(rowname + "," + ",".join(repr(float(z["norm_table"][r, c])) for c in range(len(cols))) + "\n")
    with open(os.path.join(d, full + ".txt"), "w") as f:
        f.write("\n".join([
            "CREATED:", "2026-01-01 00:00:00", "", "LIBRARY:", "Pytorch", "", "NET NAME:", short, "",
            "NET FULL NAME:", full, "", "INPUTS:", ", ".join(meta["inputs"]), "", "OUTPUTS:", ", ".join(meta["outputs"]),
            "", "TYPE:", meta["type"], "", "NORMALIZATION:", ni, "", "NORMALIZE:", "True", "",
            "WASH OUT LENGTH:", "10", "", "CONSTRUCT NETWORK:", "with cells", ""]))
    sd = {str(k): torch.from_numpy(np.array(z["w__" + str(k)])) for k in z["state_dict_keys"]}
    torch.save(sd, os.path.join(d, "ckpt.pt"))
    return os.path.join(root, full)


# ---- networks of any architecture the loader accepts -------------------------------------------------------------
SHIPPED_IN = ["Q", "angleD", "angle_cos", "angle_sin", "position", "positionD"]
SHIPPED_OUT = SHIPPED_IN[1:]
ANGLE_IN, ANGLE_OUT = ["Q", "angle", "angleD", "position", "positionD"], ["angle", "angleD", "position", "positionD"]
PERM_IN = ["Q", "position", "angle_sin", "angleD", "angle_cos", "positionD"]
PERM_OUT = PERM_IN[1:] + ["angle"]
EXTRA_IN, EXTRA_OUT = ["Q", "angle_cos", "angle_sin"], ["angle_cos", "angle_sin", "angleD", "position", "positionD"]
NOIN_IN, NOIN_OUT = ["Q"], ["angle", "angleD", "position", "positionD"]

# id: (type, hidden sizes, inputs, outputs) -- one line per kernel branch the entry exists for
ARCHS = {
    "g_mixed": ("GRU", (48, 40), SHIPPED_IN, SHIPPED_OUT),        # HT = 0, 2 layers; tensor-core eligible
    "g_3x32": ("GRU", (32, 32, 32), SHIPPED_IN, SHIPPED_OUT),     # HT = 32 with 3 layers
    "g_1x64": ("GRU", (64,), SHIPPED_IN, SHIPPED_OUT),            # HT = 64 with 1 layer
    "g_4deep": ("GRU", (16, 24, 8, 40), SHIPPED_IN, SHIPPED_OUT),  # HT = 0, 4 layers (hoff of layers 2, 3)
    "g_wide": ("GRU", (96,), SHIPPED_IN, SHIPPED_OUT),            # H0 > 64: layer 0 without the split; gradient at R = 32
    "d_128": ("Dense", (128, 128), SHIPPED_IN, SHIPPED_OUT),      # widest Dense; gradient falls back to R = 16 at large K
    "d_odd": ("Dense", (7,), SHIPPED_IN, SHIPPED_OUT),            # 1 layer of odd width (out_layer_row's two lane halves)
    "d_angle": ("Dense", (24, 24, 24), ANGLE_IN, ANGLE_OUT),      # `angle` output: sin / cos rebuilt by sinf / cosf
    "g_perm": ("GRU", (33, 31), PERM_IN, PERM_OUT),               # permuted in_idx / out_idx; angle, sin and cos all output
    "g_extra": ("GRU", (1, 5), EXTRA_IN, EXTRA_OUT),              # H = 1; n_state_in < n_out (outputs not fed back)
    "g_noin": ("GRU", (20, 12), NOIN_IN, NOIN_OUT),               # n_state_in = 0 (n_in = 1)
    "tc_angle": ("GRU", (64, 64), ANGLE_IN, ANGLE_OUT),           # tensor cores: n_in = 5, `angle` output
    "tc_perm": ("GRU", (40, 56), PERM_IN, PERM_OUT),              # tensor cores: permuted indices, n_out = 6
    "tc_extra": ("GRU", (32, 32), EXTRA_IN, EXTRA_OUT),           # tensor cores (narrow image): n_state_in < n_out
    "tc_noin": ("GRU", (24, 16), NOIN_IN, NOIN_OUT),              # tensor cores (narrow image): n_in = 1
}


def arch_norm(outputs=()):
    """(columns, table) normalisation of the reference's shipped ranges (neural.DEFAULT_RANGES), plus symmetric ranges
    of the D_* columns a differential network's outputs name (those of the reference's differential recordings)."""
    from cartpolesimulation_b200.neural import DEFAULT_RANGES
    rng = dict(DEFAULT_RANGES)
    d_ranges = {"D_angle": 18.38, "D_angleD": 90.0, "D_angle_cos": 15.0, "D_angle_sin": 15.0, "D_position": 1.125,
                "D_positionD": 9.0}
    for o in outputs:
        if o.startswith("D_"):
            rng[o] = (d_ranges[o], -d_ranges[o])
    cols = list(rng)
    table = np.array([[0.0] * len(cols), [1.0] * len(cols), [rng[c][0] for c in cols], [rng[c][1] for c in cols]])
    return cols, table


def arch_net(net_type, hsz, inputs, outputs, seed, dt=None):
    """(engine spec, oracle spec) of one randomly initialised network.

    Weights as torch initialises GRUCell / Linear, U(-1/sqrt(H), 1/sqrt(H)) with H the layer's width (the input width for
    the output layer).  A layout that rebuilds the angle as atan2(sin, cos) gets output rows for angle_cos / angle_sin
    with the bias (cos phi, sin phi) and weights scaled by 0.1, so that |(sin, cos)| stays near 1: an untrained network
    would put it near 0, where atan2 amplifies any rounding without bound and hides the kernels' own error.
    The engine spec comes from the product's neural.build_net_spec; the oracle spec holds the same weights unpacked into
    layers / out_layer tuples (oracle/net_grad.py, oracle.net_rollout)."""
    from cartpolesimulation_b200.neural import build_net_spec
    rng = np.random.default_rng(seed)
    gru = net_type == "GRU"
    G = 3 if gru else 1
    layers, n_in = [], len(inputs)
    u = lambda k, shape: rng.uniform(-k, k, shape).astype(np.float32)
    for H in hsz:
        k = 1.0 / np.sqrt(H)
        layers.append((u(k, (G * H, n_in)), u(k, (G * H, H)), u(k, G * H), u(k, G * H)) if gru else
                      (u(k, (H, n_in)), u(k, H)))
        n_in = H
    k = 1.0 / np.sqrt(n_in)
    w_out, b_out = u(k, (len(outputs), n_in)), u(k, len(outputs))
    norm = arch_norm(outputs)
    spec = build_net_spec(net_type, inputs, outputs, list(hsz), np.zeros(1), norm, dt)
    names = [(o[2:] if o[:2] == "D_" else o) for o in outputs]
    if "angle" not in names and "angle_cos" in names and "angle_sin" in names and not spec["differential"]:
        phi = rng.uniform(-np.pi, np.pi)
        A, B = spec["denorm_A"], spec["denorm_B"]
        for name, v in (("angle_cos", np.cos(phi)), ("angle_sin", np.sin(phi))):
            o = names.index(name)
            w_out[o] *= np.float32(0.1)
            b_out[o] = np.float32((v - B[o]) / A[o])
    from oracle import oracle as O
    spec["weights"] = O.pack_net_weights(net_type, layers, (w_out, b_out))
    diff = None
    if spec["differential"]:
        diff = dict(p1=spec["diff_p1"], p2=spec["diff_p2"], on_a=spec["out_norm_a"], on_b=spec["out_norm_b"],
                    out_to_in=spec["out_to_in"])
    osp = dict(net_type=net_type, hsz=list(hsz), layers=layers, out_layer=(w_out, b_out), in_idx=spec["in_idx"],
               out_idx=spec["out_idx"], norm_a=spec["norm_a"], norm_b=spec["norm_b"], denorm_A=spec["denorm_A"],
               denorm_B=spec["denorm_B"], diff=diff)
    return spec, osp


def arch(name, seed=None):
    """arch_net of a catalogue entry (seed: the entry's position, unless given)."""
    t, hsz, i, o = ARCHS[name]
    return arch_net(t, hsz, i, o, list(ARCHS).index(name) if seed is None else seed)


def atan2_layout(osp):
    """Whether the network's layout rebuilds the angle as atan2(sin, cos) (no `angle` output, both sin and cos)."""
    out = set(osp["out_idx"])
    return 0 not in out and 2 in out and 3 in out
