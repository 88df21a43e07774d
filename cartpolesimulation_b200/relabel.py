"""Offline relabelling on the GPU: add_control_along_trajectories for many recorded files at once
(SURVEY.md 8f row f4).

Mirror of SI_Toolkit/src/SI_Toolkit/General/preprocess_data_add_control_along_trajectories.py:53-140 with MPPI as the
controller: for every row of a recording the controller is stepped from the RECORDED state with the row's environment
attributes (target_position, target_equilibrium, L, ...); rows of one file are sequential (the optimizer keeps its
warm start and last control), files are independent.  The reference processes one file per process (a 120-way SLURM
array, others/EulerClusterScripts/ControllerAlongTrajectories.sh:2-17); here E files advance in lockstep, one
fleet_kernel launch per row of all files (cps_fleet_relabel), nothing returning to the host in between.

Attribute-name conventions of the reference are kept (:166-263): `<col>_random_uniform_<lo>_<hi>[_<step>]` draws the
attribute per row, `<col>_integrate_<lo>_<hi>_` averages the control over a scrambled-Sobol sample of the attribute
(`integration_num_evals` consecutive controller steps per row, :318-345), `<col>_differentiate_` labels the derivative of
the control with respect to the attribute (five controller steps per row and feature at value + {-2..2} * 0.5e-3, then a
Savitzky-Golay first derivative, :348-470).  integration_method='nquad' (:346-362, the reference's default): the
quadrature is adaptive -- the next query point depends on the controller's answers, and every answer advances the
controller's warm start -- so it cannot be laid out as a fixed table of rows.  Here scipy's own `nquad` (QUADPACK, as in
the reference) drives every file on a host thread of its own, and the integrand evaluations of all files are collected
into lockstep rounds: one masked fleet launch (cps_fleet_relabel_masked) evaluates the pending query of every file that
still has one, files that are done with the row sit the launch out.  method='nd' is not offered.  No CPU fallback.

RPGD, the reference's default optimizer, relabels the same way (Relabeller(optimizer="rpgd"), controller_config["rpgd"]):
one RpgdFleet controller period per row of all files with the plant replaced by the recording (cps_rpgd_fleet_relabel).
Plain rows, `_random_uniform_`, Monte-Carlo `_integrate_` and `_differentiate_` are sequences of rows.  `nquad` is not
offered under RPGD: files sitting rows out would need their own solve counter, Adam iteration count and number of Adam
steps, and the RPGD fleet advances those in lockstep.
"""
from __future__ import annotations

import re
import threading
from math import ceil

import numpy as np
import torch

from . import config as cfgmod
from .fleet import Fleet, RpgdFleet

STATE_COMPONENTS = ("angle", "angleD", "angle_cos", "angle_sin", "position", "positionD")  # CartPole/state_utilities.py
_CONTROLLER_ATTRIBUTES = ("target_position", "target_equilibrium", "L", "m_pole")


class Relabeller:
    """E files in lockstep on one device: a Fleet (MPPI) used in replay mode (the plant is not integrated).

    optimizer="rpgd": an RpgdFleet instead, built from RpgdFleet's keywords (num_rollouts, mpc_horizon, outer_its,
    resamp_per, period_interpolation_inducing_points, ..., integrator="neural" with network=spec); dt, substeps,
    integrator, cost, cost_config, device, noise, seed and file_offset keep their meaning.  horizon, interp_period, mppi and
    no_pairs are MPPI's and raise ValueError there."""

    def __init__(self, n_files: int, num_rollouts: int | None = None, horizon: int | None = None, dt: float = 0.02,
                 substeps: int = 10, integrator: str = "ODE", cost: str = "quadratic_boundary_grad_minimal",
                 interp_period: int | None = None, device: int | None = None, noise: str = "philox", seed: int = 0,
                 file_offset: int = 0, cost_config: dict | None = None, mppi: dict | None = None, no_pairs: bool = False,
                 optimizer: str = "mppi", **rpgd):
        if optimizer not in ("mppi", "rpgd"):
            raise ValueError(f"optimizer must be 'mppi' or 'rpgd', got {optimizer!r}")
        self.optimizer = optimizer
        if optimizer == "rpgd":
            given = [k for k, v in (("horizon", horizon), ("interp_period", interp_period), ("mppi", mppi)) if v is not None]
            if no_pairs:
                given.append("no_pairs")
            if given:
                raise ValueError(f"{given} are MPPI keywords; RPGD takes mpc_horizon / period_interpolation_inducing_points")
            if num_rollouts is not None:
                rpgd["num_rollouts"] = num_rollouts
            self.fleet = RpgdFleet(n_files, dt=dt, substeps=substeps, integrator=integrator, cost=cost,
                                   cost_config=cost_config, device=device, noise=noise, seed=seed,
                                   experiment_offset=file_offset, **rpgd)
        else:
            if rpgd:
                raise TypeError(f"unexpected keyword arguments {sorted(rpgd)} (RPGD keywords need optimizer='rpgd')")
            self.fleet = Fleet(n_files, 2000 if num_rollouts is None else num_rollouts, 50 if horizon is None else horizon,
                               dt=dt, substeps=substeps, integrator=integrator, cost=cost,
                               interp_period=10 if interp_period is None else interp_period, device=device, noise=noise,
                               seed=seed, experiment_offset=file_offset, no_pairs=no_pairs)
        self.engine = self.fleet.engine
        self.E, self.K, self.T, self.n_ind, self.device = n_files, self.fleet.K, self.fleet.T, self.fleet.n_ind, self.fleet.device
        if optimizer == "mppi":
            if cost_config is not None:
                self.engine.set_cost_params(cfgmod.cost_vector(cost, cost_config))
            if mppi:
                self.engine.set_mppi_params(**mppi)

    def close(self):
        self.fleet.close()

    def reset(self, period: int = 0, init_draws=None):
        """controller.reset() of every file (:109-110).  RPGD: init_draws as RpgdFleet.reset takes them ('supplied'
        fleets: cuda tensor [E, K, n_ind]; a 'philox' fleet draws its own)."""
        if self.optimizer == "rpgd":
            self.fleet.reset(np.zeros((self.E, 6), dtype=np.float32), period, init_draws=init_draws)
            return
        if init_draws is not None:
            raise ValueError("init_draws are RPGD's; an MPPI relabeller starts from a zero warm start")
        self.engine.use_current_stream()
        self.engine._chk(self.engine.lib.cps_fleet_reset(self.engine._h, int(period)))

    def relabel_device(self, states, target_position=None, target_equilibrium=None, pole_length=None, m_pole=None,
                       noise=None, Q_out=None, J_out=None, active=None):
        """Fleet.relabel on cuda tensors: states [R, E, 6]; attributes [R, E] or None; noise [R, E, n_ind, K] for a
        'supplied' fleet; active [R, E] int32 or None: files with 0 sit the row out (cps_fleet_relabel_masked).
        RPGD: RpgdFleet.relabel, noise = the resampling draws [R, E, K - opt_keep_k, n_ind] of a 'supplied' fleet;
        no `active`.  Returns Q_out [R, E] (no synchronisation)."""
        return self.fleet.relabel(states, target_position, target_equilibrium, pole_length, m_pole, noise, Q_out, J_out, active)

    def relabel(self, states, target_position=None, target_equilibrium=None, pole_length=None, m_pole=None, noise=None,
                chunk_rows: int = 4096) -> np.ndarray:
        """Host form: numpy [R, E, 6] / [R, E] in, numpy controls [R, E] out.  Rows are fed in chunks; each chunk is
        chunk_rows launches queued back to back."""
        states = np.ascontiguousarray(states, dtype=np.float32)
        R = states.shape[0]
        out = np.empty((R, self.E), dtype=np.float32)

        def dev(a, lo, hi):
            if a is None:
                return None
            return torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=np.float32)[lo:hi])).to(self.device)

        for lo in range(0, R, chunk_rows):
            hi = min(R, lo + chunk_rows)
            nz = None
            if noise is not None:
                nz = noise[lo:hi] if isinstance(noise, torch.Tensor) else dev(noise, lo, hi)
            q = self.relabel_device(dev(states, lo, hi), dev(target_position, lo, hi), dev(target_equilibrium, lo, hi),
                                    dev(pole_length, lo, hi), dev(m_pole, lo, hi), nz)
            out[lo:hi] = q.cpu().numpy()
        return out


# ---- the reference's attribute-name conventions ---------------------------------------------------------------------------
_RANDOM = re.compile(r'^(.+)_random_uniform_([-+]?\d*\.?\d+)_([-+]?\d*\.?\d+)(?:_([-+]?\d*\.?\d+))?_?$')
_INTEGRATE = re.compile(r'^(.+)_integrate_([-+]?\d*\.?\d+)_([-+]?\d*\.?\d+)_?$')
_DIFFERENTIATE = re.compile(r'^(.+)_differentiate_$')


def process_random_sampling(df, environment_attributes_dict, rng=None):
    """:166-223.  `rng`: numpy Generator (the reference uses the global numpy state)."""
    rng = rng or np.random.default_rng()
    env = dict(environment_attributes_dict)
    for key, value in env.items():
        m = _RANDOM.match(value)
        if not m:
            continue
        lo, hi = float(m.group(2)), float(m.group(3))
        new = f"{m.group(1)}_random_uniform"
        if m.group(4) is not None:
            step = float(m.group(4))
            if step <= 0:
                raise ValueError(f"Step value must be positive in feature name: {value}")
            df[new] = rng.choice(np.arange(lo, hi + step / 10, step), len(df), replace=True)
        else:
            df[new] = rng.uniform(lo, hi, len(df))
        env[key] = new
    return df, env


def get_integration_features(environment_attributes_dict):
    """:226-263: (features, {feature: (lo, hi)}, attribute dict with the plain column names)."""
    env = dict(environment_attributes_dict)
    features, ranges = [], {}
    for key, value in env.items():
        m = _INTEGRATE.match(value)
        if m:
            features.append(m.group(1))
            ranges[m.group(1)] = (float(m.group(2)), float(m.group(3)))
            env[key] = m.group(1)
    return features, ranges, env


def get_differentiation_features(environment_attributes_dict, output_variable_names):
    """:266-300: (features, attribute dict with plain column names, output column names)."""
    env = dict(environment_attributes_dict)
    features = []
    for key, value in env.items():
        m = _DIFFERENTIATE.match(value)
        if m:
            features.append(m.group(1))
            env[key] = m.group(1)
    if features:
        names = [f"{o}_d{f}" for o in output_variable_names for f in features] \
            + [f"{o[1:]}_d{f}" for o in output_variable_names for f in features]   # the reference's naming (:289-296)
    else:
        names = list(output_variable_names)
    return features, env, names


DIFF_STEP, DIFF_WINDOW, DIFF_POLYORDER = 0.5e-3, 5, 1   # differentiation() defaults (:352-354,:370-373)


def sobol_samples(features, ranges, num_evals, n_rows, seed=None):
    """The Monte-Carlo sample of :318-337: per row a freshly scrambled Sobol sequence of 2^ceil(log2 N) points scaled
    to the feature ranges.  Returns [n_rows, N, d]."""
    from scipy.stats import qmc
    d = len(features)
    m = int(np.log2(num_evals))
    if 2 ** m != num_evals:
        m = int(np.ceil(np.log2(num_evals)))
    lo = np.array([ranges[f][0] for f in features])
    span = np.array([ranges[f][1] - ranges[f][0] for f in features])
    ss = np.random.SeedSequence(seed)
    out = np.empty((n_rows, 2 ** m, d))
    for r, child in enumerate(ss.spawn(n_rows)):
        out[r] = lo + qmc.Sobol(d=d, scramble=True, seed=np.random.default_rng(child)).random_base2(m=m) * span
    return out


class _Lockstep:
    """Rendezvous between the per-file quadrature threads and the launching thread: workers post one query each and
    block; once every live worker has posted (or finished) the coordinator evaluates the batch and hands the answers back."""

    def __init__(self, n_live):
        self.cv = threading.Condition()
        self.req, self.res, self.done, self.n_live, self.err = {}, {}, set(), n_live, None

    def ask(self, e, vals):
        with self.cv:
            self.req[e] = vals
            self.cv.notify_all()
            while e not in self.res and self.err is None:
                self.cv.wait()
            if self.err is not None:
                raise RuntimeError("relabelling launch failed") from self.err
            return self.res.pop(e)

    def finish(self, e):
        with self.cv:
            self.done.add(e)
            self.cv.notify_all()

    def serve(self, evaluate):
        while True:
            with self.cv:
                while len(self.req) + len(self.done) < self.n_live:
                    self.cv.wait()
                if not self.req:
                    return
                batch = dict(self.req)
                self.req.clear()
            try:
                out = evaluate(batch)
            except Exception as ex:   # wake the workers up, then re-raise in the launching thread
                with self.cv:
                    self.err = ex
                    self.cv.notify_all()
                raise
            with self.cv:
                self.res.update(out)
                self.cv.notify_all()


def nquad_rows(relabeller: Relabeller, states, attrs, features, ranges, num_evals, rows, noise=None):
    """integration(method='nquad') (:346-362) for every row of every file: states [R, E, 6]; attrs {name: [R, E] or None}
    (the row's attribute values; swept features are overridden by the quadrature's query points); rows[e] = number of
    rows of file e.  noise: for a 'supplied' fleet a list, per file, of cuda tensors [n_calls_e, n_ind, K] consumed one per
    controller step of that file.  Returns (labels [R, E] float64 = integral / volume, calls [E] controller steps taken)."""
    from scipy.integrate import nquad
    E, R = relabeller.E, states.shape[0]
    d = len(features)
    limits = [ranges[f] for f in features]
    volume = float(np.prod([hi - lo for lo, hi in limits]))
    opts = {"limit": ceil(num_evals ** (1 / d)), "epsabs": 1e-2, "epsrel": 1e-2}   # :355-357
    dev = relabeller.device
    names = [k for k in _CONTROLLER_ATTRIBUTES if attrs.get(k) is not None or k in features]
    labels = np.full((R, E), np.nan)
    calls = np.zeros(E, dtype=np.int64)
    Q_dev = torch.zeros((1, E), device=dev)
    nz_dev = torch.zeros((1, E, relabeller.n_ind, relabeller.K), device=dev) if noise is not None else None
    for r in range(R):
        live = [e for e in range(E) if r < rows[e]]
        if not live:
            break
        sync = _Lockstep(len(live))
        s_dev = torch.from_numpy(np.ascontiguousarray(states[r:r + 1])).to(dev)
        base = {k: (np.zeros(E, np.float32) if attrs.get(k) is None else np.asarray(attrs[k][r], np.float32).copy()) for k in names}

        def worker(e):
            try:
                integral, _ = nquad(lambda *x: float(sync.ask(e, x)), limits, opts=[opts] * d)
                labels[r, e] = integral / volume
            except Exception:
                labels[r, e] = np.nan   # the reference prints the exception and leaves the row unlabelled
            finally:
                sync.finish(e)

        def evaluate(batch):
            vals = {k: v.copy() for k, v in base.items()}
            act = np.zeros((1, E), dtype=np.int32)
            for e, x in batch.items():
                act[0, e] = 1
                for f, v in zip(features, x):
                    vals[f][e] = np.float32(v)
                if nz_dev is not None:
                    nz_dev[0, e].copy_(noise[e][calls[e]])
                calls[e] += 1
            t = {k: torch.from_numpy(v.reshape(1, E)).to(dev) for k, v in vals.items()}
            relabeller.relabel_device(s_dev, t.get("target_position"), t.get("target_equilibrium"), t.get("L"), t.get("m_pole"),
                                      noise=nz_dev, Q_out=Q_dev, active=torch.from_numpy(act).to(dev))
            q = Q_dev.cpu().numpy()[0]
            return {e: float(q[e]) for e in batch}

        threads = [threading.Thread(target=worker, args=(e,), daemon=True) for e in live]
        for t in threads:
            t.start()
        try:
            sync.serve(evaluate)
        finally:
            for t in threads:
                t.join(timeout=60)
    return labels, calls


# keys of config_optimizers.yml's rpgd block that do not change the labels (logging, the reference's unused rtol) or
# that only the uniform sampling distribution reads, which RpgdFleet refuses itself
_RPGD_IGNORED = ("optimizer_logging", "calculate_optimal_trajectory", "rtol", "sample_whole_control_space",
                 "uniform_dist_min", "uniform_dist_max")


def rpgd_relabeller_keywords(block: dict) -> dict:
    """Relabeller(optimizer="rpgd") keywords from controller_config["rpgd"]: the rpgd block of config_optimizers.yml plus
    integrator / cost / cost_config / network / noise / device / file_offset; `seed: null` keeps the default seed."""
    kw = {k: v for k, v in dict(block).items() if k not in _RPGD_IGNORED}
    if kw.get("seed", 0) is None:
        del kw["seed"]
    return kw


def add_control_along_trajectories(dfs, controller_config, controller_output_variable_name="Q_calculated",
                                   integration_method="monte_carlo", integration_num_evals=64, save_output_only=False,
                                   df_modifier=lambda df: df, relabeller: Relabeller | None = None, seed=None,
                                   noise=None, init_draws=None, **kwargs):
    """The reference's function (:53-140) for one DataFrame or a LIST of them (one per recorded file), MPPI or RPGD as
    the controller.  controller_config: 'state_components' (default: the six CartPole state columns),
    'environment_attributes_dict' (controller attribute -> CSV column, with the reference's suffix conventions) and
    optionally 'mppi' (keyword arguments of Relabeller: num_rollouts, horizon, integrator, cost, ...) or 'rpgd' (the rpgd
    block of config_optimizers.yml plus integrator, cost, network, ...: an RpgdFleet relabels; not with 'mppi').
    noise: a 'supplied' relabeller's draws per expanded row ([rows, E, n_ind, K] MPPI, [rows, E, K - opt_keep_k, n_ind]
    RPGD); init_draws: a 'supplied' RPGD relabeller's reset draws [E, K, n_ind].
    Returns DataFrame(s) with the label column appended (or only the labels with save_output_only)."""
    import pandas as pd
    if "mppi" in controller_config and "rpgd" in controller_config:
        raise ValueError("controller_config takes one optimizer: 'mppi' or 'rpgd', not both")
    rpgd = "rpgd" in controller_config or getattr(relabeller, "optimizer", "mppi") == "rpgd"
    single = isinstance(dfs, pd.DataFrame)
    files = [dfs] if single else list(dfs)
    if not files:
        return []
    if isinstance(controller_output_variable_name, list) and len(controller_output_variable_name) != 1:
        raise ValueError("one control input: exactly one output variable name")
    env0 = dict(controller_config["environment_attributes_dict"])
    state_components = list(controller_config.get("state_components", STATE_COMPONENTS))
    rng = np.random.default_rng(seed)
    originals, tables, env = [], [], None
    for df in files:
        df, env_f = process_random_sampling(df, env0, rng)
        originals.append(df.copy())
        tables.append(df_modifier(df))
        features, ranges, env_i = get_integration_features(env_f)
        diff_features, env, names = get_differentiation_features(env_i, [controller_output_variable_name]
                                                                 if not isinstance(controller_output_variable_name, list)
                                                                 else controller_output_variable_name)
    if features and diff_features:
        raise ValueError("Cannot integrate and differentiate at the same time.")
    if features and integration_method not in ("monte_carlo", "nquad"):
        raise ValueError("Invalid integration method. Choose 'nquad' or 'monte_carlo'.")
    nquad_mode = bool(features) and integration_method == "nquad"
    if nquad_mode and rpgd:
        raise NotImplementedError("integration_method='nquad' is not offered under RPGD: its files sit rows out, which "
                                  "would need a solve counter, Adam iteration count and Adam steps per file; use "
                                  "'monte_carlo'")
    unknown = [k for k in features + diff_features if k not in _CONTROLLER_ATTRIBUTES]
    if unknown:
        raise ValueError(f"cannot sweep {unknown}: the controller's attributes are {_CONTROLLER_ATTRIBUTES}")
    ev = 1
    if features and not nquad_mode:
        m = int(np.ceil(np.log2(integration_num_evals)))
        ev = 2 ** m
    elif diff_features:
        ev = DIFF_WINDOW * len(diff_features)
    E = len(files)
    rows = [len(t) for t in tables]
    R = max(rows)
    states = np.zeros((R * ev, E, 6), dtype=np.float32)
    attrs = {k: None for k in _CONTROLLER_ATTRIBUTES}
    for k in _CONTROLLER_ATTRIBUTES:
        if k in env or k in features:
            attrs[k] = np.zeros((R * ev, E), dtype=np.float32)
    offsets = (np.arange(DIFF_WINDOW) - (DIFF_WINDOW - 1) // 2) * DIFF_STEP
    for e, t in enumerate(tables):
        n = rows[e]
        idx = np.minimum(np.arange(R), n - 1)   # shorter files idle on their last row; those labels are dropped
        s = t[state_components].to_numpy(dtype=np.float32)[idx]
        states[:, e] = np.repeat(s, ev, axis=0)
        for k in _CONTROLLER_ATTRIBUTES:
            if attrs[k] is not None and k in env and env[k] in t.columns:
                attrs[k][:, e] = np.repeat(t[env[k]].to_numpy(dtype=np.float32)[idx], ev)
        if features and not nquad_mode:
            smp = sobol_samples(features, ranges, ev, R, seed=None if seed is None else [int(seed), e])
            for j, f in enumerate(features):
                attrs[f][:, e] = smp[:, :, j].reshape(-1).astype(np.float32)
        for j, f in enumerate(diff_features):   # window j of every row sweeps feature f (:449-454)
            base = t[env[f]].to_numpy(dtype=np.float64)[idx]
            if np.isnan(base).any():
                raise ValueError(f"column {env[f]} has NaN entries; the derivative is undefined there")
            sweep = attrs[f][:, e].reshape(R, ev)
            sweep[:, j * DIFF_WINDOW:(j + 1) * DIFF_WINDOW] = (base[:, None] + offsets[None, :]).astype(np.float32)
    own = relabeller is None
    if own:
        if "rpgd" in controller_config:
            relabeller = Relabeller(E, optimizer="rpgd", **rpgd_relabeller_keywords(controller_config["rpgd"]))
        else:
            relabeller = Relabeller(E, **dict(controller_config.get("mppi", {})))
    if relabeller.E != E:
        raise ValueError(f"the relabeller was built for {relabeller.E} files, got {E}")
    try:
        if init_draws is None:
            relabeller.reset()
        else:
            relabeller.reset(init_draws=init_draws)
        if nquad_mode:
            labels_nq, _ = nquad_rows(relabeller, states, attrs, features, ranges, integration_num_evals, rows, noise=noise)
            Q = np.zeros((R, E), dtype=np.float32)
        else:
            Q = relabeller.relabel(states, attrs["target_position"], attrs["target_equilibrium"], attrs["L"], attrs["m_pole"],
                                   noise=noise)
    finally:
        if own:
            relabeller.close()
    Q = Q.reshape(R, ev, E).astype(np.float64)
    if nquad_mode:
        labels = labels_nq[:, None, :]
    elif diff_features:
        from scipy.signal import savgol_filter
        half = (DIFF_WINDOW - 1) // 2
        u = Q.reshape(R, len(diff_features), DIFF_WINDOW, E)
        der = savgol_filter(u, window_length=DIFF_WINDOW, polyorder=DIFF_POLYORDER, deriv=1, delta=DIFF_STEP, axis=2,
                            mode="constant")[:, :, half, :]
        labels = np.concatenate([der, u[:, :, half, :]], axis=1)   # [R, 2 * features, E]: jacobian, then central outputs
    else:
        labels = Q.mean(axis=1)[:, None, :]   # np.mean(evaluations) of :339-345
    out = []
    for e in range(E):
        lab = labels[:rows[e], :, e]
        if save_output_only:
            out.append(pd.DataFrame(lab, columns=names))
        else:
            d = originals[e]
            d[names] = lab
            out.append(d)
    return out[0] if single else out
