"""Fleets: many independent closed-loop experiments advanced together on the device (include/cps.h "fleet").

Host-side mirror of what the reference does for ONE cartpole per process when it generates data
(CartPole/data_generator.py:94-236 random_experiment_setter + generate_random_initial_state,
CartPole/random_target_generator.py:9-87, CartPole/__init__.py:578-739 setup/run_cartpole_random_experiment):
random initial states, a random target-position trace per experiment, the up/down target-equilibrium schedule, then
controller period after controller period of [MPPI solve -> plant].  Here the solve and the plant of ALL experiments
run in one kernel launch per controller period (cps_fleet_step); the host only prepares the target tables and, at the
end, reads the record rows back.  No CPU fallback: everything below the table preparation happens in libcps_b200.so.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _lib as L
from .core import Engine, _check_dev, _check_sizes, _ptr

TRACK_HALF_LENGTH = float(np.float32((44.0e-2 - 4.4e-2) / 2.0))


@dataclass
class DataGenConfig:
    """config_data_gen.yml:6-31 (defaults as shipped)."""
    length_of_experiment: float = 360.0
    angle_init_limits: tuple = (0.0, 180.0)          # degrees; mirrored to the left half plane with p = 0.5
    angleD_init_limit: float = 1200.0                 # degrees / s
    position_init_limit: float = 0.8                  # fraction of TrackHalfLength
    positionD_init_limit: float = 0.5
    start_at_target: bool = True
    track_fraction_usable_for_target_position: float = 1.0
    target_position_end: float | None = None
    initial_target_equilibrium: int = 1
    keep_target_equilibrium_x_seconds_up: float = 10.0
    keep_target_equilibrium_x_seconds_down: float = 2.5
    dt_simulation: float = 0.002
    dt_control: float = 0.02
    track_relative_complexity: float = 1.0
    interpolation_type: tuple = ("previous", "0-derivative-smooth")   # cycled over the experiments (:205-209)
    turning_points_period: str = "regular"
    position: float | None = None
    positionD: float | None = None
    angle: float | None = None
    angleD: float | None = None
    extra: dict = field(default_factory=dict)


def random_initial_state(rng, cfg: DataGenConfig) -> np.ndarray:
    """generate_random_initial_state (CartPole/data_generator.py:238-275); draws in the same order."""
    s = np.zeros(6, dtype=np.float32)
    thl, f32 = np.float32(TRACK_HALF_LENGTH), np.float32
    # python float * float32 0-d array * python float: float32 arithmetic under NEP 50, as in the reference
    s[4] = f32(rng.uniform(-1.0, 1.0)) * thl * f32(cfg.position_init_limit) if cfg.position is None else cfg.position
    s[5] = f32(rng.uniform(-1.0, 1.0)) * thl * f32(cfg.positionD_init_limit) if cfg.positionD is None else cfg.positionD
    if cfg.angle is None:
        lo, hi = cfg.angle_init_limits
        if rng.uniform() > 0.5:
            s[0] = rng.uniform(lo, hi) * (np.pi / 180.0)
        else:
            s[0] = rng.uniform(-hi, -lo) * (np.pi / 180.0)
    else:
        s[0] = cfg.angle
    s[1] = rng.uniform(-1.0, 1.0) * cfg.angleD_init_limit * (np.pi / 180.0) if cfg.angleD is None else cfg.angleD
    s[2], s[3] = np.cos(s[0]), np.sin(s[0])
    return s


def random_trace_function(rng, cfg: DataGenConfig, interpolation_type: str, start_at, end_at):
    """Generate_Random_Trace_Function (CartPole/random_target_generator.py:9-87)."""
    from scipy.interpolate import BPoly, interp1d
    frac = cfg.track_fraction_usable_for_target_position
    n_tp = int(np.floor(cfg.length_of_experiment * cfg.track_relative_complexity))
    y = rng.uniform(-1.0, 1.0, n_tp) * frac * TRACK_HALF_LENGTH
    if n_tp == 0:
        y = np.array([0.0, 0.0])
    elif n_tp == 1:
        if start_at is not None:
            y[0] = start_at
        elif end_at is not None:
            y[0] = end_at
        y = np.append(y, y[0])
    else:
        if start_at is not None:
            y[0] = start_at
        if end_at is not None:
            y[-1] = end_at
    random_samples = max(n_tp - 2, 0)
    if cfg.turning_points_period == "random":
        t_init = np.concatenate([[0.0], np.sort(rng.uniform(0.0, 1.0, random_samples)), [1.0]])
    elif cfg.turning_points_period == "regular":
        t_init = np.linspace(0, 1.0, num=random_samples + 2, endpoint=True)
    else:
        raise NotImplementedError("There is no mode corresponding to this value of turning_points_period variable")
    t_init = t_init * cfg.length_of_experiment
    if interpolation_type == "0-derivative-smooth":
        f = BPoly.from_derivatives(t_init, [[v, 0] for v in y], extrapolate="periodic")
    elif interpolation_type == "linear":
        f = interp1d(t_init, y, kind="linear", fill_value="extrapolate")
    elif interpolation_type == "previous":
        f = interp1d(t_init, y, kind="previous", fill_value="extrapolate")
    else:
        raise ValueError("Unknown interpolation type.")
    lim = frac * TRACK_HALF_LENGTH
    return lambda t: np.clip(f(t), -lim, lim)


def control_times(n_periods: int, cfg: DataGenConfig) -> np.ndarray:
    """Plant time at which the controller is called in period j: the reference accumulates self.time + dt_simulation
    tick by tick (CartPole/__init__.py:326-327); period 0 is solved at time 0 (set_cartpole_state_at_t0, :866-881)."""
    n_sim = int(round(cfg.dt_control / cfg.dt_simulation))
    t = np.concatenate([[0.0], np.cumsum(np.full(n_periods * n_sim, cfg.dt_simulation))])
    return t[::n_sim][:n_periods]


def target_equilibrium_schedule(n_periods: int, cfg: DataGenConfig, te0: int | None = None) -> np.ndarray:
    """update_target_equilibrium (CartPole/__init__.py:380-388) evaluated on every plant tick; returns the value the
    controller sees in each period, float32 [n_periods]."""
    n_sim = int(round(cfg.dt_control / cfg.dt_simulation))
    cur = float(cfg.initial_target_equilibrium if te0 is None else te0)
    out = np.empty(n_periods, dtype=np.float32)
    out[0] = cur
    t, t_last = 0.0, None
    for i in range(1, (n_periods - 1) * n_sim + 1):
        t = t + cfg.dt_simulation
        if t_last is None:
            t_last = t
        elif cur == -1 and (t - t_last) > cfg.keep_target_equilibrium_x_seconds_down:
            t_last, cur = t, -cur
        elif cur == 1 and (t - t_last) > cfg.keep_target_equilibrium_x_seconds_up:
            t_last, cur = t, -cur
        if i % n_sim == 0:
            out[i // n_sim] = cur
    return out


def make_experiments(n_experiments: int, n_periods: int, cfg: DataGenConfig | None = None, seed: int = 0,
                     experiment_offset: int = 0):
    """Initial states [E,6], target-position table [n_periods,E] and target-equilibrium table [n_periods,E] for
    experiments experiment_offset .. experiment_offset+E-1.  Each experiment has its own numpy Generator seeded with
    (seed, global index), so the tables do not depend on how the experiments are sharded over GPUs."""
    cfg = cfg or DataGenConfig()
    times = control_times(n_periods, cfg)
    s0 = np.zeros((n_experiments, 6), dtype=np.float32)
    tp = np.zeros((n_periods, n_experiments), dtype=np.float32)
    te_one = target_equilibrium_schedule(n_periods, cfg)
    te = np.repeat(te_one[:, None], n_experiments, axis=1)
    itypes = cfg.interpolation_type if isinstance(cfg.interpolation_type, (list, tuple)) else (cfg.interpolation_type,)
    for e in range(n_experiments):
        g = experiment_offset + e
        rng = np.random.default_rng([seed, g])
        s0[e] = random_initial_state(rng, cfg)
        start_at = float(s0[e, 4]) if cfg.start_at_target else \
            cfg.track_fraction_usable_for_target_position * TRACK_HALF_LENGTH * rng.uniform(-1.0, 1.0)
        end_at = cfg.track_fraction_usable_for_target_position * TRACK_HALF_LENGTH * rng.uniform(-1.0, 1.0) \
            if cfg.target_position_end is None else cfg.target_position_end
        f = random_trace_function(rng, cfg, itypes[g % len(itypes)], start_at, end_at)
        tp[:, e] = np.asarray(f(np.minimum(times, cfg.length_of_experiment)), dtype=np.float64).astype(np.float32)
    return s0, tp, te


def _check_fleet_args(kind: str, integrator: str, network, noise: str, dt: float, dt_simulation: float) -> int:
    """The checks Fleet and RpgdFleet make before they create a handle; returns the plant ticks per controller period."""
    if integrator == "neural" and network is None:
        raise NotImplementedError(f"{kind} with integrator='neural' needs the network: pass network=<spec dict as "
                                  "Engine.net_load takes, e.g. neural.load_model(...)[0]>")
    if network is not None and integrator != "neural":
        raise ValueError(f"network= is the neural predictor's model; integrator={integrator!r} takes none")
    if noise not in ("philox", "supplied"):
        raise ValueError("noise must be 'philox' or 'supplied'")
    n_sim = int(round(dt / dt_simulation))
    if n_sim < 1 or abs(n_sim * dt_simulation - dt) > 1e-9:
        raise ValueError("dt (control) must be a multiple of dt_simulation")
    return n_sim


def _relabel_rows(fleet, states, Q_out):
    """The number of rows R of recorded states [R, E, 6] for `fleet`'s relabel, and Q_out (allocated [R, E] when None)."""
    _check_dev(states, "states", fleet.device)
    R = int(states.shape[0]) if states.dim() == 3 else -1
    if tuple(states.shape) != (R, fleet.E, 6):
        raise ValueError(f"states has shape {tuple(states.shape)}, expected (rows, {fleet.E}, 6)")
    if Q_out is None:
        Q_out = torch.empty((R, fleet.E), device=fleet.device, dtype=torch.float32)
    return R, Q_out


class _FleetBase:
    """What the MPPI, RPGD and CEM fleets do alike: one Engine with one fleet of the kind `_abi` names (the C ABI's
    function prefix) attached, created from the config header every fleet config struct begins with."""
    _abi = ""

    def _fn(self, name):
        return getattr(self.engine.lib, f"{self._abi}_{name}")

    def _setup_engine(self, control_limits, cost_config):
        """The optimizers' control limits (set_mppi_params lo, hi) and an optional cost configuration."""
        lo, hi = (float(np.asarray(x, dtype=np.float32).reshape(-1)[0]) for x in control_limits)
        if cost_config is not None:
            self.engine.set_cost_config(cost_config)
        self.engine.set_mppi_params(lo=lo, hi=hi)

    def _create(self, config, n_sim: int, noise: str, dt_simulation: float, seed: int, experiment_offset: int, *rest):
        """<abi>_create with the header (struct_size, E, sim_substeps, draw source, dt_simulation, seed,
        experiment_offset) followed by the fleet's own fields `rest`."""
        c = config(C.sizeof(config), self.E, n_sim, L.FLEET_NOISE_PHILOX if noise == "philox" else L.FLEET_NOISE_SUPPLIED,
                   float(dt_simulation), int(seed), int(experiment_offset), *rest)
        self.noise_source = noise
        self.engine._chk(self._fn("create")(self.engine._h, C.byref(c)))

    def close(self):
        self.engine.close()

    def _host_states(self, states) -> np.ndarray:
        s = np.ascontiguousarray(states, dtype=np.float32)
        if s.shape != (self.E, 6):
            raise ValueError(f"states must have shape ({self.E}, 6)")
        self.engine.use_current_stream()
        return s

    def states(self, with_u_prev: bool = False):
        s = np.zeros((self.E, 6), dtype=np.float32)
        u_prev = np.zeros(self.E, dtype=np.float32) if with_u_prev else None
        self.engine.use_current_stream()
        self.engine._chk(self._fn("get_states")(self.engine._h, s.ctypes.data_as(L._FP),
                                                None if u_prev is None else u_prev.ctypes.data_as(L._FP)))
        return (s, u_prev) if with_u_prev else s

    @property
    def period(self) -> int:
        return int(self._fn("period")(self.engine._h))

    def nonfinite_costs(self) -> int:
        """Non-finite plan costs met so far (a NaN state or target makes them so; such costs sort after every number, as
        torch.sort does, stay in their experiment, and the run goes on).  Synchronises."""
        self.engine.use_current_stream()
        return self.engine.nonfinite_costs()

    def set_plant_models(self, *args, **kwargs):
        raise NotImplementedError(f"{type(self).__name__} has no plant-side models (control disturbance, measurement noise, "
                                  "latency)")

    def _check_rows(self, rows: int, target_position, target_equilibrium, record, J_out, *more):
        """Device and size of the [rows, E] targets, record [rows, E, 16], J_out [rows, E, K] and `more` ((tensor, name,
        numel) as _check_sizes takes them) of run / relabel; the engine on the current stream."""
        self.engine.use_current_stream()
        _check_sizes(self.device, (target_position, "target_position", rows * self.E),
                     (target_equilibrium, "target_equilibrium", rows * self.E),
                     (record, "record", rows * self.E * L.FLEET_RECORD), (J_out, "J_out", rows * self.E * self.K), *more)


class Fleet(_FleetBase):
    """E closed-loop experiments on one device = one cps_handle with a fleet attached.

    Predictor "ODE" / "ODE_v0", or "neural" with `network`: the spec dict Engine.net_load takes
    (neural.load_model(...)[0], neural.build_net_spec, neural.synthetic_net_spec), loaded before the fleet is created;
    `net_kernel` (None, 'tensor', 'fp32') is Engine's.  The network lives in the controller only; the plant stays the
    CartPole ODE.  Each experiment then owns a hidden state (net_states / set_net_states), set to the network's stored
    state by reset() and advanced on (u, s) after every solve, as optimizer_mppi does.  Plant-side models are not offered
    on neural fleets (set_plant_models raises NotImplementedError)."""
    _abi = "cps_fleet"

    def __init__(self, n_experiments: int, num_rollouts: int = 2000, horizon: int = 50, dt: float = 0.02,
                 substeps: int = 10, integrator: str = "ODE", cost: str = "quadratic_boundary_grad_minimal",
                 interp_period: int = 10, device: int | None = None, noise: str = "philox", seed: int = 0,
                 experiment_offset: int = 0, dt_simulation: float = 0.002, no_pairs: bool = False,
                 network: dict | None = None, net_kernel: str | None = None):
        n_sim = _check_fleet_args("Fleet", integrator, network, noise, dt, dt_simulation)
        self.engine = Engine(num_rollouts, horizon, dt=dt, substeps=substeps, integrator=integrator, cost=cost,
                             interp_period=interp_period, device=device, no_pairs=no_pairs, net_kernel=net_kernel)
        self.neural = network is not None
        if self.neural:
            self.engine.net_load(network)
        self.E, self.K, self.T = int(n_experiments), int(num_rollouts), int(horizon)
        self.n_ind, self.device = self.engine.n_ind, self.engine.device
        self._create(L.cps_fleet_config, n_sim, noise, dt_simulation, seed, experiment_offset)

    def reset(self, states, period: int = 0):
        s = self._host_states(states)
        self.engine._chk(self.engine.lib.cps_fleet_set_states(self.engine._h, s.ctypes.data_as(L._FP), int(period)))

    def states(self, with_u_nom: bool = False):
        s = np.zeros((self.E, 6), dtype=np.float32)
        u_nom = np.zeros((self.E, self.T), dtype=np.float32) if with_u_nom else None
        u_prev = np.zeros(self.E, dtype=np.float32) if with_u_nom else None
        self.engine.use_current_stream()
        self.engine._chk(self.engine.lib.cps_fleet_get_states(
            self.engine._h, s.ctypes.data_as(L._FP), None if u_nom is None else u_nom.ctypes.data_as(L._FP),
            None if u_prev is None else u_prev.ctypes.data_as(L._FP)))
        return (s, u_nom, u_prev) if with_u_nom else s

    def noise(self, period: int) -> torch.Tensor:
        """The draws the Philox source uses in `period`: cuda tensor [E, n_ind, K]."""
        out = torch.empty((self.E, self.n_ind, self.K), device=self.device, dtype=torch.float32)
        self.engine.use_current_stream()
        self.engine._chk(self.engine.lib.cps_fleet_noise(self.engine._h, int(period), _ptr(out)))
        return out

    def net_states(self) -> np.ndarray:
        """[E, Htot]: every experiment's hidden state (neural fleets).  Synchronises."""
        htot = getattr(self.engine, "net_htot", 0)
        out = np.zeros((self.E, max(htot, 1)), dtype=np.float32)
        self.engine.use_current_stream()
        self.engine._chk(self.engine.lib.cps_fleet_get_net_states(self.engine._h, out.ctypes.data_as(L._FP)))
        return out[:, :htot]

    def set_net_states(self, states):
        """Sets every experiment's hidden state from [E, Htot] (neural fleets; after reset(), which sets them to the
        network's stored state)."""
        v = np.ascontiguousarray(states, dtype=np.float32)
        if v.shape != (self.E, self.engine.net_htot):
            raise ValueError(f"hidden states must have shape ({self.E}, {self.engine.net_htot})")
        self.engine.use_current_stream()
        self.engine._chk(self.engine.lib.cps_fleet_set_net_states(self.engine._h, v.ctypes.data_as(L._FP)))

    _CONTROL_NOISE = {"OFF": 0, "additive": 1, "truncnorm": 2}

    def set_plant_models(self, control_noise_mode: str = "OFF", control_noise: float = 0.0, control_bias: float = 0.0,
                         noise_mode: str = "OFF", sigma_angle: float = 0.0, sigma_position: float = 0.0,
                         sigma_angleD: float = 0.0, sigma_positionD: float = 0.0, latency: float = 0.0):
        """cps_fleet_set_plant_models with the reference's configuration keys (cartpole_physical_parameters.yml:13-24:
        controlDisturbance_mode / controlDisturbance / controlBias, latency, noise.noise_mode / sigma_*).  Call before
        reset(); the first solve after reset() sees the true state (the reference's controller call at t = 0)."""
        if self.neural:
            raise NotImplementedError("plant-side models (control disturbance, measurement noise, latency) are not offered "
                                      "on fleets with the neural predictor")
        if control_noise_mode not in self._CONTROL_NOISE:
            raise ValueError(f"controlDisturbance_mode with value {control_noise_mode} not valid")
        m = L.cps_fleet_plant_models(C.sizeof(L.cps_fleet_plant_models), self._CONTROL_NOISE[control_noise_mode],
                                     float(control_noise), float(control_bias), 0 if noise_mode == "OFF" else 1,
                                     float(sigma_angle), float(sigma_position), float(sigma_angleD), float(sigma_positionD),
                                     float(latency))
        self.engine.use_current_stream()
        self.engine._chk(self.engine.lib.cps_fleet_set_plant_models(self.engine._h, C.byref(m)))
        self.plant_models = bool(m.control_noise_mode or m.measurement_noise or m.latency > 0.0)

    def observed(self) -> np.ndarray:
        """[E, 6]: the states as the controller will see them at the next solve (delayed, noisy)."""
        o = np.zeros((self.E, 6), dtype=np.float32)
        self.engine.use_current_stream()
        self.engine._chk(self.engine.lib.cps_fleet_get_observed(self.engine._h, o.ctypes.data_as(L._FP)))
        return o

    def run(self, n_periods: int, target_position=None, target_equilibrium=None, noise=None, record=None, J_out=None,
            ctrl_draws=None, meas_draws=None):
        """cps_fleet_step: n_periods launches, no synchronisation.  target_position / target_equilibrium: cuda tensors
        [n_periods, E] or None; noise: cuda tensor [n_periods, E, n_ind, K] for a 'supplied' fleet;
        record: cuda tensor [n_periods, E, 16] or None; J_out: [n_periods, E, K] or None.  With plant-side models
        (set_plant_models): ctrl_draws [n_periods, E] and meas_draws [n_periods, sim_substeps, E, 4] supply their draws
        (cps_fleet_step_noisy); a 'philox' fleet draws them itself when they are None."""
        eng = self.engine
        self._check_rows(n_periods, target_position, target_equilibrium, record, J_out,
                         (noise, "noise", n_periods * self.E * self.n_ind * self.K))
        if getattr(self, "plant_models", False):
            for t, name in ((ctrl_draws, "ctrl_draws"), (meas_draws, "meas_draws")):
                if t is not None:
                    _check_dev(t, name, self.device)
            eng._chk(eng.lib.cps_fleet_step_noisy(eng._h, int(n_periods), _ptr(target_position), _ptr(target_equilibrium),
                                                  _ptr(noise), _ptr(record), _ptr(J_out), _ptr(ctrl_draws), _ptr(meas_draws)))
            return record
        eng._chk(eng.lib.cps_fleet_step(eng._h, int(n_periods), _ptr(target_position), _ptr(target_equilibrium),
                                        _ptr(noise), _ptr(record), _ptr(J_out)))
        return record

    def relabel(self, states, target_position=None, target_equilibrium=None, L=None, m_pole=None, noise=None, Q_out=None,
                J_out=None, active=None):
        """cps_fleet_relabel: one controller step per recorded row, experiment e = file e, from the recorded states
        (cuda tensor [R, E, 6]) instead of the plant; no synchronisation.  target_position / target_equilibrium / L / m_pole:
        cuda tensors [R, E] or None; noise [R, E, n_ind, K] for a 'supplied' fleet; Q_out [R, E] (allocated when None)
        receives the controls; J_out [R, E, K] or None; active [R, E] int32 or None: files with 0 sit the row out
        (cps_fleet_relabel_masked).  Zeroing the warm starts first (Relabeller.reset: cps_fleet_reset) is the reference's
        controller.reset().  Returns Q_out."""
        eng = self.engine
        R, Q_out = _relabel_rows(self, states, Q_out)
        self._check_rows(R, target_position, target_equilibrium, None, J_out, (L, "L", R * self.E),
                         (m_pole, "m_pole", R * self.E), (noise, "noise", R * self.E * self.n_ind * self.K),
                         (Q_out, "Q_out", R * self.E))
        if active is None:
            eng._chk(eng.lib.cps_fleet_relabel(eng._h, R, _ptr(states), _ptr(target_position), _ptr(target_equilibrium),
                                               _ptr(L), _ptr(m_pole), _ptr(noise), _ptr(Q_out), _ptr(J_out)))
            return Q_out
        _check_dev(active, "active", self.device, dtype=torch.int32)
        if active.numel() != R * self.E:
            raise ValueError("active must be an int32 tensor of shape [rows, files]")
        eng._chk(eng.lib.cps_fleet_relabel_masked(eng._h, R, _ptr(states), _ptr(target_position), _ptr(target_equilibrium),
                                                  _ptr(L), _ptr(m_pole), _ptr(noise), _ptr(Q_out), _ptr(J_out),
                                                  _ptr(active)))
        return Q_out


class RpgdFleet(_FleetBase):
    """E closed-loop experiments under RPGD, the reference's shipped default optimizer (Control_Toolkit_ASF/
    config_controllers.yml:2), on one device: one cps_handle with an RPGD fleet attached (include/cps.h "RPGD fleet").

    Every controller period does, for every experiment, what optimizer_rpgd_b200.step does (Adam steps on the gradient
    of predict_and_cost, the costs of the improved plans, u = the cheapest plan's first input, the shifted warm start and
    every `resamp_per` solves the resampling of the worst plans), then what Fleet's plant does, with no host round trip.
    The keywords are optimizer_rpgd_b200's (same defaults; opt_keep_k and first_iter_count are derived as it derives
    them) and Fleet's.  Predictor "ODE", or "neural" with `network`: the spec dict Engine.net_load takes
    (neural.load_model(...)[0], neural.build_net_spec, neural.synthetic_net_spec), loaded before the fleet is created.  The
    network lives in the controller only; the plant stays the CartPole ODE.  Every gradient and cost reads the network's
    stored hidden state (zero after loading; engine.net_set_state before reset() sets another) and never advances it, as
    optimizer_rpgd_b200 and the reference's RPGD.  Cost quadratic_boundary_grad_minimal or quadratic_boundary_grad;
    uniform resampling and the plant-side models (Fleet.set_plant_models) are not implemented and raise
    NotImplementedError."""
    _abi = "cps_rpgd_fleet"

    def __init__(self, n_experiments: int, num_rollouts: int = 16, mpc_horizon: int = 35, outer_its: int = 4,
                 resamp_per: int = 10, opt_keep_k_ratio: float = 0.75, period_interpolation_inducing_points: int = 4,
                 learning_rate: float = 0.05, adam_beta_1: float = 0.9, adam_beta_2: float = 0.999,
                 adam_epsilon: float = 1e-8, gradmax_clip: float = 5.0, sample_stdev: float = 0.5,
                 sample_mean: float = 0.0, shift_previous: int = 1, warmup: bool = False, warmup_iterations: int = 250,
                 control_limits=(-1.0, 1.0), SAMPLING_DISTRIBUTION: str = "normal", dt: float = 0.02,
                 substeps: int = 10, integrator: str = "ODE", cost: str = "quadratic_boundary_grad_minimal",
                 cost_config: dict | None = None, device: int | None = None, noise: str = "philox", seed: int = 0,
                 experiment_offset: int = 0, dt_simulation: float = 0.002, network: dict | None = None):
        n_sim = _check_fleet_args("RpgdFleet", integrator, network, noise, dt, dt_simulation)
        if SAMPLING_DISTRIBUTION == "uniform":
            raise NotImplementedError("RpgdFleet resamples from the normal distribution only (SAMPLING_DISTRIBUTION='normal')")
        if SAMPLING_DISTRIBUTION != "normal":
            raise ValueError(f"RPGD cannot interpret sampling type {SAMPLING_DISTRIBUTION}")
        self.E, self.K, self.T = int(n_experiments), int(num_rollouts), int(mpc_horizon)
        self.outer_its, self.resamp_per, self.shift_previous = int(outer_its), int(resamp_per), int(shift_previous)
        self.first_iter_count = int(warmup_iterations) if warmup else self.outer_its   # as optimizer_rpgd_b200
        self.opt_keep_k = int(max(int(self.K * opt_keep_k_ratio), 1))
        self.engine = Engine(self.K, self.T, dt=dt, substeps=substeps, integrator=integrator, cost=cost,
                             interp_period=period_interpolation_inducing_points, device=device)
        self.n_ind, self.device = self.engine.n_ind, self.engine.device
        self._setup_engine(control_limits, cost_config)
        if network is not None:
            self.engine.net_load(network)
        self._create(L.cps_rpgd_fleet_config, n_sim, noise, dt_simulation, seed, experiment_offset, self.outer_its,
                     self.first_iter_count, self.resamp_per, self.opt_keep_k, self.shift_previous, float(learning_rate),
                     float(adam_beta_1), float(adam_beta_2), float(adam_epsilon), float(gradmax_clip), float(sample_stdev),
                     float(sample_mean))

    def reset(self, states, period: int = 0, init_draws=None):
        """optimizer_reset of every experiment and the initial states [E, 6].  init_draws: cuda tensor [E, K, n_ind] of
        standard normals for the initial plans ('supplied' fleets; a 'philox' fleet draws them, see draws(-1))."""
        s = self._host_states(states)
        _check_sizes(self.device, (init_draws, "init_draws", self.E * self.K * self.n_ind))
        self.engine._chk(self.engine.lib.cps_rpgd_fleet_set_states(self.engine._h, s.ctypes.data_as(L._FP),
                                                                   _ptr(init_draws), int(period)))

    def plans(self) -> dict:
        """The optimizer state of every experiment: Q, m, v [E, K, T], ages [E, K] (int32), and the shared Adam iteration
        and solve counters."""
        Q, m, v = (np.zeros((self.E, self.K, self.T), dtype=np.float32) for _ in range(3))
        ages = np.zeros((self.E, self.K), dtype=np.int32)
        it, solves = C.c_longlong(), C.c_longlong()
        self.engine.use_current_stream()
        self.engine._chk(self.engine.lib.cps_rpgd_fleet_get_plans(
            self.engine._h, Q.ctypes.data_as(L._FP), m.ctypes.data_as(L._FP), v.ctypes.data_as(L._FP),
            ages.ctypes.data_as(C.POINTER(C.c_int)), C.byref(it), C.byref(solves)))
        return dict(Q=Q, m=m, v=v, ages=ages, adam_iterations=int(it.value), solves=int(solves.value))

    def draws(self, period: int) -> torch.Tensor:
        """The draws a 'philox' fleet uses: period >= 0 its resampling draws [E, K - opt_keep_k, n_ind]; period = -1 the
        draws of reset() [E, K, n_ind]."""
        rows = self.K if period < 0 else self.K - self.opt_keep_k
        out = torch.empty((self.E, rows, self.n_ind), device=self.device, dtype=torch.float32)
        self.engine.use_current_stream()
        self.engine._chk(self.engine.lib.cps_rpgd_fleet_draws(self.engine._h, int(period), _ptr(out)))
        return out

    def run(self, n_periods: int, target_position=None, target_equilibrium=None, draws=None, record=None, J_out=None,
            Q_opt=None):
        """cps_rpgd_fleet_step: n_periods controller periods, no synchronisation.  target_position / target_equilibrium:
        cuda tensors [n_periods, E] or None; draws: [n_periods, E, K - opt_keep_k, n_ind] for a 'supplied' fleet (read in
        resampling periods only); record [n_periods, E, 16], J_out [n_periods, E, K] (costs of the improved plans) and
        Q_opt [n_periods, E, K, T] (plans after the Adam steps) or None."""
        eng = self.engine
        self._check_rows(n_periods, target_position, target_equilibrium, record, J_out,
                         (draws, "draws", n_periods * self.E * (self.K - self.opt_keep_k) * self.n_ind),
                         (Q_opt, "Q_opt", n_periods * self.E * self.K * self.T))
        eng._chk(eng.lib.cps_rpgd_fleet_step(eng._h, int(n_periods), _ptr(target_position), _ptr(target_equilibrium),
                                             _ptr(draws), _ptr(record), _ptr(J_out), _ptr(Q_opt)))
        return record

    def relabel(self, states, target_position=None, target_equilibrium=None, L=None, m_pole=None, draws=None, Q_out=None,
                J_out=None, active=None):
        """cps_rpgd_fleet_relabel: one controller step per recorded row, experiment e = file e, from the recorded states
        (cuda tensor [R, E, 6]) instead of the plant; no synchronisation.  target_position / target_equilibrium / L / m_pole:
        cuda tensors [R, E] or None (L / m_pole change predictor "ODE"'s model; the network reads neither); draws as in
        run(); Q_out [R, E] (allocated when None) receives the controls; J_out [R, E, K] or None.  reset() first is the
        reference's controller.reset().  Returns Q_out.  `active` (Fleet.relabel's per-file mask) is not implemented."""
        if active is not None:
            raise NotImplementedError("RPGD relabelling advances every file in lockstep: no per-file mask")
        eng = self.engine
        R, Q_out = _relabel_rows(self, states, Q_out)
        self._check_rows(R, target_position, target_equilibrium, None, J_out, (L, "L", R * self.E),
                         (m_pole, "m_pole", R * self.E),
                         (draws, "draws", R * self.E * (self.K - self.opt_keep_k) * self.n_ind), (Q_out, "Q_out", R * self.E))
        eng._chk(eng.lib.cps_rpgd_fleet_relabel(eng._h, R, _ptr(states), _ptr(target_position), _ptr(target_equilibrium),
                                                _ptr(L), _ptr(m_pole), _ptr(draws), _ptr(Q_out), _ptr(J_out)))
        return Q_out


class CemFleet(_FleetBase):
    """E closed-loop experiments under optimizer_cem_tf (`cem-tf` in Control_Toolkit_ASF/config_controllers.yml) on one
    device: one cps_handle with a CEM fleet attached (include/cps.h "CEM fleet").

    Every controller period does, for every experiment, what optimizer_cem_b200.step does (cem_outer_it iterations of
    sampling from the experiment's own distribution, costs, elites and the mean / stdev update; warmup_iterations on the
    first period after reset() when `warmup`; then the stdev clip, the shift and u = elite_Q[0, 0]), then what Fleet's
    plant does, with no host round trip.  The keywords are optimizer_cem_b200's (same defaults) and Fleet's.  Predictor
    "ODE" or "ODE_v0" and the four cost plugins; num_rollouts at most 8192.  Predictor "neural" takes `network`: the spec
    dict Engine.net_load takes (neural.load_model(...)[0], neural.build_net_spec, neural.synthetic_net_spec), loaded before
    the fleet is created; plain GRU / Dense networks, cost quadratic_boundary_grad_minimal or quadratic_boundary_grad.
    The network lives in the controller only; the plant stays the CartPole ODE.  Every rollout starts from the network's
    stored hidden state and none is kept per experiment (as RpgdFleet).  The plant-side models (Fleet.set_plant_models)
    are not implemented and raise NotImplementedError."""
    _abi = "cps_cem_fleet"

    def __init__(self, n_experiments: int, num_rollouts: int = 200, mpc_horizon: int = 35, cem_outer_it: int = 3,
                 cem_initial_action_stdev: float = 0.5, cem_stdev_min: float = 0.01, cem_best_k: int = 40,
                 warmup: bool = False, warmup_iterations: int = 250, control_limits=(-1.0, 1.0), dt: float = 0.02,
                 substeps: int = 10, integrator: str = "ODE", cost: str = "quadratic_boundary_grad_minimal",
                 cost_config: dict | None = None, device: int | None = None, noise: str = "philox", seed: int = 0,
                 experiment_offset: int = 0, dt_simulation: float = 0.002, network: dict | None = None):
        n_sim = _check_fleet_args("CemFleet", integrator, network, noise, dt, dt_simulation)
        self.E, self.K, self.T = int(n_experiments), int(num_rollouts), int(mpc_horizon)
        self.outer_its = int(cem_outer_it)
        self.first_iter_count = int(warmup_iterations) if warmup else self.outer_its   # as optimizer_cem_b200
        self._reset_period = None
        self.engine = Engine(self.K, self.T, dt=dt, substeps=substeps, integrator=integrator, cost=cost, device=device)
        self.device = self.engine.device
        self._setup_engine(control_limits, cost_config)
        if network is not None:
            self.engine.net_load(network)
        self._create(L.cps_cem_fleet_config, n_sim, noise, dt_simulation, seed, experiment_offset, self.outer_its,
                     self.first_iter_count, int(cem_best_k), float(cem_initial_action_stdev), float(cem_stdev_min))

    def reset(self, states, period: int = 0):
        """optimizer_reset of every experiment (mid-range mean, cem_initial_action_stdev, u_prev = 0, solve counter 0),
        the initial states [E, 6] and the period counter."""
        s = self._host_states(states)
        self.engine._chk(self.engine.lib.cps_cem_fleet_set_states(self.engine._h, s.ctypes.data_as(L._FP), int(period)))
        self._reset_period = int(period)

    def iterations(self, period: int) -> int:
        """The outer iterations of controller period `period`: first_iter_count on the period reset() set, else
        cem_outer_it."""
        return self.first_iter_count if period == self._reset_period else self.outer_its

    def distribution(self):
        """(mean, stdev), each [E, T]: every experiment's sampling distribution.  Synchronises."""
        mu, sd = np.zeros((self.E, self.T), dtype=np.float32), np.zeros((self.E, self.T), dtype=np.float32)
        self.engine.use_current_stream()
        self.engine._chk(self.engine.lib.cps_cem_fleet_get_distribution(self.engine._h, mu.ctypes.data_as(L._FP),
                                                                        sd.ctypes.data_as(L._FP)))
        return mu, sd

    def draws(self, period: int) -> torch.Tensor:
        """The draws a 'philox' fleet uses in `period`: cuda tensor [iterations(period), E, T, K]."""
        if self._reset_period is None:
            raise RuntimeError("CemFleet.draws: reset() first (the first period's iteration count depends on it)")
        out = torch.empty((self.iterations(period), self.E, self.T, self.K), device=self.device, dtype=torch.float32)
        self.engine.use_current_stream()
        self.engine._chk(self.engine.lib.cps_cem_fleet_draws(self.engine._h, int(period), _ptr(out)))
        return out

    def run(self, n_periods: int, target_position=None, target_equilibrium=None, draws=None, record=None, J_out=None,
            Q_out=None):
        """cps_cem_fleet_step: n_periods controller periods, no synchronisation.  target_position / target_equilibrium:
        cuda tensors [n_periods, E] or None; draws: the periods' standard normals back to back, [sum of iterations(p), E,
        T, K], for a 'supplied' fleet; record [n_periods, E, 16], J_out [n_periods, E, K] and Q_out [n_periods, E, T, K]
        (costs and plans of each period's last iteration) or None."""
        eng = self.engine
        p0 = self.period
        n_it = sum(self.iterations(p0 + j) for j in range(n_periods))
        self._check_rows(n_periods, target_position, target_equilibrium, record, J_out,
                         (draws, "draws", n_it * self.E * self.T * self.K), (Q_out, "Q_out", n_periods * self.E * self.T * self.K))
        eng._chk(eng.lib.cps_cem_fleet_step(eng._h, int(n_periods), _ptr(target_position), _ptr(target_equilibrium),
                                            _ptr(draws), _ptr(record), _ptr(J_out), _ptr(Q_out)))
        return record


class CemGmmFleet(_FleetBase):
    """E closed-loop experiments under optimizer_cem_gmm_tf (`cem-gmm-tf` in Control_Toolkit_ASF/config_controllers.yml) on
    one device: one cps_handle with a CEM-GMM fleet attached (include/cps.h "CEM-GMM and random-action fleets").

    Every controller period does, for every experiment, what optimizer_cem_gmm_b200.step does (cem_outer_it iterations of
    sampling from the experiment's own two-component mixture, costs, elites, the two clusters around the two cheapest
    elites and their mean / stdev / weight; then u = elite_Q[0, 0] and the shift), then what Fleet's plant does, with no
    host round trip.  The keywords are optimizer_cem_gmm_b200's (same defaults) and Fleet's.  Predictor "ODE" or "ODE_v0"
    and the four cost plugins; num_rollouts at most 8192, cem_best_k at least 2.  Predictor "neural" takes `network`: the spec
    dict Engine.net_load takes (neural.load_model(...)[0], neural.build_net_spec, neural.synthetic_net_spec), loaded before
    the fleet is created; plain GRU / Dense networks, cost quadratic_boundary_grad_minimal or quadratic_boundary_grad.
    The network lives in the controller only; the plant stays the CartPole ODE.  Every rollout starts from the network's
    stored hidden state and none is kept per experiment (as RpgdFleet).  The plant-side models (Fleet.set_plant_models)
    are not implemented and raise NotImplementedError."""
    _abi = "cps_cem_gmm_fleet"

    def __init__(self, n_experiments: int, num_rollouts: int = 200, mpc_horizon: int = 35, cem_outer_it: int = 3,
                 cem_initial_action_stdev: float = 0.5, cem_stdev_min: float = 0.01, cem_best_k: int = 40,
                 control_limits=(-1.0, 1.0), dt: float = 0.02, substeps: int = 10, integrator: str = "ODE",
                 cost: str = "quadratic_boundary_grad_minimal", cost_config: dict | None = None, device: int | None = None,
                 noise: str = "philox", seed: int = 0, experiment_offset: int = 0, dt_simulation: float = 0.002,
                 network: dict | None = None):
        n_sim = _check_fleet_args("CemGmmFleet", integrator, network, noise, dt, dt_simulation)
        self.E, self.K, self.T = int(n_experiments), int(num_rollouts), int(mpc_horizon)
        self.outer_its = int(cem_outer_it)
        self.engine = Engine(self.K, self.T, dt=dt, substeps=substeps, integrator=integrator, cost=cost, device=device)
        self.device = self.engine.device
        self._setup_engine(control_limits, cost_config)
        if network is not None:
            self.engine.net_load(network)
        self._create(L.cps_cem_gmm_fleet_config, n_sim, noise, dt_simulation, seed, experiment_offset, self.outer_its,
                     int(cem_best_k), float(cem_initial_action_stdev), float(cem_stdev_min))

    def reset(self, states, period: int = 0):
        """optimizer_reset of every experiment (both components at mid-range with cem_initial_action_stdev, p1 = 0.5,
        u_prev = 0), the initial states [E, 6] and the period counter."""
        s = self._host_states(states)
        self.engine._chk(self.engine.lib.cps_cem_gmm_fleet_set_states(self.engine._h, s.ctypes.data_as(L._FP), int(period)))

    def distribution(self):
        """(loc [E, 2, T], scale [E, 2, T], p1 [E]): every experiment's mixture.  Synchronises."""
        loc, scale = (np.zeros((self.E, 2, self.T), dtype=np.float32) for _ in range(2))
        p1 = np.zeros(self.E, dtype=np.float32)
        self.engine.use_current_stream()
        self.engine._chk(self.engine.lib.cps_cem_gmm_fleet_get_distribution(
            self.engine._h, loc.ctypes.data_as(L._FP), scale.ctypes.data_as(L._FP), p1.ctypes.data_as(L._FP)))
        return loc, scale, p1

    def draws(self, period: int):
        """The draws a 'philox' fleet uses in `period`: cuda tensors eps [cem_outer_it, E, 2, T, K] (standard normals of
        both components) and u01 [cem_outer_it, E, T, K] (the component-picking uniforms)."""
        eps = torch.empty((self.outer_its, self.E, 2, self.T, self.K), device=self.device, dtype=torch.float32)
        u01 = torch.empty((self.outer_its, self.E, self.T, self.K), device=self.device, dtype=torch.float32)
        self.engine.use_current_stream()
        self.engine._chk(self.engine.lib.cps_cem_gmm_fleet_draws(self.engine._h, int(period), _ptr(eps), _ptr(u01)))
        return eps, u01

    def run(self, n_periods: int, target_position=None, target_equilibrium=None, eps=None, u01=None, record=None,
            J_out=None, Q_out=None):
        """cps_cem_gmm_fleet_step: n_periods controller periods, no synchronisation.  target_position /
        target_equilibrium: cuda tensors [n_periods, E] or None; eps [n_periods * cem_outer_it, E, 2, T, K] and u01
        [n_periods * cem_outer_it, E, T, K] for a 'supplied' fleet; record [n_periods, E, 16], J_out [n_periods, E, K] and
        Q_out [n_periods, E, T, K] (costs and plans of each period's last iteration) or None."""
        eng = self.engine
        n_it = n_periods * self.outer_its
        self._check_rows(n_periods, target_position, target_equilibrium, record, J_out,
                         (eps, "eps", n_it * self.E * 2 * self.T * self.K), (u01, "u01", n_it * self.E * self.T * self.K),
                         (Q_out, "Q_out", n_periods * self.E * self.T * self.K))
        eng._chk(eng.lib.cps_cem_gmm_fleet_step(eng._h, int(n_periods), _ptr(target_position), _ptr(target_equilibrium),
                                                _ptr(eps), _ptr(u01), _ptr(record), _ptr(J_out), _ptr(Q_out)))
        return record


class RandomActionFleet(_FleetBase):
    """E closed-loop experiments under optimizer_random_action_tf (`random-action-tf` in Control_Toolkit_ASF/
    config_controllers.yml) on one device: one cps_handle with a random-action fleet attached (include/cps.h "CEM-GMM and
    random-action fleets").

    Every controller period does, for every experiment, what optimizer_random_action_b200.step does (K plans uniform in the
    control limits, their costs from the experiment's state, u_prev and targets, u = the cheapest plan's first input),
    then what Fleet's plant does, with no host round trip.  The keywords are optimizer_random_action_b200's (same
    defaults) and Fleet's.  Predictor "ODE" or "ODE_v0" and the four cost plugins; num_rollouts at most 8192.  Predictor "neural" takes `network`: the spec
    dict Engine.net_load takes (neural.load_model(...)[0], neural.build_net_spec, neural.synthetic_net_spec), loaded before
    the fleet is created; plain GRU / Dense networks, cost quadratic_boundary_grad_minimal or quadratic_boundary_grad.
    The network lives in the controller only; the plant stays the CartPole ODE.  Every rollout starts from the network's
    stored hidden state and none is kept per experiment (as RpgdFleet).  The plant-side models (Fleet.set_plant_models)
    are not implemented and raise NotImplementedError."""
    _abi = "cps_random_action_fleet"

    def __init__(self, n_experiments: int, num_rollouts: int = 200, mpc_horizon: int = 35, control_limits=(-1.0, 1.0),
                 dt: float = 0.02, substeps: int = 10, integrator: str = "ODE", cost: str = "quadratic_boundary_grad_minimal",
                 cost_config: dict | None = None, device: int | None = None, noise: str = "philox", seed: int = 0,
                 experiment_offset: int = 0, dt_simulation: float = 0.002, network: dict | None = None):
        n_sim = _check_fleet_args("RandomActionFleet", integrator, network, noise, dt, dt_simulation)
        self.E, self.K, self.T = int(n_experiments), int(num_rollouts), int(mpc_horizon)
        self.engine = Engine(self.K, self.T, dt=dt, substeps=substeps, integrator=integrator, cost=cost, device=device)
        self.device = self.engine.device
        self._setup_engine(control_limits, cost_config)
        if network is not None:
            self.engine.net_load(network)
        self._create(L.cps_random_action_fleet_config, n_sim, noise, dt_simulation, seed, experiment_offset)

    def reset(self, states, period: int = 0):
        """u_prev = 0, the initial states [E, 6] and the period counter."""
        s = self._host_states(states)
        self.engine._chk(self.engine.lib.cps_random_action_fleet_set_states(self.engine._h, s.ctypes.data_as(L._FP),
                                                                            int(period)))

    def draws(self, period: int) -> torch.Tensor:
        """The plans a 'philox' fleet evaluates in `period`: cuda tensor [E, T, K]."""
        out = torch.empty((self.E, self.T, self.K), device=self.device, dtype=torch.float32)
        self.engine.use_current_stream()
        self.engine._chk(self.engine.lib.cps_random_action_fleet_draws(self.engine._h, int(period), _ptr(out)))
        return out

    def run(self, n_periods: int, target_position=None, target_equilibrium=None, plans=None, record=None, J_out=None,
            Q_out=None):
        """cps_random_action_fleet_step: n_periods controller periods, no synchronisation.  target_position /
        target_equilibrium: cuda tensors [n_periods, E] or None; plans [n_periods, E, T, K] for a 'supplied' fleet;
        record [n_periods, E, 16], J_out [n_periods, E, K] and Q_out [n_periods, E, T, K] (the plans evaluated) or None."""
        eng = self.engine
        self._check_rows(n_periods, target_position, target_equilibrium, record, J_out,
                         (plans, "plans", n_periods * self.E * self.T * self.K),
                         (Q_out, "Q_out", n_periods * self.E * self.T * self.K))
        eng._chk(eng.lib.cps_random_action_fleet_step(eng._h, int(n_periods), _ptr(target_position),
                                                      _ptr(target_equilibrium), _ptr(plans), _ptr(record), _ptr(J_out),
                                                      _ptr(Q_out)))
        return record


class LegacyFleet(_FleetBase):
    """E closed-loop experiments under the legacy controller_mppi_cartpole (`mppi-cartpole` in
    Control_Toolkit_ASF/config_controllers.yml:9-30) on one device: one cps_handle with a legacy fleet attached
    (include/cps.h "Legacy controller fleet").

    Every controller period does, for every experiment, what controller_mppi_cartpole_b200.step does (on solve periods the
    K x T perturbations of SAMPLING_TYPE, the unclipped rollouts, q() + phi(), the exp-weighted unclipped update and the
    zero-fill shift; on the others the shift alone; then the actuator noise and the clip), then what Fleet's plant does,
    with no host round trip.  The keywords are controller_mppi_cartpole_b200's (config: the "mppi-cartpole" block, missing
    keys take DEFAULT_CONFIG; **kwargs override it) and Fleet's.  The block's `seed` keys the reference's host generator and
    has no meaning here: it is accepted and ignored, and `seed=` keys the Philox streams.  Predictor "ODE" or "ODE_v0"
    (optionally "ODE:n").  The legacy cost has no target equilibrium: target_equilibrium is only recorded.  cost_noise
    != 0, the "neural" predictor and the plant-side models (Fleet.set_plant_models) raise NotImplementedError."""
    _abi = "cps_legacy_fleet"
    SAMPLING = {"iid": 0, "random_walk": 1, "uniform": 2, "repeated": 3, "interpolated": 4}

    def __init__(self, n_experiments: int, config: dict | None = None, dt: float = 0.02, intermediate_steps: int = 10,
                 actuator_noise: float = 0.0, device: int | None = None, noise: str = "philox", seed: int = 0,
                 experiment_offset: int = 0, dt_simulation: float = 0.002, **kwargs):
        from .controller_mppi_cartpole_b200 import DEFAULT_CONFIG
        cfg = dict(DEFAULT_CONFIG)
        cfg.update(config or {})
        cfg.update(kwargs)
        self.config = cfg
        spec = str(cfg["predictor_specification"]).split(":")
        if spec[0] not in ("ODE", "ODE_v0"):
            raise NotImplementedError(f"LegacyFleet: predictor {spec[0]!r} (ODE and ODE_v0 are built)")
        if float(cfg["cost_noise"]) != 0.0:
            raise NotImplementedError("LegacyFleet: cost_noise != 0 would need cost weights per experiment")
        sampling = "iid" if cfg["SAMPLING_TYPE"] is None else cfg["SAMPLING_TYPE"]
        if sampling not in self.SAMPLING:
            raise ValueError(f"LegacyFleet: unknown SAMPLING_TYPE {sampling!r} (one of {sorted(self.SAMPLING)})")
        n_sim = _check_fleet_args("LegacyFleet", spec[0], None, noise, dt, dt_simulation)
        self.E, self.K, self.T = int(n_experiments), int(cfg["num_rollouts"]), int(cfg["mpc_horizon"])
        self.sampling_type, self.update_every = sampling, int(cfg["update_every"])
        self.intermediate_steps = int(spec[1]) if len(spec) > 1 else int(intermediate_steps)
        self.dt, self.p_Q = float(dt), float(actuator_noise)
        self.stdev = float(cfg["SQRTRHOINV"] * (1 / np.sqrt(self.dt)))   # float64, as the mirror's SQRTRHODTINV
        self.n_draws = {"repeated": 1, "interpolated": int(np.ceil(self.T / 10)) + 1}.get(sampling, self.T)
        self._reset_period = None
        self.engine = Engine(self.K, self.T, dt=self.dt, substeps=self.intermediate_steps, integrator=spec[0],
                             cost="legacy_mppi", noise_mode="direct", device=device)
        self.device = self.engine.device
        self.engine.set_cost_params([cfg["dd_weight"], cfg["ep_weight"], cfg["ekp_weight"], cfg["ekc_weight"],
                                     cfg["ccrc_weight"]])
        self.engine.set_mppi_params(cc_weight=cfg["cc_weight"], R=cfg["R"], LBD=cfg["LBD"], NU=cfg["NU"],
                                    SQRTRHOINV=cfg["SQRTRHOINV"])
        self._create(L.cps_legacy_fleet_config, n_sim, noise, dt_simulation, seed, experiment_offset,
                     self.SAMPLING[sampling], self.update_every, self.stdev, self.p_Q)

    def reset(self, states, period: int = 0):
        """Every experiment as a freshly configured controller (u = u_prev = 0, iteration counter restarted so that
        `period` solves), the initial states [E, 6] and the period counter."""
        s = self._host_states(states)
        self.engine._chk(self.engine.lib.cps_legacy_fleet_set_states(self.engine._h, s.ctypes.data_as(L._FP), int(period)))
        self._reset_period = int(period)

    def solves(self, period: int) -> bool:
        """Whether controller period `period` runs a solve (iteration % update_every == 0)."""
        if self._reset_period is None:
            raise RuntimeError("LegacyFleet: reset() first")
        return (period - self._reset_period) % self.update_every == 0

    def inputs(self):
        """(u, u_prev), each [E, T]: every experiment's nominal inputs (already shifted) and previous ones.  Synchronises."""
        u, up = np.zeros((self.E, self.T), np.float32), np.zeros((self.E, self.T), np.float32)
        self.engine.use_current_stream()
        self.engine._chk(self.engine.lib.cps_legacy_fleet_get_inputs(self.engine._h, u.ctypes.data_as(L._FP),
                                                                     up.ctypes.data_as(L._FP)))
        return u, up

    def _draw(self, name: str, period: int, shape) -> torch.Tensor:
        out = torch.empty(shape, device=self.device, dtype=torch.float32)
        self.engine.use_current_stream()
        self.engine._chk(self._fn(name)(self.engine._h, int(period), _ptr(out)))
        return out

    def draws(self, period: int) -> torch.Tensor:
        """The raw draws a 'philox' fleet uses in `period`: cuda tensor [E, K, n_draws] (standard normals, or uniforms in
        [-1, 1) for "uniform"; n_draws = T, 1 for "repeated", ceil(T / 10) + 1 for "interpolated")."""
        return self._draw("draws", period, (self.E, self.K, self.n_draws))

    def act_draws(self, period: int) -> torch.Tensor:
        """The actuator-noise uniforms in [-1, 1) of `period`: cuda tensor [E]."""
        return self._draw("act_draws", period, (self.E,))

    def perturbations(self, period: int) -> torch.Tensor:
        """The perturbations delta_u a 'philox' fleet's solve of `period` uses: cuda tensor [E, K, T]."""
        return self._draw("perturbations", period, (self.E, self.K, self.T))

    def run(self, n_periods: int, target_position=None, target_equilibrium=None, draws=None, act_draws=None, record=None,
            S_out=None):
        """cps_legacy_fleet_step: n_periods controller periods, no synchronisation.  target_position / target_equilibrium:
        cuda tensors [n_periods, E] or None; draws [n_periods, E, K, n_draws] and act_draws [n_periods, E] for a
        'supplied' fleet (draws are read in solve periods only); record [n_periods, E, 16] and S_out [n_periods, E, K]
        (rollout costs, written in solve periods) or None."""
        eng = self.engine
        p0 = self.period
        reads = any(self.solves(p0 + j) for j in range(n_periods)) if self._reset_period is not None else False
        if self.noise_source == "philox" and (draws is not None or act_draws is not None):
            raise ValueError("LegacyFleet: this fleet generates its draws (Philox); pass draws=None, act_draws=None")
        if self.noise_source == "supplied" and n_periods > 0 and (act_draws is None or (reads and draws is None)):
            raise ValueError("LegacyFleet: a 'supplied' fleet needs draws (in solve periods) and act_draws")
        self._check_rows(n_periods, target_position, target_equilibrium, record, S_out,
                         (draws, "draws", n_periods * self.E * self.K * self.n_draws),
                         (act_draws, "act_draws", n_periods * self.E))
        eng._chk(eng.lib.cps_legacy_fleet_step(eng._h, int(n_periods), _ptr(target_position), _ptr(target_equilibrium),
                                               _ptr(draws), _ptr(act_draws), _ptr(record), _ptr(S_out)))
        return record
