"""optimizer_mppi_b200 -- drop-in replacement for Control_Toolkit/Optimizers/optimizer_mppi.py:13-230.

Same constructor keywords, `configure`, `step(s, time) -> np scalar`, `optimizer_reset`, and the attributes other
code reads (`u_nom`, `u`, `rollout_trajectories`, `logging_values`, `optimal_trajectory`,
`optimal_control_sequence`, `num_rollouts`, `mpc_horizon`, `optimizer_name`).  The whole of
`_predict_and_cost` (:180-192), including the hidden-state update of a recurrent predictor (:191,194-196), runs as one
CUDA kernel launch (cps_mppi_step); predictors: ODE, ODE_v0 and neural (GRU / Dense); the predictor and cost-function
objects handed in are only inspected for their configuration (predictor type / substeps, cost plugin name and
weights, variable_parameters), so both this package's wrappers and the reference's own
PredictorWrapper / CostFunctionWrapper instances work.

Preserved semantics (SURVEY.md 8b): warm-start shift at the START of a solve repeating the last element (:183);
`u_old` given to the cost is the last RETURNED control, 0.0 initially (:210, Optimizers/__init__.py:35); clip before
the rollout and after the update (:186,:189); predictor.update is a no-op for ODE predictors
(predictor_wrapper.py:173-177); target_position / target_equilibrium / L / m_pole are re-read every step
(CartPole/__init__.py:512-519).
"""
from __future__ import annotations

import sys

import numpy as np
import torch

from . import _lib as L
from . import config as cfgmod
from .core import Engine
from .predictors import read_variable


class CudaNormalGenerator:
    """`rng.normal(shape, dtype)` like the reference's torch_gen_like_TF
    (Control_Toolkit/others/globals_and_utils.py:62-70), and `uniform` with the call shape of tf.random.Generator, both
    drawing on the device."""

    def __init__(self, seed, device):
        if seed is None:  # create_rng (:73-78): seed with the clock
            import time
            seed = int(time.time() * 1000.0) % (2 ** 63)
        self.seed = int(seed)
        self.device = device
        self.rng = torch.Generator(device=device).manual_seed(self.seed)

    def normal(self, shape, dtype=torch.float32):
        return torch.randn(tuple(shape), generator=self.rng, device=self.device, dtype=dtype)

    def uniform(self, shape, minval=0.0, maxval=1.0, dtype=torch.float32):
        out = torch.empty(tuple(shape), device=self.device, dtype=dtype)
        return out.uniform_(float(minval), float(maxval), generator=self.rng)


def _extract_cost(cost_function):
    """(plugin name, weight config or None) from this package's or the reference's CostFunctionWrapper."""
    name = getattr(cost_function, "cost_function_name", None)
    cf = getattr(cost_function, "cost_function", None)
    if name is None and cf is not None:
        name = type(cf).__name__
    if name is None and isinstance(cost_function, str):
        name = cost_function
    if name is None:
        raise ValueError("cannot determine the cost function plugin name; configure the CostFunctionWrapper first")
    name = name.replace("-", "_")
    cfg = None
    if cf is not None and isinstance(getattr(cf, "config", None), dict):
        cfg = dict(cf.config)  # *_grad* plugins and this package's plugins keep their YAML block here
    elif cf is not None:
        mod = sys.modules.get(type(cf).__module__)  # default / quadratic_boundary keep module-level constants
        keys = ("dd_weight", "ep_weight", "cc_weight", "ccrc_weight", "R")
        if mod is not None and all(hasattr(mod, k) for k in keys):
            cfg = {k: float(getattr(mod, k)) for k in keys}
    return name, cfg


def _extract_predictor(predictor, predictor_specification):
    """(integrator name 'ODE' | 'ODE_v0' | 'neural', intermediate_steps)."""
    ptype = getattr(predictor, "predictor_type", None)
    pcfg = getattr(predictor, "predictor_config", None) or {}
    if ptype is None and isinstance(predictor_specification, str):
        ptype = predictor_specification.split(":")[0]
    if ptype is None and isinstance(predictor, str):
        ptype = predictor
    n = int(pcfg.get("intermediate_steps", 10)) if hasattr(pcfg, "get") else 10
    inner = getattr(predictor, "predictor", None)
    if inner is not None and hasattr(inner, "intermediate_steps"):
        n = int(inner.intermediate_steps)
    return ptype, n


def _extract_net_spec(predictor):
    """The network of a configured neural predictor: this package's predictor_autoregressive_neural (net_spec) or the
    reference's own object (torch net + net_info + normalization_info)."""
    from . import neural
    inner = getattr(predictor, "predictor", predictor)
    net_spec = getattr(inner, "net_spec", None)
    if net_spec is None:
        if not hasattr(inner, "net_info"):
            raise ValueError("neural predictor: configure the PredictorWrapper before the optimizer "
                             "(controller_mpc.py:69-76 does)")
        net_spec = neural.spec_from_reference_predictor(inner)
    return net_spec


class _template_optimizer:
    """What the drop-ins share with the reference's template_optimizer (Control_Toolkit/Optimizers/__init__.py): the
    constructor attributes, configure, the variable / cost parameter refresh, the state check at the start of step, the
    draw rings and the pinned staging of the state.  A subclass sets PREDICTORS and PREDICTOR_REFUSAL, `_engine_kw`
    (Engine keywords) in its constructor, and may override `_set_mppi_params`."""
    supported_computation_libraries = ("Numpy", "TF", "Pytorch")
    PREDICTORS = ("ODE", "ODE_v0")           # predictor types configure accepts
    PREDICTOR_REFUSAL = NotImplementedError  # what configure raises for any other
    NOISE_RING = 256   # solves per device RNG call when the optimizer draws its own numbers

    def __init__(self, predictor, cost_function, control_limits, computation_library=None, seed=None,
                 mpc_horizon: int = 35, num_rollouts: int = 200, optimizer_logging: bool = False,
                 calculate_optimal_trajectory: bool = False, device=None, **kwargs):
        self.lib = computation_library
        self.num_rollouts = int(num_rollouts)
        self.mpc_horizon = int(mpc_horizon)
        self.cost_function = cost_function
        self.predictor = predictor
        self.u = 0.0  # template_optimizer.__init__ (Optimizers/__init__.py:35)
        self.num_states = None
        self.num_control_inputs = None
        lo, hi = control_limits
        self.action_low = np.asarray(lo, dtype=np.float32).reshape(-1)
        self.action_high = np.asarray(hi, dtype=np.float32).reshape(-1)
        self.seed = seed
        self.logging_values = {}
        self.optimizer_logging = bool(optimizer_logging)
        self._device_arg = device
        self._engine_kw = {}
        self.engine = None
        self.rng = None
        self._own_rng = None
        self._rings = {}
        self._var = None

    def _configure(self, num_states, num_control_inputs, dt, predictor_specification):
        name = type(self).__name__
        if int(num_control_inputs) != 1 or int(num_states) != 6:
            raise ValueError(f"{name} implements the CartPole path: 6 states, 1 control input")
        self.num_states, self.num_control_inputs = int(num_states), int(num_control_inputs)
        ptype, n = _extract_predictor(self.predictor, predictor_specification)
        if ptype not in self.PREDICTORS:
            raise self.PREDICTOR_REFUSAL(f"{name} supports the {' / '.join(self.PREDICTORS)} predictors, not {ptype!r} "
                                         "(no CPU fallback)")
        net_spec = _extract_net_spec(self.predictor) if ptype == "neural" else None
        cost_name, cost_cfg = _extract_cost(self.cost_function)
        self.dt = float(dt)
        self.engine = Engine(num_rollouts=self.num_rollouts, horizon=self.mpc_horizon, dt=self.dt, substeps=n,
                             integrator=ptype, cost=cost_name, device=self._device_arg, **self._engine_kw)
        self.device = self.engine.device
        self.cost_name, self.predictor_type = cost_name, ptype
        if net_spec is not None:
            self.engine.net_load(net_spec)
        self.engine.set_cost_params(cfgmod.cost_vector(cost_name, cost_cfg))
        self._set_mppi_params()
        self._own_rng = CudaNormalGenerator(self.seed, self.device)
        self.rng = self._own_rng
        self._s_dev = torch.zeros(6, device=self.device)
        self._s_pin = torch.zeros(6, pin_memory=torch.cuda.is_available())
        self._var = None
        self._configure_engine()

    def _set_mppi_params(self):
        # only the control limits of this block are used by the planners
        self.engine.set_mppi_params(lo=float(self.action_low[0]), hi=float(self.action_high[0]))

    def _configure_engine(self):
        pass

    @property
    def optimizer_name(self):
        return self.__class__.__name__.replace("optimizer_", "").replace("_", "-").lower()

    def _refresh_variable_parameters(self):
        vp = getattr(self.cost_function, "variable_parameters", None)
        if vp is None:
            vp = getattr(getattr(self.cost_function, "cost_function", None), "variable_parameters", None)
        var = (read_variable(vp, "target_position", 0.0), read_variable(vp, "target_equilibrium", 1.0),
               read_variable(vp, "L", cfgmod.DEFAULT_PHYSICS["L"]),
               read_variable(vp, "m_pole", cfgmod.DEFAULT_PHYSICS["m_pole"]))
        if var != self._var:
            self.engine.set_variable_parameters(*var)
            self._var = var

    def refresh_cost_parameters(self):
        """Call after the cost plugin's weights changed (the reference's hot reload re-reads the YAML into the plugin,
        cost_function_wrapper.py:71-74); re-uploads them to the kernel parameter block."""
        _, cfg = _extract_cost(self.cost_function)
        self.engine.set_cost_params(cfgmod.cost_vector(self.cost_name, cfg))

    def _state(self, s):
        """The start of every step: s as 6 float32, the logging record started, the variable parameters re-read."""
        if self.engine is None:
            raise RuntimeError(f"{type(self).__name__}.step called before configure")
        s = np.asarray(s, dtype=np.float32).reshape(-1)
        if s.shape[0] != 6:
            raise ValueError(f"state must have 6 entries, got {s.shape[0]}")
        if self.optimizer_logging:
            self.logging_values = {"s_logged": s.copy()}
        self._refresh_variable_parameters()
        return s

    def _state_dev(self, s):
        """s on the device through pinned staging: the copy is stream-ordered, no synchronisation."""
        self._s_pin.copy_(torch.from_numpy(s))
        self._s_dev.copy_(self._s_pin, non_blocking=True)
        return self._s_dev

    def _u_prev(self):
        return float(np.asarray(self.u).reshape(-1)[0])

    def _ring_draw(self, kind, shape, *args):
        """One solve's draws (tensor of the tuple `shape`) from the own generator's `kind` ('normal' or 'uniform' with `args`), out
        of a ring per kind that one generator call fills for up to NOISE_RING solves (64 MiB at most): a device RNG launch
        costs ~8 us of host time, a good part of a solve at these sizes."""
        r = self._rings.get(kind)   # [draws, solves in the ring, next solve, shape]: the check stays in plain Python
        if r is None or r[2] == r[1] or r[3] != shape:
            n = max(1, min(self.NOISE_RING, (64 << 20) // (4 * int(np.prod(shape)))))
            r = self._rings[kind] = [getattr(self._own_rng, kind)((n,) + shape, *args), n, 0, shape]
        r[2] += 1
        return r[0][r[2] - 1]


class optimizer_mppi_b200(_template_optimizer):
    PREDICTORS = ("ODE", "ODE_v0", "neural")
    PREDICTOR_REFUSAL = ValueError

    def __init__(self, predictor, cost_function, control_limits, computation_library=None, seed=None,
                 cc_weight: float = 1.0, R: float = 1.0, LBD: float = 100.0, mpc_horizon: int = 35,
                 num_rollouts: int = 3500, NU: float = 1000.0, SQRTRHOINV: float = 0.03,
                 period_interpolation_inducing_points: int = 10, optimizer_logging: bool = False,
                 calculate_optimal_trajectory: bool = False, device=None, fast_sincos: bool = False,
                 exact_atan2: bool = False, materialize_rollouts: bool | None = None, **kwargs):
        super().__init__(predictor, cost_function, control_limits, computation_library, seed, mpc_horizon, num_rollouts,
                         optimizer_logging, device=device)
        self.cc_weight, self.R, self.LBD, self.NU, self._SQRTRHOINV = cc_weight, R, LBD, NU, SQRTRHOINV
        self.period_interpolation_inducing_points = int(period_interpolation_inducing_points)
        self.calculate_optimal_trajectory = bool(calculate_optimal_trajectory)
        self.optimal_trajectory = None
        self.materialize_rollouts = self.optimizer_logging if materialize_rollouts is None else bool(materialize_rollouts)
        self._engine_kw = dict(noise_mode="inducing", interp_period=self.period_interpolation_inducing_points,
                               fast_sincos=fast_sincos, exact_atan2=exact_atan2)
        self._J = self._traj = self._u_run = None

    # --------------------------------------------------------------------------------------------------
    def configure(self, num_states: int, num_control_inputs: int, dt: float, predictor_specification: str = None,
                  **kwargs):
        self._configure(num_states, num_control_inputs, dt, predictor_specification)
        self.optimizer_reset()

    def _set_mppi_params(self):
        self.engine.set_mppi_params(self.cc_weight, self.R, self.LBD, self.NU, self._SQRTRHOINV,
                                    float(self.action_low[0]), float(self.action_high[0]))

    def _configure_engine(self):
        self.SQRTRHODTINV = np.float32(np.array(self._SQRTRHOINV) * (1 / np.sqrt(self.dt)))
        self.number_of_interpolation_inducing_points = self.engine.n_ind

    # u_nom lives on the device inside the handle; expose the reference's [1, T, 1] tensor view on demand
    @property
    def u_nom(self):
        return torch.from_numpy(self.engine.get_u_nom()).reshape(1, self.mpc_horizon, 1)

    @u_nom.setter
    def u_nom(self, value):
        v = value.detach().cpu().numpy() if isinstance(value, torch.Tensor) else np.asarray(value)
        self.engine.set_u_nom(v.reshape(-1))

    @property
    def optimal_control_sequence(self):
        """numpy [1, T, 1] copy of u_nom (optimizer_mppi.py:219), fetched from the device when read."""
        if self.engine is None:
            return None
        return self.engine.get_u_nom().reshape(1, self.mpc_horizon, 1)

    @property
    def rollout_trajectories(self):
        return self._traj

    def optimizer_reset(self):
        """u_nom = 0.5 (lo + hi) (optimizer_mppi.py:226-230).  The stored hidden state of a recurrent predictor is
        NOT reset, as in the reference."""
        self.engine.mppi_reset(0.5 * float(self.action_low[0] + self.action_high[0]))

    def _draw_noise(self):
        K, n_ind = self.num_rollouts, self.engine.n_ind
        if self.rng is self._own_rng:
            return self._ring_draw("normal", (n_ind, K)), L.TIME_MAJOR
        # a caller-supplied generator (e.g. injected draws): reference call shape and layout (:172-174)
        eps = self.rng.normal([K, n_ind, 1], dtype=torch.float32)
        eps = torch.as_tensor(eps).to(device=self.device, dtype=torch.float32).reshape(K, n_ind).contiguous()
        return eps, L.ROLLOUT_MAJOR

    # --------------------------------------------------------------------------------------------------
    def step(self, s: np.ndarray, time=None):
        s = self._state(s)
        noise, layout = self._draw_noise()
        u_prev = self._u_prev()
        h_before = None
        if self.calculate_optimal_trajectory and self.predictor_type == "neural" and self.engine.net_htot:
            h_before = torch.from_numpy(self.engine.net_get_state()).to(self.device)
        if self.materialize_rollouts or self.optimizer_logging:
            K, T = self.num_rollouts, self.mpc_horizon
            if self._J is None:
                self._J = torch.empty(K, device=self.device)
                self._traj = torch.empty((K, T + 1, 6), device=self.device)
                self._u_run = torch.empty((K, T, 1), device=self.device)
            u_dev = self.engine.mppi_step(self._state_dev(s), noise, layout, u_prev, None, self._J, self._traj,
                                          L.ROLLOUT_MAJOR, self._u_run)
            u = float(u_dev.cpu()[0])
        else:
            u = self.engine.mppi_step_host(s, noise, layout, u_prev)
        self.u = np.array(u, dtype=np.float32)
        if self.optimizer_logging:
            self.logging_values["Q_logged"] = self._u_run.cpu().numpy()
            self.logging_values["J_logged"] = self._J.cpu().numpy()
            self.logging_values["rollout_trajectories_logged"] = self._traj.cpu().numpy()
            self.logging_values["u_logged"] = self.u
        if self.calculate_optimal_trajectory:  # _predict_optimal_trajectory (:198-201): nominal rollout from s
            un = torch.from_numpy(self.engine.get_u_nom().reshape(1, -1)).to(self.device)
            s_dev = self._state_dev(s)
            if self.predictor_type == "neural":
                # the reference's batch-1 predictor copy rolls out from its own hidden state and advances it AFTER
                # predicting (:198-201), i.e. from the state before this solve's update
                traj, _ = self.engine.net_rollout(s_dev, un, h0=h_before)
            else:
                traj, _ = self.engine.rollout(s_dev, un)
            self.optimal_trajectory = traj.cpu().numpy()
        return self.u
