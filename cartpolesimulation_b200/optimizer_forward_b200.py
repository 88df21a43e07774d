"""optimizer_random_action_b200, optimizer_cem_b200 and optimizer_cem_gmm_b200 -- the reference's forward-only optimizers
on the GPU (SURVEY.md 8f row f3).

Mirrors of Control_Toolkit/Optimizers/optimizer_random_action_tf.py:12-86 and optimizer_cem_tf.py:12-117: the same
constructor keywords, `configure`, `step(s, time) -> np scalar`, `optimizer_reset`, and the attributes other code
reads (`u`, `logging_values`, `num_rollouts`, `mpc_horizon`, `optimizer_name`; CEM: `dist_mue`, `stdev`, `count`).
`predict_and_cost` (predictor.predict_core + cost_function.get_trajectory_cost) and the selection on the sorted costs
run as one CUDA kernel launch per evaluation (cps_plan_random_action / cps_cem_step); a CEM solve is `cem_outer_it`
launches with no host round trip in between.  The predictor and cost-function objects handed in are only inspected
for their configuration, so this package's wrappers and the reference's own work alike.  ODE / ODE_v0 predictors (RPGD
also the neural predictor); no CPU fallback.

Semantics kept from the reference: `self.u` (the `u_prev` of the cost's control-change term) is the last RETURNED
control, 0.0 initially (Optimizers/__init__.py:35); CEM samples Q = clip(mean + normal * stdev) (:66-68), takes the
`cem_best_k` cheapest plans (ties: lowest index), updates mean / population stdev from them (:79-81), and only after
the last outer iteration clips the stdev to [cem_stdev_min, 1e8] and shifts both vectors (:96-99); the first call runs
`warmup_iterations` iterations when `warmup` is set (:93); u = elite_Q[0, 0] of the last iteration.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib as L
from . import config as cfgmod
from .core import Engine
from .optimizer_mppi_b200 import CudaNormalGenerator, _extract_cost, _extract_net_spec, _extract_predictor
from .predictors import read_variable


class CudaGenerator(CudaNormalGenerator):
    """normal / uniform draws on the device with the call shapes of tf.random.Generator."""

    def uniform(self, shape, minval=0.0, maxval=1.0, dtype=torch.float32):
        out = torch.empty(tuple(shape), device=self.device, dtype=dtype)
        return out.uniform_(float(minval), float(maxval), generator=self.rng)


class _forward_optimizer:
    supported_computation_libraries = ("Numpy", "TF", "Pytorch")
    PREDICTORS = ("ODE", "ODE_v0")   # predictor types configure accepts
    NOISE_RING = 256   # solves per device RNG call when the optimizer draws its own numbers

    def _ring_draw(self, shape, draw):
        """One solve's draws (tensor of `shape`) out of a ring filled by a single generator call per NOISE_RING solves:
        a device RNG launch costs ~8 us of host time, a good part of a solve at these sizes."""
        ring = getattr(self, "_ring", None)
        if ring is None or tuple(ring.shape[1:]) != tuple(shape) or self._ring_i >= ring.shape[0]:
            n = max(1, min(self.NOISE_RING, (64 << 20) // (4 * int(np.prod(shape)))))
            self._ring = draw((n,) + tuple(shape))
            self._ring_i = 0
        out = self._ring[self._ring_i]
        self._ring_i += 1
        return out

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
        self.engine = None
        self.rng = None
        self._own_rng = None
        self._var = None

    def configure(self, num_states: int, num_control_inputs: int, default_configure: bool = True, dt: float = None,
                  predictor_specification: str = None, **kwargs):
        if int(num_control_inputs) != 1 or int(num_states) != 6:
            raise ValueError(f"{type(self).__name__} implements the CartPole path: 6 states, 1 control input")
        self.num_states, self.num_control_inputs = int(num_states), int(num_control_inputs)
        ptype, n = _extract_predictor(self.predictor, predictor_specification)
        if ptype not in self.PREDICTORS:
            raise NotImplementedError(f"{type(self).__name__} supports the {' / '.join(self.PREDICTORS)} predictors, not "
                                      f"{ptype!r} (no CPU fallback)")
        net_spec = _extract_net_spec(self.predictor) if ptype == "neural" else None
        if dt is None:
            dt = getattr(self.predictor, "dt", None) or 0.02
        cost_name, cost_cfg = _extract_cost(self.cost_function)
        self.dt = float(dt)
        self.engine = Engine(num_rollouts=self.num_rollouts, horizon=self.mpc_horizon, dt=self.dt, substeps=n,
                             integrator=ptype, cost=cost_name, device=self._device_arg)
        self.device = self.engine.device
        self.cost_name, self.predictor_type = cost_name, ptype
        if net_spec is not None:
            self.engine.net_load(net_spec)
        self.engine.set_cost_params(cfgmod.cost_vector(cost_name, cost_cfg))
        # only the control limits of this block are used by the planners
        self.engine.set_mppi_params(lo=float(self.action_low[0]), hi=float(self.action_high[0]))
        self._own_rng = CudaGenerator(self.seed, self.device)
        self.rng = self._own_rng
        self._var = None
        self._configure_engine()
        if default_configure:
            self.optimizer_reset()

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
        _, cfg = _extract_cost(self.cost_function)
        self.engine.set_cost_params(cfgmod.cost_vector(self.cost_name, cfg))

    def _state(self, s):
        if self.engine is None:
            raise RuntimeError(f"{type(self).__name__}.step called before configure")
        s = np.asarray(s, dtype=np.float32).reshape(-1)
        if s.shape[0] != 6:
            raise ValueError(f"state must have 6 entries, got {s.shape[0]}")
        if self.optimizer_logging:
            self.logging_values = {"s_logged": s.copy()}
        self._refresh_variable_parameters()
        return s

    def _log_rollouts(self, s, Q_kt):
        """Q_logged / J_logged / rollout_trajectories_logged of the reference: a second evaluation of the final plans
        with the trajectories materialised (logging only; not on the control path)."""
        u_prev = float(np.asarray(self._u_prev_logged).reshape(-1)[0])
        J, traj = self.engine.plan_cost(torch.from_numpy(s).to(self.device), Q_kt.contiguous(), L.ROLLOUT_MAJOR, u_prev,
                                        want_traj=True)
        self.logging_values["Q_logged"] = Q_kt.cpu().numpy()[:, :, None]
        self.logging_values["J_logged"] = J.cpu().numpy()
        self.logging_values["rollout_trajectories_logged"] = traj.cpu().numpy()
        self.logging_values["u_logged"] = self.u


class optimizer_random_action_b200(_forward_optimizer):
    """optimizer_random_action_tf: K uniform random plans, the cheapest one's first input."""

    def _draw(self):
        K, T = self.num_rollouts, self.mpc_horizon
        lo, hi = float(self.action_low[0]), float(self.action_high[0])
        if self.rng is self._own_rng:
            return self._ring_draw((T, K), lambda shp: self._own_rng.uniform(shp, lo, hi)), L.TIME_MAJOR
        Q = self.rng.uniform(shape=[K, T, 1], minval=lo, maxval=hi, dtype=torch.float32)  # reference call (:58-63)
        return torch.as_tensor(Q).to(device=self.device, dtype=torch.float32).reshape(K, T).contiguous(), L.ROLLOUT_MAJOR

    def step(self, s: np.ndarray, time=None):
        s = self._state(s)
        Q, layout = self._draw()
        self._u_prev_logged = self.u
        u = self.engine.plan_random_action_host(s, Q, layout, float(np.asarray(self.u).reshape(-1)[0]))
        self.u = np.array(u, dtype=np.float32)
        if self.optimizer_logging:
            self._log_rollouts(s, Q.t() if layout == L.TIME_MAJOR else Q)
        return self.u

    def optimizer_reset(self):
        if self.rng is not None and self.rng is self._own_rng:
            self._draw()  # the reference draws (and discards) one batch here (:81-86), advancing the generator


class optimizer_cem_b200(_forward_optimizer):
    """optimizer_cem_tf: cross-entropy method with a per-step Gaussian over the input plan."""

    def __init__(self, predictor, cost_function, control_limits, computation_library=None, seed=None,
                 mpc_horizon: int = 35, cem_outer_it: int = 3, cem_initial_action_stdev: float = 0.5,
                 num_rollouts: int = 200, cem_stdev_min: float = 0.01, cem_best_k: int = 40, warmup: bool = False,
                 warmup_iterations: int = 250, optimizer_logging: bool = False,
                 calculate_optimal_trajectory: bool = False, device=None, **kwargs):
        super().__init__(predictor=predictor, cost_function=cost_function, control_limits=control_limits,
                         computation_library=computation_library, seed=seed, mpc_horizon=mpc_horizon,
                         num_rollouts=num_rollouts, optimizer_logging=optimizer_logging,
                         calculate_optimal_trajectory=calculate_optimal_trajectory, device=device)
        self.cem_outer_it = int(cem_outer_it)
        self.cem_initial_action_stdev = float(cem_initial_action_stdev)
        self.cem_stdev_min = float(cem_stdev_min)
        self.cem_best_k = int(cem_best_k)
        self.warmup = bool(warmup)
        self.warmup_iterations = int(warmup_iterations)
        self.count = 0

    def _configure_engine(self):
        self.engine.cem_configure(self.cem_best_k, self.cem_initial_action_stdev, self.cem_stdev_min)

    # the distribution lives on the device inside the handle; the reference's [1, T, 1] tensors on demand
    @property
    def dist_mue(self):
        return torch.from_numpy(self.engine.cem_get_distribution()[0]).reshape(1, self.mpc_horizon, 1)

    @dist_mue.setter
    def dist_mue(self, value):
        v = value.detach().cpu().numpy() if isinstance(value, torch.Tensor) else np.asarray(value)
        self.engine.cem_set_distribution(mean=v.reshape(-1))

    @property
    def stdev(self):
        return torch.from_numpy(self.engine.cem_get_distribution()[1]).reshape(1, self.mpc_horizon, 1)

    @stdev.setter
    def stdev(self, value):
        v = value.detach().cpu().numpy() if isinstance(value, torch.Tensor) else np.asarray(value)
        self.engine.cem_set_distribution(stdev=v.reshape(-1))

    def _draw(self, iterations):
        K, T = self.num_rollouts, self.mpc_horizon
        if self.rng is self._own_rng:
            if iterations != self.cem_outer_it:   # the warm-up solve
                return self._own_rng.normal((iterations, T, K)), L.TIME_MAJOR
            return self._ring_draw((iterations, T, K), self._own_rng.normal), L.TIME_MAJOR
        eps = [torch.as_tensor(self.rng.normal(shape=(K, T, 1), dtype=torch.float32)).reshape(K, T)
               for _ in range(iterations)]  # one reference-shaped call per outer iteration (:66-67)
        return torch.stack(eps).to(device=self.device, dtype=torch.float32).contiguous(), L.ROLLOUT_MAJOR

    def step(self, s: np.ndarray, time=None):
        s = self._state(s)
        iterations = self.warmup_iterations if self.warmup and self.count == 0 else self.cem_outer_it
        eps, layout = self._draw(iterations)
        u_prev = float(np.asarray(self.u).reshape(-1)[0])
        self._u_prev_logged = self.u
        if self.optimizer_logging:
            K, T = self.num_rollouts, self.mpc_horizon
            Q = torch.empty((T, K) if layout == L.TIME_MAJOR else (K, T), device=self.device)
            u_dev = self.engine.cem_step(torch.from_numpy(s).to(self.device), eps, layout, u_prev, Q_out=Q)
            u = float(u_dev.cpu()[0])
        else:
            u = self.engine.cem_step_host(s, eps, layout, u_prev)
        self.u = np.array(u, dtype=np.float32)
        if self.optimizer_logging:
            self._log_rollouts(s, Q.t() if layout == L.TIME_MAJOR else Q)
        self.count += 1
        return self.u

    def optimizer_reset(self):
        self.engine.cem_reset()
        self.count = 0
        self.u = 0.0


class optimizer_cem_gmm_b200(_forward_optimizer):
    """optimizer_cem_gmm_tf (Control_Toolkit/Optimizers/optimizer_cem_gmm_tf.py:14-140): CEM whose sampling distribution is
    a two-component Gaussian mixture per horizon step; the elites are clustered around the two cheapest plans.  Same
    constructor keywords; the mixture lives on the device (`engine.cem_gmm_get_distribution()`); `sampling_dist` exposes
    it in the reference's shapes (loc / scale [T, 1, 2], probs [2]).  cps_cem_gmm_step: three launches per outer iteration,
    no host round trip inside a solve.

    Draws: every (iteration, rollout, step) consumes two standard normals (one per component, as
    MixtureSameFamily.sample does) and one uniform that picks the component (index 0 iff u < probs[0]).  A caller-supplied
    generator is asked for `normal([K, T, 1, 2])` and `uniform([K, T, 1])` once per outer iteration."""

    def __init__(self, predictor, cost_function, control_limits, computation_library=None, seed=None,
                 mpc_horizon: int = 35, cem_outer_it: int = 3, cem_initial_action_stdev: float = 0.5,
                 num_rollouts: int = 200, cem_stdev_min: float = 0.01, cem_best_k: int = 40,
                 optimizer_logging: bool = False, calculate_optimal_trajectory: bool = False, device=None, **kwargs):
        super().__init__(predictor=predictor, cost_function=cost_function, control_limits=control_limits,
                         computation_library=computation_library, seed=seed, mpc_horizon=mpc_horizon,
                         num_rollouts=num_rollouts, optimizer_logging=optimizer_logging,
                         calculate_optimal_trajectory=calculate_optimal_trajectory, device=device)
        self.cem_outer_it = int(cem_outer_it)
        self.cem_initial_action_stdev = float(cem_initial_action_stdev)
        self.cem_stdev_min = float(cem_stdev_min)
        self.cem_best_k = int(cem_best_k)

    def _configure_engine(self):
        self.engine.cem_gmm_configure(self.cem_best_k, self.cem_initial_action_stdev, self.cem_stdev_min)

    @property
    def sampling_dist(self):
        loc, scale, p1 = self.engine.cem_gmm_get_distribution()
        T = self.mpc_horizon
        return dict(loc=torch.from_numpy(loc.T.copy()).reshape(T, 1, 2), scale=torch.from_numpy(scale.T.copy()).reshape(T, 1, 2),
                    probs=torch.tensor([p1, 1.0 - p1]))

    def _draw(self):
        K, T, it = self.num_rollouts, self.mpc_horizon, self.cem_outer_it
        if self.rng is self._own_rng:
            eps = self._ring_draw((it, 2, T, K), self._own_rng.normal)
            ring = getattr(self, "_uring", None)
            if ring is None or self._uring_i >= ring.shape[0]:
                n = max(1, min(self.NOISE_RING, (64 << 20) // (4 * it * T * K)))
                self._uring = self._own_rng.uniform((n, it, T, K))
                self._uring_i = 0
            u01 = self._uring[self._uring_i]
            self._uring_i += 1
            return eps, u01, L.TIME_MAJOR
        eps, u01 = [], []
        for _ in range(it):
            eps.append(torch.as_tensor(self.rng.normal(shape=(K, T, 1, 2), dtype=torch.float32)).reshape(K, T, 2))
            u01.append(torch.as_tensor(self.rng.uniform(shape=(K, T, 1), minval=0.0, maxval=1.0, dtype=torch.float32)).reshape(K, T))
        to = dict(device=self.device, dtype=torch.float32)
        return torch.stack(eps).to(**to).contiguous(), torch.stack(u01).to(**to).contiguous(), L.ROLLOUT_MAJOR

    def step(self, s: np.ndarray, time=None):
        s = self._state(s)
        eps, u01, layout = self._draw()
        u_prev = float(np.asarray(self.u).reshape(-1)[0])
        self._u_prev_logged = self.u
        if self.optimizer_logging:
            K, T = self.num_rollouts, self.mpc_horizon
            Q = torch.empty((T, K) if layout == L.TIME_MAJOR else (K, T), device=self.device)
            u_dev = self.engine.cem_gmm_step(torch.from_numpy(s).to(self.device), eps, u01, layout, u_prev, Q_out=Q)
            u = float(u_dev.cpu()[0])
        else:
            u = self.engine.cem_gmm_step_host(s, eps, u01, layout, u_prev)
        self.u = np.array(u, dtype=np.float32)
        if self.optimizer_logging:
            self._log_rollouts(s, Q.t() if layout == L.TIME_MAJOR else Q)
        return self.u

    def optimizer_reset(self):
        self.engine.cem_gmm_reset()


class optimizer_rpgd_b200(_forward_optimizer):
    """optimizer_rpgd_tf (Control_Toolkit/Optimizers/optimizer_rpgd_tf.py:15-420; `rpgd` is the reference's shipped
    default optimizer, Control_Toolkit_ASF/config_controllers.yml:2): resampling parallel gradient descent.  K input plans
    are improved by `outer_its` Adam steps on d(traj_cost)/dQ, the cheapest plan's first input is applied, all plans are
    shifted by `shift_previous` as the next warm start, and every `resamp_per` solves the worst K - opt_keep_k plans are
    replaced by fresh samples (their Adam moments zeroed, the kept ones' shifted).

    The gradient -- a GradientTape around predict_and_cost in the reference -- is one adjoint kernel launch
    (cps_rpgd_grad_step: gradient, clip_by_norm, Adam, clip to the limits); the plans and the Adam moments stay on the
    device, the per-solve bookkeeping of step() (:297-356: argsort of K costs, gather, shift) is a handful of torch index
    operations on those device tensors.  Predictors "ODE" and "neural" (plain GRU / Dense networks; differential D_* networks
    are not supported); cost quadratic_boundary_grad_minimal (the shipped configuration) or quadratic_boundary_grad; no CPU
    fallback.

    Hidden state of a recurrent network: step() does not advance it.  optimizer_rpgd_tf's predict_and_cost is
    predict_core + get_trajectory_cost (:167-168), whereas optimizer_mppi advances the memory inside its _predict_and_cost
    (optimizer_mppi.py:191); every rollout and gradient here starts from the stored hidden state of this optimizer's engine
    and leaves it as it was.  A caller that wants the memory to follow the plant calls `engine.net_update(s, u)` after each step."""

    PREDICTORS = ("ODE", "ODE_v0", "neural")

    def __init__(self, predictor, cost_function, control_limits, computation_library=None, seed=None,
                 mpc_horizon: int = 35, num_rollouts: int = 16, outer_its: int = 4, sample_stdev: float = 0.5,
                 sample_mean: float = 0.0, sample_whole_control_space: bool = False, uniform_dist_min: float = -0.8,
                 uniform_dist_max: float = 0.8, resamp_per: int = 10, period_interpolation_inducing_points: int = 4,
                 SAMPLING_DISTRIBUTION: str = "normal", shift_previous: int = 1, warmup: bool = False,
                 warmup_iterations: int = 250, learning_rate: float = 0.05, opt_keep_k_ratio: float = 0.75,
                 gradmax_clip: float = 5.0, rtol: float = 1e-3, adam_beta_1: float = 0.9, adam_beta_2: float = 0.999,
                 adam_epsilon: float = 1e-8, optimizer_logging: bool = False, calculate_optimal_trajectory: bool = False,
                 device=None, **kwargs):
        super().__init__(predictor=predictor, cost_function=cost_function, control_limits=control_limits,
                         computation_library=computation_library, seed=seed, mpc_horizon=mpc_horizon,
                         num_rollouts=num_rollouts, optimizer_logging=optimizer_logging,
                         calculate_optimal_trajectory=calculate_optimal_trajectory, device=device)
        if SAMPLING_DISTRIBUTION not in ("normal", "uniform"):
            raise ValueError(f"RPGD cannot interpret sampling type {SAMPLING_DISTRIBUTION}")
        self.outer_its, self.sample_stdev, self.sample_mean = int(outer_its), float(sample_stdev), float(sample_mean)
        if sample_whole_control_space:
            self.sample_min, self.sample_max = float(self.action_low[0]), float(self.action_high[0])
        else:
            self.sample_min, self.sample_max = float(uniform_dist_min), float(uniform_dist_max)
        self.resamp_per, self.shift_previous = int(resamp_per), int(shift_previous)
        self.period_interpolation_inducing_points = int(period_interpolation_inducing_points)
        self.SAMPLING_DISTRIBUTION = SAMPLING_DISTRIBUTION
        self.first_iter_count = int(warmup_iterations) if warmup else self.outer_its
        self.opt_keep_k = int(max(int(self.num_rollouts * opt_keep_k_ratio), 1))
        self.learning_rate, self.gradmax_clip, self.rtol = float(learning_rate), float(gradmax_clip), float(rtol)
        self.adam_beta_1, self.adam_beta_2, self.adam_epsilon = float(adam_beta_1), float(adam_beta_2), float(adam_epsilon)
        self.calculate_optimal_trajectory = bool(calculate_optimal_trajectory)
        self.optimal_trajectory = self.optimal_control_sequence = self.u_nom = None
        self.count = 0

    def _configure_engine(self):
        K, T, p = self.num_rollouts, self.mpc_horizon, self.period_interpolation_inducing_points
        n_ind = int(self.engine.lib.cps_num_inducing_points(T, p))
        # Interpolator.calculate_interpolation_matrix (Control_Toolkit/others/Interpolator.py:54-78): tent weights, the last
        # inducing point enters its own step with weight 1 / p
        W = np.zeros(((n_ind - 1) * p + 1, n_ind), dtype=np.float32)
        for i in range(n_ind - 1):
            for j in range(p):
                W[i * p + j, i], W[i * p + j, i + 1] = p - j, j
        W[-1, -1] = 1
        self._W = torch.from_numpy((W[:T] / np.float32(p)).T.copy()).to(self.device)   # [n_ind, T]
        self.number_of_interpolation_inducing_points = n_ind
        self.Q_tf = torch.zeros((K, T), device=self.device)
        self.trajectory_ages = torch.zeros(K, dtype=torch.int32, device=self.device)

    def sample_actions(self, batch_size: int):
        """:149-171: draws at the inducing points, clipped, then interpolated over the horizon."""
        n_ind = self.number_of_interpolation_inducing_points
        if self.SAMPLING_DISTRIBUTION == "normal":
            if self.rng is self._own_rng:
                Qn = self.rng.normal((batch_size, n_ind)) * self.sample_stdev + self.sample_mean
            else:
                Qn = torch.as_tensor(self.rng.normal([batch_size, n_ind, 1], mean=self.sample_mean, stddev=self.sample_stdev,
                                                     dtype=torch.float32)).reshape(batch_size, n_ind)
        else:
            Qn = torch.as_tensor(self.rng.uniform([batch_size, n_ind, 1], minval=self.sample_min, maxval=self.sample_max,
                                                  dtype=torch.float32)).reshape(batch_size, n_ind)
        Qn = Qn.to(device=self.device, dtype=torch.float32).clamp(float(self.action_low[0]), float(self.action_high[0]))
        return Qn @ self._W

    def step(self, s: np.ndarray, time=None):
        s = self._state(s)
        K, T, keep = self.num_rollouts, self.mpc_horizon, self.opt_keep_k
        if getattr(self, "_s_pin", None) is None:   # pinned staging: the state's copy is stream-ordered, no synchronisation
            self._s_pin = torch.empty(6, dtype=torch.float32).pin_memory()
            self._s_dev = torch.empty(6, dtype=torch.float32, device=self.device)
        self._s_pin.copy_(torch.from_numpy(s))
        self._s_dev.copy_(self._s_pin, non_blocking=True)
        s_dev = self._s_dev
        u_prev = float(np.asarray(self.u).reshape(-1)[0])
        for _ in range(self.first_iter_count if self.count == 0 else self.outer_its):   # grad_step (:166-180)
            self.engine.rpgd_grad_step(s_dev, self.Q_tf, u_prev, self.learning_rate, self.adam_beta_1, self.adam_beta_2,
                                       self.adam_epsilon, self.gradmax_clip)
        # get_action (:182-224): costs of the improved plans, the best opt_keep_k of them, the shifted warm start
        J = self.engine.plan_cost(s_dev, self.Q_tf, L.ROLLOUT_MAJOR, u_prev)[0]
        if self.optimizer_logging:
            self._u_prev_logged = self.u
            self._log_rollouts(s, self.Q_tf)
            self.logging_values["trajectory_ages_logged"] = self.trajectory_ages.cpu().numpy()
        resample = self.count % self.resamp_per == 0
        if K <= 4096 and not (resample and keep == K):
            # one launch: stable order of the costs, the cheapest plan, shift, resampling permutation of plans / moments / ages
            fresh = self.sample_actions(K - keep).contiguous() if resample else None
            u_nom = self.engine.rpgd_finish(J, self.Q_tf, fresh, keep, self.shift_previous, self.trajectory_ages)
            self.optimal_control_sequence = u_nom.reshape(1, T, 1)
            self.u_nom = torch.from_numpy(self.optimal_control_sequence)   # host view; moved to the device only where needed
        else:
            best_idx = torch.sort(J, stable=True).indices[:keep]
            self.u_nom = self.Q_tf[best_idx[0]].clone().reshape(1, T, 1)
            sp = self.shift_previous
            Qn = torch.cat([self.Q_tf[:, sp:], self.Q_tf[:, -1:].repeat(1, sp)], dim=1)
            self.optimal_control_sequence = self.u_nom.cpu().numpy()
            m, v, _ = self.engine.rpgd_adam_state()
            zeros = torch.zeros((K, 1), device=self.device)
            if resample:   # :299-343: the worst plans are redrawn, the kept ones sorted by cost
                Qn = torch.cat([self.sample_actions(K - keep), Qn[best_idx]], dim=0)
                self.trajectory_ages = torch.cat([torch.zeros(K - keep, dtype=torch.int32, device=self.device),
                                                  self.trajectory_ages[best_idx]])
                fresh = torch.zeros((K - keep, T), device=self.device)
                m.copy_(torch.cat([fresh, torch.cat([m[best_idx][:, 1:], zeros[:keep]], dim=1)], dim=0))
                v.copy_(torch.cat([fresh, torch.cat([v[best_idx][:, 1:], zeros[:keep]], dim=1)], dim=0))
            else:                                   # :344-356: every plan keeps its moments, shifted by one step
                m.copy_(torch.cat([m[:, 1:], zeros], dim=1))
                v.copy_(torch.cat([v[:, 1:], zeros], dim=1))
            self.trajectory_ages += 1
            self.Q_tf.copy_(Qn)
        self.count += 1
        if self.calculate_optimal_trajectory:
            u_nom = self.u_nom.reshape(1, T).to(self.device)
            if self.predictor_type == "neural":
                traj, _ = self.engine.net_rollout(s_dev, u_nom)
            else:
                traj, _ = self.engine.rollout(s_dev, u_nom)
            self.optimal_trajectory = traj.cpu().numpy()
        self.u = np.array(self.optimal_control_sequence[0, 0, 0], dtype=np.float32)   # already on the host: no second sync
        return self.u

    def optimizer_reset(self):
        """:379-408: fresh plans, Adam moments and iteration count zeroed."""
        self.Q_tf.copy_(self.sample_actions(self.num_rollouts))
        self.count = 0
        self.engine.rpgd_reset()
        self.trajectory_ages.zero_()
