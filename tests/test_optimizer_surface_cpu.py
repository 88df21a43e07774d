"""The drop-in optimizers' public surface, frozen: constructor, configure and step signatures (names, order, defaults) and
the public attributes right after construction, which controller_mpc and user code read.  Needs no GPU."""
import inspect

import numpy as np
import pytest

SURFACE = {
    'optimizer_mppi_b200': dict(
        __init__='predictor cost_function control_limits computation_library=None seed=None cc_weight=1.0 R=1.0 '
                 'LBD=100.0 mpc_horizon=35 num_rollouts=3500 NU=1000.0 SQRTRHOINV=0.03 '
                 'period_interpolation_inducing_points=10 optimizer_logging=False calculate_optimal_trajectory=False '
                 'device=None fast_sincos=False exact_atan2=False materialize_rollouts=None **kwargs',
        configure='num_states num_control_inputs dt predictor_specification=None **kwargs',
        step='s time=None',
        attributes='LBD NU R action_high action_low calculate_optimal_trajectory cc_weight cost_function engine lib '
                   'logging_values materialize_rollouts mpc_horizon num_control_inputs num_rollouts num_states '
                   'optimal_trajectory optimizer_logging period_interpolation_inducing_points predictor rng seed u'),
    'optimizer_random_action_b200': dict(
        __init__='predictor cost_function control_limits computation_library=None seed=None mpc_horizon=35 '
                 'num_rollouts=200 optimizer_logging=False calculate_optimal_trajectory=False device=None **kwargs',
        configure='num_states num_control_inputs default_configure=True dt=None predictor_specification=None **kwargs',
        step='s time=None',
        attributes='action_high action_low cost_function engine lib logging_values mpc_horizon num_control_inputs '
                   'num_rollouts num_states optimizer_logging predictor rng seed u'),
    'optimizer_cem_b200': dict(
        __init__='predictor cost_function control_limits computation_library=None seed=None mpc_horizon=35 '
                 'cem_outer_it=3 cem_initial_action_stdev=0.5 num_rollouts=200 cem_stdev_min=0.01 cem_best_k=40 '
                 'warmup=False warmup_iterations=250 optimizer_logging=False calculate_optimal_trajectory=False '
                 'device=None **kwargs',
        configure='num_states num_control_inputs default_configure=True dt=None predictor_specification=None **kwargs',
        step='s time=None',
        attributes='action_high action_low cem_best_k cem_initial_action_stdev cem_outer_it cem_stdev_min cost_function '
                   'count engine lib logging_values mpc_horizon num_control_inputs num_rollouts num_states '
                   'optimizer_logging predictor rng seed u warmup warmup_iterations'),
    'optimizer_cem_gmm_b200': dict(
        __init__='predictor cost_function control_limits computation_library=None seed=None mpc_horizon=35 '
                 'cem_outer_it=3 cem_initial_action_stdev=0.5 num_rollouts=200 cem_stdev_min=0.01 cem_best_k=40 '
                 'optimizer_logging=False calculate_optimal_trajectory=False device=None **kwargs',
        configure='num_states num_control_inputs default_configure=True dt=None predictor_specification=None **kwargs',
        step='s time=None',
        attributes='action_high action_low cem_best_k cem_initial_action_stdev cem_outer_it cem_stdev_min cost_function '
                   'engine lib logging_values mpc_horizon num_control_inputs num_rollouts num_states optimizer_logging '
                   'predictor rng seed u'),
    'optimizer_rpgd_b200': dict(
        __init__='predictor cost_function control_limits computation_library=None seed=None mpc_horizon=35 '
                 'num_rollouts=16 outer_its=4 sample_stdev=0.5 sample_mean=0.0 sample_whole_control_space=False '
                 'uniform_dist_min=-0.8 uniform_dist_max=0.8 resamp_per=10 period_interpolation_inducing_points=4 '
                 "SAMPLING_DISTRIBUTION='normal' shift_previous=1 warmup=False warmup_iterations=250 "
                 'learning_rate=0.05 opt_keep_k_ratio=0.75 gradmax_clip=5.0 rtol=0.001 adam_beta_1=0.9 '
                 'adam_beta_2=0.999 adam_epsilon=1e-08 optimizer_logging=False calculate_optimal_trajectory=False '
                 'device=None **kwargs',
        configure='num_states num_control_inputs default_configure=True dt=None predictor_specification=None **kwargs',
        step='s time=None',
        attributes='SAMPLING_DISTRIBUTION action_high action_low adam_beta_1 adam_beta_2 adam_epsilon '
                   'calculate_optimal_trajectory cost_function count engine first_iter_count gradmax_clip learning_rate '
                   'lib logging_values mpc_horizon num_control_inputs num_rollouts num_states opt_keep_k '
                   'optimal_control_sequence optimal_trajectory optimizer_logging outer_its '
                   'period_interpolation_inducing_points predictor resamp_per rng rtol sample_max sample_mean sample_min '
                   'sample_stdev seed shift_previous u u_nom'),
}


def _classes():
    from cartpolesimulation_b200 import optimizer_forward_b200 as F
    from cartpolesimulation_b200.optimizer_mppi_b200 import optimizer_mppi_b200
    return {c.__name__: c for c in (optimizer_mppi_b200, F.optimizer_random_action_b200, F.optimizer_cem_b200,
                                    F.optimizer_cem_gmm_b200, F.optimizer_rpgd_b200)}


def _signature(f):
    out = []
    for p in list(inspect.signature(f).parameters.values())[1:]:   # without self
        if p.kind is p.VAR_KEYWORD:
            out.append("**" + p.name)
        else:
            out.append(p.name if p.default is inspect.Parameter.empty else f"{p.name}={p.default!r}")
    return out


@pytest.mark.parametrize("name", sorted(SURFACE))
def test_signatures(name):
    cls = _classes()[name]
    for method in ("__init__", "configure", "step"):
        assert _signature(getattr(cls, method)) == SURFACE[name][method].split(), method


@pytest.mark.parametrize("name", sorted(SURFACE))
def test_public_attributes_after_init(name):
    limits = (np.array([-1.0], np.float32), np.array([1.0], np.float32))
    opt = _classes()[name](predictor="ODE", cost_function="quadratic_boundary_grad_minimal", control_limits=limits)
    assert sorted(k for k in vars(opt) if not k.startswith("_")) == SURFACE[name]["attributes"].split()
    assert opt.u == 0.0 and opt.engine is None and opt.rng is None and opt.logging_values == {}
