"""ctypes loader of libcps_b200.so (the C ABI declared in include/cps.h).

There is no CPU fallback: if the library has not been built, or it cannot be loaded, importing callers get
a RuntimeError that says how to build it.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
# CPS_B200_LIB: another build of the same library (kernel A/B measurements, tools/); the product is the in-tree file
_SO = os.environ.get("CPS_B200_LIB") or os.path.join(_PKG, "libcps_b200.so")
_CSRC = os.path.join(_PKG, "csrc")

CPS_OK = 0
STATUS_NAMES = {0: "CPS_OK", 1: "CPS_ERR_INVALID", 2: "CPS_ERR_CUDA", 3: "CPS_ERR_UNSUPPORTED",
                4: "CPS_ERR_NOT_CONFIGURED"}

EULER_V0, EULER_CROMER, PREDICTOR_NEURAL = 0, 1, 2
NET_GRU, NET_DENSE, NET_MAX_LAYERS = 0, 1, 4
COST_NONE, COST_DEFAULT, COST_QUADRATIC_BOUNDARY, COST_QB_GRAD_MINIMAL, COST_QB_GRAD = -1, 0, 1, 2, 3
COST_LEGACY_MPPI = 4
NOISE_INDUCING, NOISE_DIRECT = 0, 1
ROLLOUT_MAJOR, TIME_MAJOR = 0, 1
FLAG_FAST_SINCOS, FLAG_EXACT_ATAN2, FLAG_FAST_DIV, FLAG_SUBSTEP_SINCOS = 0x1, 0x2, 0x4, 0x8
FLAG_NET_TENSOR_CORES, FLAG_NET_FP32, FLAG_NO_PAIRS = 0x10, 0x20, 0x40
PAIR_MIN_BATCH = 262144
PH_COUNT = 9
FLEET_NOISE_SUPPLIED, FLEET_NOISE_PHILOX, FLEET_RECORD = 0, 1, 16
FLEET_RECORD_COLUMNS = ("time", "angle", "angleD", "angleDD", "angle_cos", "angle_sin", "position", "positionD",
                        "positionDD", "Q_calculated", "Q_applied", "u", "target_position", "target_equilibrium")


class cps_config(C.Structure):
    _fields_ = [("struct_size", C.c_int), ("device", C.c_int), ("num_rollouts", C.c_int), ("horizon", C.c_int),
                ("substeps", C.c_int), ("dt", C.c_float), ("integrator", C.c_int), ("cost_id", C.c_int),
                ("noise_mode", C.c_int), ("interp_period", C.c_int), ("flags", C.c_uint)]


class cps_net_desc(C.Structure):
    _fields_ = [("struct_size", C.c_int), ("net_type", C.c_int), ("n_layers", C.c_int),
                ("hidden", C.c_int * 4), ("n_state_in", C.c_int), ("in_idx", C.c_int * 6), ("n_out", C.c_int),
                ("out_idx", C.c_int * 6), ("norm_a", C.c_float * 7), ("norm_b", C.c_float * 7),
                ("denorm_A", C.c_float * 6), ("denorm_B", C.c_float * 6), ("differential", C.c_int),
                ("diff_p1", C.c_float * 6), ("diff_p2", C.c_float * 6), ("out_norm_a", C.c_float * 6),
                ("out_norm_b", C.c_float * 6), ("out_to_in", C.c_int * 6)]


class cps_fleet_config(C.Structure):
    _fields_ = [("struct_size", C.c_int), ("n_experiments", C.c_int), ("sim_substeps", C.c_int),
                ("noise_source", C.c_int), ("dt_simulation", C.c_double), ("seed", C.c_ulonglong),
                ("experiment_offset", C.c_longlong)]


class cps_fleet_plant_models(C.Structure):
    _fields_ = [("struct_size", C.c_int), ("control_noise_mode", C.c_int), ("control_noise_mult", C.c_float),
                ("control_noise_add", C.c_float), ("measurement_noise", C.c_int), ("sigma_angle", C.c_float),
                ("sigma_position", C.c_float), ("sigma_angleD", C.c_float), ("sigma_positionD", C.c_float),
                ("latency", C.c_double)]


class cps_rpgd_fleet_config(C.Structure):
    _fields_ = [("struct_size", C.c_int), ("n_experiments", C.c_int), ("sim_substeps", C.c_int),
                ("draw_source", C.c_int), ("dt_simulation", C.c_double), ("seed", C.c_ulonglong),
                ("experiment_offset", C.c_longlong), ("outer_its", C.c_int), ("first_iter_count", C.c_int),
                ("resamp_per", C.c_int), ("opt_keep_k", C.c_int), ("shift_previous", C.c_int),
                ("learning_rate", C.c_float), ("adam_beta_1", C.c_float), ("adam_beta_2", C.c_float),
                ("adam_epsilon", C.c_float), ("gradmax_clip", C.c_float), ("sample_stdev", C.c_float),
                ("sample_mean", C.c_float)]


class cps_cem_fleet_config(C.Structure):
    _fields_ = [("struct_size", C.c_int), ("n_experiments", C.c_int), ("sim_substeps", C.c_int),
                ("draw_source", C.c_int), ("dt_simulation", C.c_double), ("seed", C.c_ulonglong),
                ("experiment_offset", C.c_longlong), ("outer_its", C.c_int), ("first_iter_count", C.c_int),
                ("best_k", C.c_int), ("initial_stdev", C.c_float), ("stdev_min", C.c_float)]


class cps_cem_gmm_fleet_config(C.Structure):
    _fields_ = [("struct_size", C.c_int), ("n_experiments", C.c_int), ("sim_substeps", C.c_int),
                ("draw_source", C.c_int), ("dt_simulation", C.c_double), ("seed", C.c_ulonglong),
                ("experiment_offset", C.c_longlong), ("outer_its", C.c_int), ("best_k", C.c_int),
                ("initial_stdev", C.c_float), ("stdev_min", C.c_float)]


class cps_random_action_fleet_config(C.Structure):
    _fields_ = [("struct_size", C.c_int), ("n_experiments", C.c_int), ("sim_substeps", C.c_int),
                ("draw_source", C.c_int), ("dt_simulation", C.c_double), ("seed", C.c_ulonglong),
                ("experiment_offset", C.c_longlong)]


class cps_legacy_fleet_config(C.Structure):
    _fields_ = [("struct_size", C.c_int), ("n_experiments", C.c_int), ("sim_substeps", C.c_int),
                ("draw_source", C.c_int), ("dt_simulation", C.c_double), ("seed", C.c_ulonglong),
                ("experiment_offset", C.c_longlong), ("sampling_type", C.c_int), ("update_every", C.c_int),
                ("stdev", C.c_double), ("p_Q", C.c_double)]


# name -> (restype, argtypes); every symbol include/cps.h declares
_FP = C.POINTER(C.c_float)
_VP = C.c_void_p
SYMBOLS = {
    "cps_create": (C.c_int, [C.POINTER(cps_config), C.POINTER(_VP)]),
    "cps_destroy": (None, [_VP]),
    "cps_last_error": (C.c_char_p, [_VP]),
    "cps_abi_version": (C.c_int, []),
    "cps_num_inducing_points": (C.c_int, [C.c_int, C.c_int]),
    "cps_set_stream": (C.c_int, [_VP, _VP]),
    "cps_set_physics": (C.c_int, [_VP, _FP, C.c_int]),
    "cps_set_cost_params": (C.c_int, [_VP, _FP, C.c_int]),
    "cps_set_mppi_params": (C.c_int, [_VP] + [C.c_float] * 7),
    "cps_set_variable_parameters": (C.c_int, [_VP] + [C.c_float] * 4),
    "cps_mppi_step": (C.c_int, [_VP, _VP, _VP, C.c_int, C.c_float, _VP, _VP, _VP, _VP, C.c_int, _VP]),
    "cps_mppi_step_host": (C.c_int, [_VP, _FP, _VP, C.c_int, C.c_float, _FP]),
    "cps_mppi_reset": (C.c_int, [_VP, C.c_float]),
    "cps_mppi_get_u_nom": (C.c_int, [_VP, _FP]),
    "cps_mppi_set_u_nom": (C.c_int, [_VP, _FP]),
    "cps_mppi_u_nom_dev": (_VP, [_VP]),
    "cps_mppi_set_shard": (C.c_int, [_VP, C.c_int, _VP]),
    "cps_mppi_partial_size": (C.c_int, [_VP]),
    "cps_mppi_finalize": (C.c_int, [_VP, _VP, C.c_int, _VP, _VP]),
    "cps_mppi_peer_buffer_floats": (C.c_longlong, [_VP, C.c_int]),
    "cps_mppi_set_peers": (C.c_int, [_VP, C.c_int, C.c_int, C.POINTER(_VP)]),
    "cps_mppi_peer_timeouts": (C.c_int, [_VP, C.POINTER(C.c_int)]),
    "cps_legacy_step": (C.c_int, [_VP, _VP, _VP, C.c_int, _VP, _VP, _VP, C.c_int, _VP]),
    "cps_legacy_step_host": (C.c_int, [_VP, _FP, _VP, C.c_int, _FP]),
    "cps_legacy_step_host_knots": (C.c_int, [_VP, _FP, _VP, C.c_int, C.c_int, _FP]),
    "cps_legacy_get_perturbations": (C.c_int, [_VP, _VP]),
    "cps_legacy_advance": (C.c_int, [_VP, _FP]),
    "cps_legacy_reset": (C.c_int, [_VP]),
    "cps_legacy_get_inputs": (C.c_int, [_VP, _FP, _FP]),
    "cps_legacy_set_inputs": (C.c_int, [_VP, _FP, _FP]),
    "cps_rollout": (C.c_int, [_VP, _VP, C.c_int, _VP, C.c_int, C.c_int, C.c_int, _VP, C.c_int, _VP]),
    "cps_rollout_host": (C.c_int, [_VP, _VP, C.c_int, _VP, C.c_int, C.c_int, C.c_int, _VP, C.c_int, _VP]),
    "cps_net_load": (C.c_int, [_VP, C.POINTER(cps_net_desc), _FP, C.c_longlong]),
    "cps_net_rollout": (C.c_int, [_VP, _VP, C.c_int, _VP, C.c_int, C.c_int, C.c_int, _VP, C.c_int, _VP, C.c_int, _VP]),
    "cps_net_update": (C.c_int, [_VP, _VP, _VP]),
    "cps_net_state_size": (C.c_int, [_VP]),
    "cps_net_reset_state": (C.c_int, [_VP]),
    "cps_net_get_state": (C.c_int, [_VP, _FP]),
    "cps_net_set_state": (C.c_int, [_VP, _FP]),
    "cps_trajectory_cost": (C.c_int, [_VP, _VP, _VP, C.c_float, C.c_int, C.c_int, _VP]),
    "cps_stage_cost": (C.c_int, [_VP, _VP, C.c_int, _VP, C.c_float, C.c_int, C.c_int, C.c_int, _VP]),
    "cps_terminal_cost": (C.c_int, [_VP, _VP, C.c_int, _VP]),
    "cps_fleet_create": (C.c_int, [_VP, C.POINTER(cps_fleet_config)]),
    "cps_fleet_set_states": (C.c_int, [_VP, _FP, C.c_longlong]),
    "cps_fleet_get_states": (C.c_int, [_VP, _FP, _FP, _FP]),
    "cps_fleet_period": (C.c_longlong, [_VP]),
    "cps_fleet_step": (C.c_int, [_VP, C.c_int, _VP, _VP, _VP, _VP, _VP]),
    "cps_fleet_set_plant_models": (C.c_int, [_VP, C.POINTER(cps_fleet_plant_models)]),
    "cps_fleet_get_observed": (C.c_int, [_VP, _FP]),
    "cps_fleet_step_noisy": (C.c_int, [_VP, C.c_int, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "cps_fleet_relabel": (C.c_int, [_VP, C.c_int, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "cps_fleet_relabel_masked": (C.c_int, [_VP, C.c_int, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "cps_fleet_reset": (C.c_int, [_VP, C.c_longlong]),
    "cps_fleet_noise": (C.c_int, [_VP, C.c_longlong, _VP]),
    "cps_fleet_get_net_states": (C.c_int, [_VP, _FP]),
    "cps_fleet_set_net_states": (C.c_int, [_VP, _FP]),
    "cps_rpgd_fleet_create": (C.c_int, [_VP, C.POINTER(cps_rpgd_fleet_config)]),
    "cps_rpgd_fleet_set_states": (C.c_int, [_VP, _FP, _VP, C.c_longlong]),
    "cps_rpgd_fleet_step": (C.c_int, [_VP, C.c_int, _VP, _VP, _VP, _VP, _VP, _VP]),
    "cps_rpgd_fleet_relabel": (C.c_int, [_VP, C.c_int, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "cps_rpgd_fleet_get_states": (C.c_int, [_VP, _FP, _FP]),
    "cps_rpgd_fleet_get_plans": (C.c_int, [_VP, _FP, _FP, _FP, C.POINTER(C.c_int), C.POINTER(C.c_longlong),
                                           C.POINTER(C.c_longlong)]),
    "cps_rpgd_fleet_period": (C.c_longlong, [_VP]),
    "cps_rpgd_fleet_draws": (C.c_int, [_VP, C.c_longlong, _VP]),
    "cps_cem_fleet_create": (C.c_int, [_VP, C.POINTER(cps_cem_fleet_config)]),
    "cps_cem_fleet_set_states": (C.c_int, [_VP, _FP, C.c_longlong]),
    "cps_cem_fleet_get_states": (C.c_int, [_VP, _FP, _FP]),
    "cps_cem_fleet_get_distribution": (C.c_int, [_VP, _FP, _FP]),
    "cps_cem_fleet_step": (C.c_int, [_VP, C.c_int, _VP, _VP, _VP, _VP, _VP, _VP]),
    "cps_cem_fleet_draws": (C.c_int, [_VP, C.c_longlong, _VP]),
    "cps_cem_fleet_period": (C.c_longlong, [_VP]),
    "cps_cem_gmm_fleet_create": (C.c_int, [_VP, C.POINTER(cps_cem_gmm_fleet_config)]),
    "cps_cem_gmm_fleet_set_states": (C.c_int, [_VP, _FP, C.c_longlong]),
    "cps_cem_gmm_fleet_get_states": (C.c_int, [_VP, _FP, _FP]),
    "cps_cem_gmm_fleet_get_distribution": (C.c_int, [_VP, _FP, _FP, _FP]),
    "cps_cem_gmm_fleet_step": (C.c_int, [_VP, C.c_int, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "cps_cem_gmm_fleet_draws": (C.c_int, [_VP, C.c_longlong, _VP, _VP]),
    "cps_cem_gmm_fleet_period": (C.c_longlong, [_VP]),
    "cps_random_action_fleet_create": (C.c_int, [_VP, C.POINTER(cps_random_action_fleet_config)]),
    "cps_random_action_fleet_set_states": (C.c_int, [_VP, _FP, C.c_longlong]),
    "cps_random_action_fleet_get_states": (C.c_int, [_VP, _FP, _FP]),
    "cps_random_action_fleet_step": (C.c_int, [_VP, C.c_int, _VP, _VP, _VP, _VP, _VP, _VP]),
    "cps_random_action_fleet_draws": (C.c_int, [_VP, C.c_longlong, _VP]),
    "cps_random_action_fleet_period": (C.c_longlong, [_VP]),
    "cps_legacy_fleet_create": (C.c_int, [_VP, C.POINTER(cps_legacy_fleet_config)]),
    "cps_legacy_fleet_set_states": (C.c_int, [_VP, _FP, C.c_longlong]),
    "cps_legacy_fleet_get_states": (C.c_int, [_VP, _FP, _FP]),
    "cps_legacy_fleet_get_inputs": (C.c_int, [_VP, _FP, _FP]),
    "cps_legacy_fleet_step": (C.c_int, [_VP, C.c_int, _VP, _VP, _VP, _VP, _VP, _VP]),
    "cps_legacy_fleet_draws": (C.c_int, [_VP, C.c_longlong, _VP]),
    "cps_legacy_fleet_act_draws": (C.c_int, [_VP, C.c_longlong, _VP]),
    "cps_legacy_fleet_perturbations": (C.c_int, [_VP, C.c_longlong, _VP]),
    "cps_legacy_fleet_period": (C.c_longlong, [_VP]),
    "cps_plan_cost": (C.c_int, [_VP, _VP, _VP, C.c_int, C.c_int, C.c_int, C.c_float, _VP, _VP, C.c_int]),
    "cps_plan_random_action": (C.c_int, [_VP, _VP, _VP, C.c_int, C.c_float, _VP, _VP, _VP]),
    "cps_plan_random_action_host": (C.c_int, [_VP, _FP, _VP, C.c_int, C.c_float, _FP]),
    "cps_cem_configure": (C.c_int, [_VP, C.c_int, C.c_float, C.c_float]),
    "cps_cem_reset": (C.c_int, [_VP]),
    "cps_cem_step": (C.c_int, [_VP, _VP, _VP, C.c_int, C.c_int, C.c_float, _VP, _VP, _VP]),
    "cps_cem_step_host": (C.c_int, [_VP, _FP, _VP, C.c_int, C.c_int, C.c_float, _FP]),
    "cps_cem_get_distribution": (C.c_int, [_VP, _FP, _FP]),
    "cps_cem_set_distribution": (C.c_int, [_VP, _FP, _FP]),
    "cps_cem_gmm_configure": (C.c_int, [_VP, C.c_int, C.c_float, C.c_float]),
    "cps_cem_gmm_reset": (C.c_int, [_VP]),
    "cps_cem_gmm_step": (C.c_int, [_VP, _VP, _VP, _VP, C.c_int, C.c_int, C.c_float, _VP, _VP, _VP]),
    "cps_cem_gmm_step_host": (C.c_int, [_VP, _FP, _VP, _VP, C.c_int, C.c_int, C.c_float, _FP]),
    "cps_cem_gmm_get_distribution": (C.c_int, [_VP, _FP, _FP, _FP]),
    "cps_cem_gmm_set_distribution": (C.c_int, [_VP, _FP, _FP, _FP]),
    "cps_measure_peaks": (C.c_int, [_VP, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "cps_selftest_sincos": (C.c_int, [_VP, C.POINTER(C.c_longlong)]),
    "cps_plan_cost_grad": (C.c_int, [_VP, _VP, _VP, C.c_int, C.c_float, _VP, _VP]),
    "cps_rpgd_reset": (C.c_int, [_VP]),
    "cps_rpgd_grad_step": (C.c_int, [_VP, _VP, _VP] + [C.c_float] * 6 + [_VP]),
    "cps_rpgd_adam_state": (C.c_int, [_VP, C.POINTER(_VP), C.POINTER(_VP), C.POINTER(C.c_longlong)]),
    "cps_rpgd_set_iterations": (C.c_int, [_VP, C.c_longlong]),
    "cps_rpgd_finish": (C.c_int, [_VP, _VP, _VP, _VP, C.c_int, C.c_int, _VP, _VP]),
    "cps_launch_count": (C.c_longlong, [_VP]),
    "cps_net_last_kernel": (C.c_int, [_VP]),
    "cps_rollout_last_kernel": (C.c_int, [_VP]),
    "cps_nonfinite_costs": (C.c_int, [_VP, C.POINTER(C.c_int)]),
}


def library_path() -> str:
    return _SO


def build(verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into the in-tree libcps_b200.so (nvcc cross-compiles without a GPU)."""
    out = subprocess.run(["make", "-j4", "-C", _CSRC], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout[-4000:])
        print(out.stderr[-4000:])
    if out.returncode != 0:
        raise RuntimeError("building libcps_b200.so failed")
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            raise RuntimeError(
                f"{_SO} is missing: the CUDA extension has not been built.  Build it with "
                "`python -c 'import __graft_entry__ as g; g.build()'` (or `make -C cartpolesimulation_b200/csrc`). "
                "cartpolesimulation_b200 has no CPU fallback.")
        L = C.CDLL(_SO)
        for name, (res, args) in SYMBOLS.items():
            if os.environ.get("CPS_B200_LIB") and not hasattr(L, name):
                continue  # an older build under A/B measurement may lack the newest entry points
            fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        if L.cps_abi_version() != 1:
            raise RuntimeError("libcps_b200.so ABI version mismatch")
        _lib = L
    return _lib


class CpsError(RuntimeError):
    pass


def check(rc: int, handle=None):
    if rc == CPS_OK:
        return
    msg = lib().cps_last_error(handle)
    msg = msg.decode() if msg else ""
    name = STATUS_NAMES.get(rc, str(rc))
    if rc == 1:
        raise ValueError(f"{name}: {msg}")
    if rc == 3:
        raise NotImplementedError(f"{name}: {msg}")
    if rc == 4:
        raise RuntimeError(f"{name}: {msg}")
    raise CpsError(f"{name}: {msg}")
