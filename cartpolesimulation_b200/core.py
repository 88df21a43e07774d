"""Thin Python object around one cps_handle (include/cps.h).  Device memory, streams and pointers come
from torch (plumbing); all arithmetic happens in libcps_b200.so.  No CPU fallback."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib as L
from . import config as cfgmod


def _ptr(t):
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def _check_dev(t, name, device, dtype=torch.float32):
    if not isinstance(t, torch.Tensor) or t.device != device:
        raise ValueError(f"{name} must be a torch tensor on {device}")
    if t.dtype != dtype:
        raise ValueError(f"{name} must be {dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    return t


def _check_sizes(device, *checks):
    """_check_dev and the element count of every (tensor, name, numel) whose tensor is not None."""
    for t, name, numel in checks:
        if t is not None:
            _check_dev(t, name, device)
            if t.numel() != numel:
                raise ValueError(f"{name} has {t.numel()} elements, expected {numel}")


INTEGRATORS = {"ODE_v0": L.EULER_V0, "ODE": L.EULER_CROMER, "neural": L.PREDICTOR_NEURAL}
COSTS = {None: L.COST_NONE, "none": L.COST_NONE, "default": L.COST_DEFAULT,
         "quadratic_boundary": L.COST_QUADRATIC_BOUNDARY,
         "quadratic_boundary_grad_minimal": L.COST_QB_GRAD_MINIMAL,
         "quadratic_boundary_grad": L.COST_QB_GRAD,
         "legacy_mppi": L.COST_LEGACY_MPPI}  # q() + phi() of controller_mppi_cartpole (legacy front-end)


class Engine:
    """One configured rollout engine = one cps_handle.

    Parameters mirror what controller_mpc.configure wires together
    (Control_Toolkit/Controllers/controller_mpc.py:42-92): K rollouts, horizon T, n substeps, dt,
    integrator ('ODE_v0' | 'ODE'), cost plugin name, noise mode.
    """

    def __init__(self, num_rollouts: int, horizon: int, dt: float = 0.02, substeps: int = 10,
                 integrator: str = "ODE", cost: str | None = "quadratic_boundary_grad_minimal",
                 noise_mode: str = "inducing", interp_period: int = 10, device: int | None = None,
                 fast_sincos: bool = False, exact_atan2: bool = False, fast_div: bool = False,
                 substep_sincos: bool = False, net_kernel: str | None = None, no_pairs: bool = False):
        if integrator not in INTEGRATORS:
            raise ValueError(f"unknown integrator {integrator!r}; expected one of {list(INTEGRATORS)}")
        if cost not in COSTS:
            raise ValueError(f"unknown cost function {cost!r}; expected one of {list(COSTS)}")
        if not torch.cuda.is_available():
            raise RuntimeError("cartpolesimulation_b200 needs a CUDA device (no CPU fallback)")
        self.lib = L.lib()
        dev = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", dev)
        if fast_sincos or exact_atan2:
            substep_sincos = True  # both only make sense when sin/cos are evaluated every substep
        flags = (L.FLAG_FAST_SINCOS if fast_sincos else 0) | (L.FLAG_EXACT_ATAN2 if exact_atan2 else 0) \
            | (L.FLAG_FAST_DIV if fast_div else 0) | (L.FLAG_SUBSTEP_SINCOS if substep_sincos else 0)
        if net_kernel not in (None, "tensor", "fp32"):
            raise ValueError("net_kernel must be None (choose by batch size), 'tensor' or 'fp32'")
        flags |= {None: 0, "tensor": L.FLAG_NET_TENSOR_CORES, "fp32": L.FLAG_NET_FP32}[net_kernel]
        flags |= L.FLAG_NO_PAIRS if no_pairs else 0
        self.K, self.T, self.n, self.dt, self.p = int(num_rollouts), int(horizon), int(substeps), float(dt), int(interp_period)
        self.integrator, self.cost_name = integrator, cost
        self.noise_mode = {"inducing": L.NOISE_INDUCING, "direct": L.NOISE_DIRECT}[noise_mode]
        c = L.cps_config(C.sizeof(L.cps_config), dev, self.K, self.T, self.n, self.dt, INTEGRATORS[integrator],
                         COSTS[cost], self.noise_mode, self.p, flags)
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            torch.cuda.init()
            L.check(self.lib.cps_create(C.byref(c), C.byref(h)), None)
        self._h = h
        self.n_ind = self.lib.cps_num_inducing_points(self.T, self.p)
        self.n_noise = self.n_ind if self.noise_mode == L.NOISE_INDUCING else self.T
        self._stream = None
        self._u_dev = torch.zeros(1, device=self.device)
        self._s_dev = torch.zeros(6, device=self.device)
        self._u_host = (C.c_float * 1)()
        self._s_host = (C.c_float * 6)()

    # -- lifetime -------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self.lib.cps_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        L.check(rc, self._h)

    def _s_host_from(self, s_np):
        """The host-form entry points' state argument: s_np's 6 entries as float32 in a buffer the handle reads."""
        for i in range(6):
            self._s_host[i] = s_np[i]
        return self._s_host

    def use_current_stream(self):
        s = torch.cuda.current_stream(self.device).cuda_stream
        if s != self._stream:
            self._chk(self.lib.cps_set_stream(self._h, C.c_void_p(s)))
            self._stream = s

    # -- parameters -----------------------------------------------------------------------------------
    def set_physics(self, **params):
        v = cfgmod.physics_vector(**params)
        self._chk(self.lib.cps_set_physics(self._h, v.ctypes.data_as(L._FP), len(v)))
        u_max = float(v[cfgmod.PHYS_ORDER.index("u_max")])
        if u_max != getattr(self, "_u_max", 1.77):
            # MAX_COST of the shifted plugins contains u_max^2 (default.py:20, quadratic_boundary.py:23): keep it in step
            self._u_max = u_max
            if getattr(self, "_cost_cfg_set", False):
                self.set_cost_config(self._cost_cfg)

    def set_cost_params(self, vec):
        v = np.ascontiguousarray(vec, dtype=np.float32)
        self._chk(self.lib.cps_set_cost_params(self._h, v.ctypes.data_as(L._FP), len(v)))

    def set_cost_config(self, cfg: dict | None = None):
        self._cost_cfg, self._cost_cfg_set = cfg, True
        self.set_cost_params(cfgmod.cost_vector(self.cost_name, cfg, u_max=getattr(self, "_u_max", 1.77)))

    def set_mppi_params(self, cc_weight=1.0, R=1.0, LBD=100.0, NU=1000.0, SQRTRHOINV=0.03, lo=-1.0, hi=1.0):
        sigma = np.float32(np.array(SQRTRHOINV) * (1 / np.sqrt(self.dt)))  # optimizer_mppi.py:130
        self._chk(self.lib.cps_set_mppi_params(self._h, cc_weight, R, LBD, NU, float(sigma), lo, hi))

    def set_variable_parameters(self, target_position=0.0, target_equilibrium=1.0, L=0.395, m_pole=0.087):
        self._chk(self.lib.cps_set_variable_parameters(self._h, float(target_position), float(target_equilibrium),
                                                        float(np.float32(L)), float(np.float32(m_pole))))

    # -- MPPI -----------------------------------------------------------------------------------------
    def noise_shape(self, layout=L.TIME_MAJOR):
        return (self.n_noise, self.K) if layout == L.TIME_MAJOR else (self.K, self.n_noise)

    def mppi_step(self, s, noise, noise_layout=L.TIME_MAJOR, u_prev=0.0, u_nom=None, J_out=None, traj_out=None,
                  traj_layout=L.ROLLOUT_MAJOR, u_run_out=None):
        """Device-pointer form (cps_mppi_step).  s: cuda tensor [6]; noise: cuda tensor of noise_shape(layout);
        u_nom: cuda tensor [T] updated in place (default: the handle's own).  Returns the cuda tensor [1]
        holding u (no synchronisation)."""
        self.use_current_stream()
        _check_dev(s, "s", self.device)
        _check_dev(noise, "noise", self.device)
        if tuple(noise.shape[:2]) != self.noise_shape(noise_layout) or noise.numel() != self.n_noise * self.K:
            raise ValueError(f"noise has shape {tuple(noise.shape)}, expected {self.noise_shape(noise_layout)}")
        unom_ptr = self.lib.cps_mppi_u_nom_dev(self._h) if u_nom is None else _check_dev(u_nom, "u_nom", self.device).data_ptr()
        _check_sizes(self.device, (J_out, "J_out", self.K), (traj_out, "traj_out", self.K * (self.T + 1) * 6),
                     (u_run_out, "u_run_out", self.K * self.T))
        self._chk(self.lib.cps_mppi_step(self._h, _ptr(s), _ptr(noise), noise_layout, float(u_prev),
                                         C.c_void_p(unom_ptr), _ptr(self._u_dev), _ptr(J_out), _ptr(traj_out),
                                         traj_layout, _ptr(u_run_out)))
        return self._u_dev

    def mppi_step_host(self, s_np, noise, noise_layout=L.TIME_MAJOR, u_prev=0.0) -> float:
        """Host form (cps_mppi_step_host): numpy state in, python float control out; synchronises."""
        self.use_current_stream()
        _check_dev(noise, "noise", self.device)
        if noise.numel() != self.n_noise * self.K:
            raise ValueError(f"noise has {noise.numel()} elements, expected {self.n_noise * self.K}")
        self._chk(self.lib.cps_mppi_step_host(self._h, self._s_host_from(s_np), _ptr(noise), noise_layout, float(u_prev),
                                              self._u_host))
        return self._u_host[0]

    def mppi_reset(self, value=0.0):
        self.use_current_stream()
        self._chk(self.lib.cps_mppi_reset(self._h, float(value)))

    def get_u_nom(self) -> np.ndarray:
        self.use_current_stream()
        out = np.zeros(self.T, dtype=np.float32)
        self._chk(self.lib.cps_mppi_get_u_nom(self._h, out.ctypes.data_as(L._FP)))
        return out

    def set_u_nom(self, u_nom):
        self.use_current_stream()
        v = np.ascontiguousarray(np.asarray(u_nom, dtype=np.float32).reshape(-1))
        if v.shape[0] != self.T:
            raise ValueError(f"u_nom has {v.shape[0]} entries, expected {self.T}")
        self._chk(self.lib.cps_mppi_set_u_nom(self._h, v.ctypes.data_as(L._FP)))

    # -- legacy front-end (controller_mppi_cartpole) ------------------------------------------------
    def legacy_step(self, s, delta_u, layout=L.ROLLOUT_MAJOR, S_out=None, traj_out=None, traj_layout=L.ROLLOUT_MAJOR,
                    u_upd_out=None):
        """Device-pointer form (cps_legacy_step).  s: cuda [6]; delta_u: cuda K x T in `layout` order.  Returns the cuda
        tensor [1] holding u[0] after the update (no synchronisation)."""
        self.use_current_stream()
        _check_dev(s, "s", self.device)
        _check_dev(delta_u, "delta_u", self.device)
        if delta_u.numel() != self.K * self.T:
            raise ValueError(f"delta_u has {delta_u.numel()} elements, expected {self.K * self.T}")
        _check_sizes(self.device, (S_out, "S_out", self.K), (traj_out, "traj_out", self.K * (self.T + 1) * 6),
                     (u_upd_out, "u_upd_out", self.T))
        self._chk(self.lib.cps_legacy_step(self._h, _ptr(s), _ptr(delta_u), layout, _ptr(self._u_dev), _ptr(S_out),
                                           _ptr(traj_out), traj_layout, _ptr(u_upd_out)))
        return self._u_dev

    def legacy_step_host(self, s_np, delta_u_np, layout=L.ROLLOUT_MAJOR) -> float:
        """Host form (cps_legacy_step_host): numpy state and numpy float32 perturbations in, python float out."""
        self.use_current_stream()
        if delta_u_np.dtype != np.float32 or not delta_u_np.flags.c_contiguous or delta_u_np.size != self.K * self.T:
            raise ValueError(f"delta_u must be a C-contiguous float32 array of {self.K * self.T} elements")
        self._chk(self.lib.cps_legacy_step_host(self._h, self._s_host_from(s_np), C.c_void_p(delta_u_np.ctypes.data), layout,
                                                self._u_host))
        return self._u_host[0]

    def legacy_step_host_knots(self, s_np, knots_np, knot_step: int) -> float:
        """cps_legacy_step_host_knots: the "interpolated" sampler's knot draws [K, n_knots] (float32) in, python float out;
        the perturbations between the knots are interpolated on the device."""
        self.use_current_stream()
        if knots_np.dtype != np.float32 or not knots_np.flags.c_contiguous or knots_np.ndim != 2 or knots_np.shape[0] != self.K:
            raise ValueError(f"knots must be a C-contiguous float32 array [K = {self.K}, n_knots]")
        self._chk(self.lib.cps_legacy_step_host_knots(self._h, self._s_host_from(s_np), C.c_void_p(knots_np.ctypes.data),
                                                      int(knots_np.shape[1]), int(knot_step), self._u_host))
        return self._u_host[0]

    def legacy_get_perturbations(self) -> np.ndarray:
        """delta_u [K, T] of the last host-form legacy step (cps_legacy_get_perturbations)."""
        self.use_current_stream()
        out = np.empty((self.K, self.T), dtype=np.float32)
        self._chk(self.lib.cps_legacy_get_perturbations(self._h, C.c_void_p(out.ctypes.data)))
        return out

    def legacy_advance(self) -> float:
        self.use_current_stream()
        self._chk(self.lib.cps_legacy_advance(self._h, self._u_host))
        return self._u_host[0]

    def legacy_reset(self):
        self.use_current_stream()
        self._chk(self.lib.cps_legacy_reset(self._h))

    def legacy_get_inputs(self):
        self.use_current_stream()
        u, up = np.zeros(self.T, np.float32), np.zeros(self.T, np.float32)
        self._chk(self.lib.cps_legacy_get_inputs(self._h, u.ctypes.data_as(L._FP), up.ctypes.data_as(L._FP)))
        return u, up

    def legacy_set_inputs(self, u=None, u_prev=None):
        self.use_current_stream()
        ptrs = []
        for v in (u, u_prev):
            if v is None:
                ptrs.append(None)
                continue
            v = np.ascontiguousarray(np.asarray(v, dtype=np.float32).reshape(-1))
            if v.shape[0] != self.T:
                raise ValueError(f"expected {self.T} entries, got {v.shape[0]}")
            ptrs.append(v)
        self._chk(self.lib.cps_legacy_set_inputs(self._h, *[None if v is None else v.ctypes.data_as(L._FP) for v in ptrs]))

    def partial_size(self):
        return self.lib.cps_mppi_partial_size(self._h)

    def set_shard(self, partial_out):
        if partial_out is None:
            self._chk(self.lib.cps_mppi_set_shard(self._h, 0, None))
        else:
            _check_dev(partial_out, "partial_out", self.device)
            if partial_out.numel() < self.partial_size():
                raise ValueError("partial_out too small")
            self._chk(self.lib.cps_mppi_set_shard(self._h, 1, _ptr(partial_out)))
        self._shard_buf = partial_out

    def peer_buffer_floats(self, world: int) -> int:
        return int(self.lib.cps_mppi_peer_buffer_floats(self._h, int(world)))

    def set_peers(self, world: int, rank: int, peer_ptrs):
        """K sharded over `world` GPUs with the exchange inside the solve launch (cps_mppi_set_peers): peer_ptrs[r] is the
        device address, as mapped on this GPU, of rank r's zero-initialised exchange buffer of peer_buffer_floats(world)
        floats.  None / world <= 1 switches it off."""
        if peer_ptrs is None or world <= 1:
            self._chk(self.lib.cps_mppi_set_peers(self._h, 0, 0, None))
            return
        arr = (C.c_void_p * int(world))(*[int(p) for p in peer_ptrs])
        self._chk(self.lib.cps_mppi_set_peers(self._h, int(world), int(rank), arr))

    def peer_timeouts(self) -> int:
        n = C.c_int(0)
        self._chk(self.lib.cps_mppi_peer_timeouts(self._h, C.byref(n)))
        return int(n.value)

    def mppi_finalize(self, partials, u_nom=None):
        self.use_current_stream()
        _check_dev(partials, "partials", self.device)
        n = partials.numel() // self.partial_size()
        unom_ptr = self.lib.cps_mppi_u_nom_dev(self._h) if u_nom is None else u_nom.data_ptr()
        self._chk(self.lib.cps_mppi_finalize(self._h, _ptr(partials), n, C.c_void_p(unom_ptr), _ptr(self._u_dev)))
        return self._u_dev

    # -- rollouts -------------------------------------------------------------------------------------
    def _rollout_io(self, s0, Q, q_layout, traj_layout, want_traj, traj_out):
        """(Q as 2-D, B, T, batched, traj_out) of a device rollout from s0 [6] (shared) or [B, 6]; traj_out allocated
        when wanted and not given."""
        _check_dev(s0, "s0", self.device)
        _check_dev(Q, "Q", self.device)
        Q2 = Q.reshape(Q.shape[0], Q.shape[1])
        B, T = (Q2.shape if q_layout == L.ROLLOUT_MAJOR else Q2.shape[::-1])
        if s0.numel() == 6:
            batched = 0
        elif s0.shape[0] == B and s0.numel() == 6 * B:
            batched = 1
        else:
            raise ValueError("Batch size of control input contradict batch size of initial state")
        if want_traj and traj_out is None:
            shape = (B, T + 1, 6) if traj_layout == L.ROLLOUT_MAJOR else (T + 1, 6, B)
            traj_out = torch.empty(shape, device=self.device, dtype=torch.float32)
        return Q2, B, T, batched, traj_out

    def rollout(self, s0, Q, q_layout=L.ROLLOUT_MAJOR, traj_layout=L.ROLLOUT_MAJOR, want_traj=True,
                want_final=False, traj_out=None, final_out=None):
        """cps_rollout on device tensors.  s0: [6] or [B,6]; Q: [B,T] (ROLLOUT_MAJOR) or [T,B] (TIME_MAJOR).
        Returns (traj, final): traj is [B,T+1,6] (ROLLOUT_MAJOR) or [T+1,6,B] (TIME_MAJOR)."""
        self.use_current_stream()
        Q2, B, T, batched, traj_out = self._rollout_io(s0, Q, q_layout, traj_layout, want_traj, traj_out)
        if want_final and final_out is None:
            final_out = torch.empty((B, 6), device=self.device, dtype=torch.float32)
        self._chk(self.lib.cps_rollout(self._h, _ptr(s0), batched, _ptr(Q2), q_layout, B, T, _ptr(traj_out),
                                       traj_layout, _ptr(final_out)))
        return traj_out, final_out

    def rollout_host(self, s0_np, Q_np, q_layout=L.ROLLOUT_MAJOR, traj_layout=L.ROLLOUT_MAJOR, traj_out=None,
                     final_out=None):
        """cps_rollout_host on host (numpy) buffers; synchronises.  Outputs are written into the given arrays."""
        self.use_current_stream()
        s0_np = np.ascontiguousarray(s0_np, dtype=np.float32)
        Q_np = np.ascontiguousarray(Q_np, dtype=np.float32)
        Q2 = Q_np.reshape(Q_np.shape[0], Q_np.shape[1])
        B, T = (Q2.shape if q_layout == L.ROLLOUT_MAJOR else Q2.shape[::-1])
        batched = 0 if s0_np.size == 6 else 1
        if batched and s0_np.shape[0] != B:
            raise ValueError("Batch size of control input contradict batch size of initial state")
        vp = lambda a: None if a is None else C.c_void_p(a.ctypes.data)
        self._chk(self.lib.cps_rollout_host(self._h, vp(s0_np), batched, vp(Q2), q_layout, B, T, vp(traj_out),
                                            traj_layout, vp(final_out)))
        return traj_out, final_out

    # -- neural predictor ------------------------------------------------------------------------------
    def net_load(self, spec: dict):
        """cps_net_load.  spec: dict(net_type 'GRU'|'Dense', hsz, weights (flat float32, include/cps.h order), in_idx,
        out_idx, norm_a, norm_b, denorm_A, denorm_B[, differential, diff_p1, diff_p2, out_norm_a, out_norm_b,
        out_to_in])."""
        d = L.cps_net_desc()
        d.struct_size = C.sizeof(L.cps_net_desc)
        if spec["net_type"] not in ("GRU", "Dense"):
            raise NotImplementedError(f"network type {spec['net_type']!r} is not supported (GRU and Dense are)")
        d.net_type = {"GRU": L.NET_GRU, "Dense": L.NET_DENSE}[spec["net_type"]]
        hsz = [int(x) for x in spec["hsz"]]
        if len(hsz) > L.NET_MAX_LAYERS:
            raise NotImplementedError(f"at most {L.NET_MAX_LAYERS} hidden layers are supported")
        d.n_layers = len(hsz)
        for i, v in enumerate(hsz):
            d.hidden[i] = v
        d.n_state_in, d.n_out = len(spec["in_idx"]), len(spec["out_idx"])
        for i, v in enumerate(spec["in_idx"]):
            d.in_idx[i] = int(v)
        for i, v in enumerate(spec["out_idx"]):
            d.out_idx[i] = int(v)
        for name in ("norm_a", "norm_b", "denorm_A", "denorm_B", "diff_p1", "diff_p2", "out_norm_a", "out_norm_b"):
            if spec.get(name) is not None:
                for i, v in enumerate(np.asarray(spec[name], dtype=np.float32).reshape(-1)):
                    getattr(d, name)[i] = float(v)
        d.differential = int(bool(spec.get("differential", False)))
        for i, v in enumerate(spec.get("out_to_in", []) or []):
            d.out_to_in[i] = int(v)
        w = np.ascontiguousarray(spec["weights"], dtype=np.float32).reshape(-1)
        self.use_current_stream()
        self._chk(self.lib.cps_net_load(self._h, C.byref(d), w.ctypes.data_as(L._FP), w.shape[0]))
        self.net_htot = int(self.lib.cps_net_state_size(self._h))

    def net_rollout(self, s0, Q, q_layout=L.ROLLOUT_MAJOR, traj_layout=L.ROLLOUT_MAJOR, h0=None, want_traj=True,
                    want_h=False, traj_out=None):
        """cps_net_rollout on device tensors; h0 None = the stored hidden state, [Htot] shared, or [B, Htot]."""
        self.use_current_stream()
        Q2, B, T, batched, traj_out = self._rollout_io(s0, Q, q_layout, traj_layout, want_traj, traj_out)
        h_b = 0
        if h0 is not None:
            _check_dev(h0, "h0", self.device)
            if h0.numel() == self.net_htot:
                h_b = 0
            elif h0.numel() == self.net_htot * B:
                h_b = 1
            else:
                raise ValueError(f"h0 has {h0.numel()} elements, expected {self.net_htot} or {self.net_htot * B}")
        h_final = torch.empty((B, self.net_htot), device=self.device, dtype=torch.float32) if want_h else None
        self._chk(self.lib.cps_net_rollout(self._h, _ptr(s0), batched, _ptr(Q2), q_layout, B, T, _ptr(h0), h_b,
                                           _ptr(traj_out), traj_layout, _ptr(h_final)))
        return traj_out, h_final

    def net_update(self, s, q0):
        """cps_net_update: advance the stored hidden state by one step on (q0 [1], s [6]) -- device tensors."""
        self.use_current_stream()
        _check_dev(s, "s", self.device)
        _check_dev(q0, "q0", self.device)
        self._chk(self.lib.cps_net_update(self._h, _ptr(s), _ptr(q0)))

    def net_reset_state(self):
        self.use_current_stream()
        self._chk(self.lib.cps_net_reset_state(self._h))

    def net_get_state(self) -> np.ndarray:
        self.use_current_stream()
        out = np.zeros(max(self.net_htot, 1), dtype=np.float32)
        self._chk(self.lib.cps_net_get_state(self._h, out.ctypes.data_as(L._FP)))
        return out[:self.net_htot]

    def net_set_state(self, state):
        self.use_current_stream()
        v = np.ascontiguousarray(np.asarray(state, dtype=np.float32).reshape(-1))
        if v.shape[0] != self.net_htot:
            raise ValueError(f"hidden state has {v.shape[0]} entries, expected {self.net_htot}")
        if self.net_htot:
            self._chk(self.lib.cps_net_set_state(self._h, v.ctypes.data_as(L._FP)))

    # -- standalone costs -----------------------------------------------------------------------------
    def trajectory_cost(self, traj, Q, u_prev=0.0):
        self.use_current_stream()
        _check_dev(traj, "traj", self.device)
        _check_dev(Q, "Q", self.device)
        K, T = traj.shape[0], traj.shape[1] - 1
        J = torch.empty((K,), device=self.device, dtype=torch.float32)
        self._chk(self.lib.cps_trajectory_cost(self._h, _ptr(traj), _ptr(Q), float(u_prev), K, T, _ptr(J)))
        return J

    def stage_cost(self, traj, Q, u_prev=0.0, unshifted=False):
        self.use_current_stream()
        _check_dev(traj, "traj", self.device)
        _check_dev(Q, "Q", self.device)
        K, rows, T = traj.shape[0], traj.shape[1], Q.shape[1]
        st = torch.empty((K, T), device=self.device, dtype=torch.float32)
        self._chk(self.lib.cps_stage_cost(self._h, _ptr(traj), rows, _ptr(Q), float(u_prev), K, T, int(unshifted),
                                          _ptr(st)))
        return st

    def terminal_cost(self, states):
        self.use_current_stream()
        _check_dev(states, "states", self.device)
        K = states.shape[0]
        out = torch.empty((K,), device=self.device, dtype=torch.float32)
        self._chk(self.lib.cps_terminal_cost(self._h, _ptr(states), K, _ptr(out)))
        return out

    # -- forward-only planners (random action, CEM) ----------------------------------------------------
    def _q_dims(self, Q, layout, name=None):
        """(K, T) of plans Q in `layout`; given a `name`, they must be the handle's K plans of T steps."""
        if Q.dim() < 2:
            raise ValueError("Q must be [K, T] (ROLLOUT_MAJOR) or [T, K] (TIME_MAJOR)")
        a, b = int(Q.shape[0]), int(Q.shape[1])
        if Q.numel() != a * b:
            raise ValueError("one control input only: trailing dimensions of Q must be 1")
        dims = (b, a) if layout == L.TIME_MAJOR else (a, b)
        if name is not None and dims != (self.K, self.T):
            raise ValueError(f"{name} has shape {tuple(Q.shape)}, expected K = {self.K}, T = {self.T}")
        return dims

    def plan_cost(self, s, Q, q_layout=L.ROLLOUT_MAJOR, u_prev=0.0, want_traj=False, traj_layout=L.ROLLOUT_MAJOR):
        """predict_and_cost of the forward-only optimizers (cps_plan_cost): J [K], and the trajectories if asked."""
        self.use_current_stream()
        _check_dev(s, "s", self.device)
        _check_dev(Q, "Q", self.device)
        K, T = self._q_dims(Q, q_layout)
        J = torch.empty((K,), device=self.device, dtype=torch.float32)
        traj = None
        if want_traj:
            shape = (T + 1, 6, K) if traj_layout == L.TIME_MAJOR else (K, T + 1, 6)
            traj = torch.empty(shape, device=self.device, dtype=torch.float32)
        self._chk(self.lib.cps_plan_cost(self._h, _ptr(s), _ptr(Q), q_layout, K, T, float(u_prev), _ptr(J), _ptr(traj),
                                         traj_layout))
        return J, traj

    def plan_random_action(self, s, Q, q_layout=L.ROLLOUT_MAJOR, u_prev=0.0, J_out=None, best_out=None):
        """cps_plan_random_action: returns the cuda tensor [1] holding Q[argmin J, 0] (no synchronisation)."""
        self.use_current_stream()
        _check_dev(s, "s", self.device)
        _check_dev(Q, "Q", self.device)
        self._q_dims(Q, q_layout, "Q")
        if best_out is not None:
            _check_dev(best_out, "best_out", self.device, torch.int32)
        self._chk(self.lib.cps_plan_random_action(self._h, _ptr(s), _ptr(Q), q_layout, float(u_prev), _ptr(self._u_dev),
                                                  _ptr(J_out), _ptr(best_out)))
        return self._u_dev

    def plan_random_action_host(self, s_np, Q, q_layout=L.ROLLOUT_MAJOR, u_prev=0.0) -> float:
        self.use_current_stream()
        _check_dev(Q, "Q", self.device)
        self._q_dims(Q, q_layout, "Q")
        self._chk(self.lib.cps_plan_random_action_host(self._h, self._s_host_from(s_np), _ptr(Q), q_layout, float(u_prev),
                                                       self._u_host))
        return self._u_host[0]

    def cem_configure(self, best_k, initial_stdev, stdev_min):
        self.use_current_stream()
        self._chk(self.lib.cps_cem_configure(self._h, int(best_k), float(initial_stdev), float(stdev_min)))

    def cem_reset(self):
        self.use_current_stream()
        self._chk(self.lib.cps_cem_reset(self._h))

    def _cem_eps(self, eps, layout):
        _check_dev(eps, "eps", self.device)
        if eps.dim() < 3 or eps.numel() != eps.shape[0] * self.K * self.T:
            raise ValueError(f"eps has shape {tuple(eps.shape)}, expected [iterations, K, T] or [iterations, T, K]")
        self._q_dims(eps[0], layout, "eps[0]")
        return int(eps.shape[0])

    def cem_step(self, s, eps, eps_layout=L.ROLLOUT_MAJOR, u_prev=0.0, Q_out=None, J_out=None):
        """cps_cem_step: eps.shape[0] outer iterations; returns the cuda tensor [1] holding u (no synchronisation)."""
        self.use_current_stream()
        _check_dev(s, "s", self.device)
        n_it = self._cem_eps(eps, eps_layout)
        self._chk(self.lib.cps_cem_step(self._h, _ptr(s), _ptr(eps), eps_layout, n_it, float(u_prev), _ptr(self._u_dev),
                                        _ptr(Q_out), _ptr(J_out)))
        return self._u_dev

    def cem_step_host(self, s_np, eps, eps_layout=L.ROLLOUT_MAJOR, u_prev=0.0) -> float:
        self.use_current_stream()
        n_it = self._cem_eps(eps, eps_layout)
        self._chk(self.lib.cps_cem_step_host(self._h, self._s_host_from(s_np), _ptr(eps), eps_layout, n_it, float(u_prev),
                                             self._u_host))
        return self._u_host[0]

    def cem_get_distribution(self):
        self.use_current_stream()
        mu, sd = np.zeros(self.T, dtype=np.float32), np.zeros(self.T, dtype=np.float32)
        self._chk(self.lib.cps_cem_get_distribution(self._h, mu.ctypes.data_as(L._FP), sd.ctypes.data_as(L._FP)))
        return mu, sd

    def cem_set_distribution(self, mean=None, stdev=None):
        self.use_current_stream()
        def arr(v):
            if v is None:
                return None, None
            a = np.ascontiguousarray(np.asarray(v, dtype=np.float32).reshape(-1))
            if a.shape[0] != self.T:
                raise ValueError(f"distribution vectors have {self.T} entries")
            return a, a.ctypes.data_as(L._FP)
        m, mp_ = arr(mean)
        s_, sp = arr(stdev)
        self._chk(self.lib.cps_cem_set_distribution(self._h, mp_, sp))

    # -- CEM with a Gaussian-mixture sampling distribution (optimizer_cem_gmm_tf) -----------------------------
    def cem_gmm_configure(self, best_k, initial_stdev, stdev_min):
        self.use_current_stream()
        self._chk(self.lib.cps_cem_gmm_configure(self._h, int(best_k), float(initial_stdev), float(stdev_min)))

    def cem_gmm_reset(self):
        self.use_current_stream()
        self._chk(self.lib.cps_cem_gmm_reset(self._h))

    def _gmm_draws(self, eps, u01, layout):
        _check_dev(eps, "eps", self.device)
        _check_dev(u01, "u01", self.device)
        n_it = int(u01.shape[0])
        want_e = (n_it, 2, self.T, self.K) if layout == L.TIME_MAJOR else (n_it, self.K, self.T, 2)
        want_u = (n_it, self.T, self.K) if layout == L.TIME_MAJOR else (n_it, self.K, self.T)
        if tuple(eps.shape) != want_e or tuple(u01.shape) != want_u:
            raise ValueError(f"draws have shapes {tuple(eps.shape)} / {tuple(u01.shape)}, expected {want_e} / {want_u}")
        return n_it

    def cem_gmm_step(self, s, eps, u01, layout=L.ROLLOUT_MAJOR, u_prev=0.0, Q_out=None, J_out=None):
        """cps_cem_gmm_step: u01.shape[0] outer iterations; returns the cuda tensor [1] holding u (no synchronisation)."""
        self.use_current_stream()
        _check_dev(s, "s", self.device)
        n_it = self._gmm_draws(eps, u01, layout)
        self._chk(self.lib.cps_cem_gmm_step(self._h, _ptr(s), _ptr(eps), _ptr(u01), layout, n_it, float(u_prev),
                                            _ptr(self._u_dev), _ptr(Q_out), _ptr(J_out)))
        return self._u_dev

    def cem_gmm_step_host(self, s_np, eps, u01, layout=L.ROLLOUT_MAJOR, u_prev=0.0) -> float:
        self.use_current_stream()
        n_it = self._gmm_draws(eps, u01, layout)
        self._chk(self.lib.cps_cem_gmm_step_host(self._h, self._s_host_from(s_np), _ptr(eps), _ptr(u01), layout, n_it, float(u_prev),
                                                 self._u_host))
        return self._u_host[0]

    def cem_gmm_get_distribution(self):
        """(loc [2, T], scale [2, T], p1): component-major copies of the device-resident mixture."""
        self.use_current_stream()
        loc, sc = np.zeros((2, self.T), dtype=np.float32), np.zeros((2, self.T), dtype=np.float32)
        p1 = np.zeros(1, dtype=np.float32)
        self._chk(self.lib.cps_cem_gmm_get_distribution(self._h, loc.ctypes.data_as(L._FP), sc.ctypes.data_as(L._FP),
                                                        p1.ctypes.data_as(L._FP)))
        return loc, sc, float(p1[0])

    def cem_gmm_set_distribution(self, loc=None, scale=None, p1=None):
        self.use_current_stream()
        keep = []
        def arr(v, n):
            if v is None:
                return None
            a = np.ascontiguousarray(np.asarray(v, dtype=np.float32).reshape(-1))
            if a.shape[0] != n:
                raise ValueError(f"expected {n} values")
            keep.append(a)
            return a.ctypes.data_as(L._FP)
        self._chk(self.lib.cps_cem_gmm_set_distribution(self._h, arr(loc, 2 * self.T), arr(scale, 2 * self.T), arr(p1, 1)))

    # -- gradient of predict_and_cost, RPGD --------------------------------------------------------------------
    def plan_cost_grad(self, s, Q, q_layout=L.ROLLOUT_MAJOR, u_prev=0.0, want_J=True):
        """cps_plan_cost_grad: (J [K] or None, dJ/dQ in the layout of Q) as cuda tensors (no synchronisation)."""
        self.use_current_stream()
        _check_dev(s, "s", self.device)
        _check_dev(Q, "Q", self.device)
        self._q_dims(Q, q_layout, "Q")
        G = torch.empty_like(Q)
        J = torch.empty(self.K, device=self.device) if want_J else None
        self._chk(self.lib.cps_plan_cost_grad(self._h, _ptr(s), _ptr(Q), q_layout, float(u_prev), _ptr(J), _ptr(G)))
        return J, G

    def rpgd_reset(self):
        self.use_current_stream()
        self._chk(self.lib.cps_rpgd_reset(self._h))

    def rpgd_grad_step(self, s, Q, u_prev=0.0, learning_rate=0.05, beta_1=0.9, beta_2=0.999, epsilon=1e-8, gradmax_clip=5.0,
                       J_out=None):
        """cps_rpgd_grad_step: gradient, clip_by_norm, Adam, clip to the limits -- in place on Q [K, T] (rollout-major)."""
        self.use_current_stream()
        _check_dev(s, "s", self.device)
        _check_dev(Q, "Q", self.device)
        if tuple(Q.shape[:2]) != (self.K, self.T) or not Q.is_contiguous():
            raise ValueError(f"Q must be a contiguous [{self.K}, {self.T}] tensor")
        self._chk(self.lib.cps_rpgd_grad_step(self._h, _ptr(s), _ptr(Q), float(u_prev), float(learning_rate), float(beta_1),
                                              float(beta_2), float(epsilon), float(gradmax_clip), _ptr(J_out)))

    def rpgd_adam_state(self):
        """(m, v, iterations): the Adam moments as cuda tensors [K, T] aliasing the handle's buffers."""
        m, v, it = C.c_void_p(), C.c_void_p(), C.c_longlong()
        self._chk(self.lib.cps_rpgd_adam_state(self._h, C.byref(m), C.byref(v), C.byref(it)))
        if not hasattr(self, "_adam_views") or self._adam_views[2] != (m.value, v.value):
            import ctypes

            def view(ptr):
                n = self.K * self.T
                # a non-owning tensor over the handle's buffer (CUDA array interface)
                class _Buf:
                    __cuda_array_interface__ = {"shape": (self.K, self.T), "typestr": "<f4", "data": (ptr, False), "version": 2}
                return torch.as_tensor(_Buf(), device=self.device)
            self._adam_views = (view(m.value), view(v.value), (m.value, v.value))
        return self._adam_views[0], self._adam_views[1], int(it.value)

    def rpgd_finish(self, J, Q, fresh, keep: int, shift_previous: int, ages=None) -> np.ndarray:
        """cps_rpgd_finish: get_action and the per-solve bookkeeping of RPGD's step() in place on Q [K, T] (and on the
        handle's Adam moments, `ages` int32 [K]); returns the cheapest plan [T] on the host (synchronises)."""
        self.use_current_stream()
        for t, name in ((J, "J"), (Q, "Q")):
            _check_dev(t, name, self.device)
        if tuple(Q.shape[:2]) != (self.K, self.T) or not Q.is_contiguous() or J.numel() != self.K:
            raise ValueError("rpgd_finish: Q must be a contiguous [K, T] tensor and J [K]")
        if fresh is not None:
            _check_dev(fresh, "fresh", self.device)
            if tuple(fresh.shape) != (self.K - keep, self.T) or not fresh.is_contiguous():
                raise ValueError(f"rpgd_finish: fresh has shape {tuple(fresh.shape)}, expected {(self.K - keep, self.T)}")
        if ages is not None and (ages.dtype != torch.int32 or ages.numel() != self.K):
            raise ValueError("rpgd_finish: ages must be int32 [K]")
        out = np.empty(self.T, dtype=np.float32)
        self._chk(self.lib.cps_rpgd_finish(self._h, _ptr(J), _ptr(Q), _ptr(fresh), int(keep), int(shift_previous), _ptr(ages),
                                           out.ctypes.data_as(C.c_void_p)))
        return out

    def rpgd_set_iterations(self, n: int):
        self._chk(self.lib.cps_rpgd_set_iterations(self._h, int(n)))

    def measure_peaks(self):
        """(FP32 TFLOP/s, MUFU Gop/s) measured on this device by two microbenchmark kernels."""
        self.use_current_stream()
        f, m = C.c_double(0), C.c_double(0)
        self._chk(self.lib.cps_measure_peaks(self._h, C.byref(f), C.byref(m)))
        return f.value, m.value

    def selftest_sincos(self) -> int:
        """Number of floats in [-pi, pi] on which the kernels' folded sincos differs from sincosf / cosf (0 expected)."""
        self.use_current_stream()
        n = C.c_longlong(-1)
        self._chk(self.lib.cps_selftest_sincos(self._h, C.byref(n)))
        return int(n.value)

    # -- diagnostics ----------------------------------------------------------------------------------
    def launch_count(self) -> int:
        return int(self.lib.cps_launch_count(self._h))

    def rollout_last_kernel(self) -> str | None:
        """'rollout_kernel' | 'rollout_pair_kernel': what the last open-loop rollout call launched (None: none yet)."""
        return {0: None, 1: "rollout_kernel", 2: "rollout_pair_kernel"}[int(self.lib.cps_rollout_last_kernel(self._h))]

    def net_last_kernel(self) -> str | None:
        """'fp32' | 'tensor': the network kernel the last neural rollout / solve launched (None: none yet)."""
        return {0: None, 1: "fp32", 2: "tensor"}[int(self.lib.cps_net_last_kernel(self._h))]

    def nonfinite_costs(self) -> int:
        n = C.c_int(0)
        self._chk(self.lib.cps_nonfinite_costs(self._h, C.byref(n)))
        return n.value
