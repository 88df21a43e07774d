// cps_lib.cu -- kernels and C ABI of libcps_b200.so (see include/cps.h).
//
// Kernels
//   mppi_kernel      (cps_mppi_inst.cuh, one translation unit per cost plugin) K1+K2: one MPPI solve in one launch (optimizer_mppi.py:180-192).  One thread = one rollout,
//                    state in registers, stage/terminal/correction cost accumulated in the same pass, block
//                    partials (min J, sum w, sum w*noise[i]) merged by the last block to finish (ticket) with the
//                    online-softmax rule, which then writes the clipped u_nom and u.
//   rollout_kernel   K3: open-loop batched rollouts (predictor.predict_core), optional trajectory output.
//   cost_kernel      standalone get_trajectory_cost / get_stage_cost on materialised trajectories.
//   finalize_kernel  merge of per-GPU partials when K is sharded over ranks.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>

#include "cps_internal.cuh"

// =====================================================================================================
// K1 + K2: the MPPI solve
// =====================================================================================================
// Merge of gathered per-rank partials (K sharded over GPUs).
__global__ void __launch_bounds__(128) finalize_kernel(const __grid_constant__ FinalizeArgs a, int direct_noise) {
    extern __shared__ float smem[];
    float *s_unom = smem;            // [T]
    float *s_E = s_unom + a.mp.T;    // [n_red + 2 + nwarps]
    const int T = a.mp.T;
    for (int t = threadIdx.x; t < T; t += blockDim.x) s_unom[t] = a.u_nom[min(t + 1, T - 1)];
    __syncthreads();
    merge_and_finish(a.mp, a.partials, a.n_parts, s_E, s_unom, a.u_nom, a.u_out, a.shard_out, direct_noise != 0);
}

// =====================================================================================================
// K3: open-loop batched rollouts
// =====================================================================================================
template <int INTEG, int SC, bool FAST_DIV, bool EXACT_ATAN2>
__global__ void __launch_bounds__(256, 4) rollout_kernel(const __grid_constant__ RolloutArgs a) {
    const OdeParams ode = pin_params(a.ode, a.s0[0]);
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < a.B; b += stride) {
        State z = load_state(a.s0 + b * a.ss_b);
        const float *q = a.Q + b * a.qs_b;
        float *traj = a.traj_out ? a.traj_out + b * a.ts_k : nullptr;
        float qn = q[0];
#pragma unroll 1
        for (int t = 0; t < a.T; ++t) {
            const float Q = qn;
            if (t + 1 < a.T) qn = q[(long long)(t + 1) * a.qs_t];  // prefetch under the integration
            if (traj) store_state(traj + (long long)t * a.ts_t, a.ts_c, z);
            control_step<INTEG, SC, FAST_DIV, EXACT_ATAN2, true>(ode, z, Q);
        }
        if (traj) store_state(traj + (long long)a.T * a.ts_t, a.ts_c, z);
        if (a.final_out) store_state(a.final_out + b * 6, 1, z);
    }
}

#ifndef CPS_PAIR_MIN_BLOCKS
#define CPS_PAIR_MIN_BLOCKS 8
#endif
// Two cartpoles per thread (packed FP32, see cps_device.cuh "two cartpoles per thread"): thread p owns cartpoles
// 2p and 2p+1 of a time-major batch, so controls arrive as one 8-byte load and every state channel leaves as one
// 8-byte store per control step (256 B per warp and channel).  Bit-identical to rollout_kernel<INTEG, SC_ROTATE>.
// Stores the six channels at *tp and advances it to the same cartpoles one control step on: one 64-bit pointer walked
// channel by channel (cb = channel stride, tb = step stride minus five channel strides, both in bytes).
__device__ __forceinline__ void store_state2_walk(char *&tp, long long cb, long long tb, const State2 &z) {
    *reinterpret_cast<unsigned long long *>(tp) = z.th.v; tp += cb;
    *reinterpret_cast<unsigned long long *>(tp) = z.w.v; tp += cb;
    *reinterpret_cast<unsigned long long *>(tp) = z.c.v; tp += cb;
    *reinterpret_cast<unsigned long long *>(tp) = z.s.v; tp += cb;
    *reinterpret_cast<unsigned long long *>(tp) = z.x.v; tp += cb;
    *reinterpret_cast<unsigned long long *>(tp) = z.v.v; tp += tb;
}

// Without the trajectory stores the 9-block / 56-register allocation is the faster one (606 vs 641 us), with them the
// 8-block / 64-register one (636 vs 644 us): ptxas' schedule, not occupancy, decides at this point.
// Occupancy A/B (1M x 500, B200, round 1): 56 registers / 9 blocks per SM 812 us; 48 / 10 805 us; 64 / 8 823 us; 40 / 12
// (spills) 827 us; 80 / 6 878 us -- a plateau.  Per control step (round 2): the angle resync of both halves in packed
// arithmetic (resync_angle2), the redo copy of the state in shared memory, the trajectory pointer advanced instead of
// recomputed.
template <int INTEG, bool FAST_DIV, int NSUB, bool TRAJ>
__global__ void __launch_bounds__(128, TRAJ ? CPS_PAIR_MIN_BLOCKS : CPS_PAIR_MIN_BLOCKS + 1) rollout_pair_kernel(const __grid_constant__ RolloutArgs a) {
    __shared__ unsigned long long s_save[5 * 128];
    const OdeParams ode = pin_params(a.ode, a.s0[0]);
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long n_pairs = (long long)a.B >> 1;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n_pairs; p += stride) {
        const long long b = 2 * p;
        State2 z = join_states(load_state(a.s0 + b * a.ss_b), load_state(a.s0 + (b + 1) * a.ss_b));
        const float *q = a.Q + b;
        char *tp = TRAJ ? reinterpret_cast<char *>(a.traj_out + b) : nullptr;
        const long long cb = a.ts_c * 4, tb = (a.ts_t - 5 * a.ts_c) * 4;
        unsigned long long qn = *reinterpret_cast<const unsigned long long *>(q);
#pragma unroll 1
        for (int t = 0; t < a.T; ++t) {
            F2 Q;
            Q.v = qn;
            q += a.qs_t;
            if (t + 1 < a.T) qn = *reinterpret_cast<const unsigned long long *>(q);
            if (TRAJ) store_state2_walk(tp, cb, tb, z);
            control_step2<INTEG, FAST_DIV, NSUB>(ode, z, Q, s_save + threadIdx.x, 128);
        }
        if (TRAJ) store_state2_walk(tp, cb, tb, z);
        if (a.final_out) {
            store_state(a.final_out + b * 6, 1, half_state(z, 0));
            store_state(a.final_out + (b + 1) * 6, 1, half_state(z, 1));
        }
    }
}

// =====================================================================================================
// standalone cost plugin
// =====================================================================================================
// get_trajectory_cost sums its T+1 entries in the reference backend's order for every plugin (RowSumPlan, cps_device.cuh;
// dynamic shared memory: row_sum_slots(T + 1) x blockDim floats) and divides by T+1.
template <int COST>
__global__ void __launch_bounds__(256) cost_kernel(const __grid_constant__ CostArgs a) {
    extern __shared__ float smem[];
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= a.K) return;
    const float *tr = a.traj + (size_t)k * a.rows * 6;
    const float *q = a.Q + (size_t)k * a.T;
    const float shift = a.unshifted ? 0.0f : a.cost.max_cost;
    const RowSumPlan rsp = row_sum_plan(a.T + 1);
    float *sl = smem + threadIdx.x;
    const int ss = blockDim.x;
    float tail = 0.0f, up = a.u_prev;
    if (a.J) row_sum_init(rsp, sl, ss);
    for (int t = 0; t < a.T; ++t) {
        const float *s = tr + (size_t)t * 6;
        const float u = q[t];
        const float c = stage_cost<COST>(a.cost, cosf(s[IDX_ANGLE]), s[IDX_ANGLED], s[IDX_POS], u, up) - shift;
        if (a.stage) a.stage[(size_t)k * a.T + t] = c;
        if (a.J) row_sum_push(rsp, sl, ss, tail, t, c);
        up = u;
    }
    if (a.J) {
        const float *s = tr + (size_t)a.T * 6;
        row_sum_push(rsp, sl, ss, tail, a.T, terminal_cost<COST>(a.cost, s[IDX_ANGLE], s[IDX_POS]));
        a.J[k] = __fdiv_rn(row_sum_finish(rsp, sl, ss, tail), (float)(a.T + 1));
    }
}

template <int COST>
__global__ void __launch_bounds__(256) terminal_cost_kernel(CostParams C, const float *states, int K, float *out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    out[k] = terminal_cost<COST>(C, states[(size_t)k * 6 + IDX_ANGLE], states[(size_t)k * 6 + IDX_POS]);
}

// =====================================================================================================
// host side
// =====================================================================================================
thread_local std::string g_create_err;

static void fold_ode(cps_handle *h) {
    const double k = h->phys[CPS_PH_K], mc = h->phys[CPS_PH_M_CART], g = h->phys[CPS_PH_G];
    const double J = h->phys[CPS_PH_J_FRIC], M = h->phys[CPS_PH_M_FRIC], umax = h->phys[CPS_PH_U_MAX];
    // predictor_ODE takes L and m_pole from variable_parameters (predictors_customization.py:51-60);
    // predictor_ODE_v0 only L (predictors_customization_v0.py:47-54)
    const double L = h->L_var;
    const double mp = (h->cfg.integrator == CPS_EULER_V0) ? (double)h->phys[CPS_PH_M_POLE] : (double)h->m_pole_var;
    const double kp1 = k + 1.0, Lh = L / 2.0;
    OdeParams &o = h->ode;
    o.KM = (float)(kp1 * (mc + mp));
    o.m_p = (float)mp;
    o.c1 = (float)(mp * g);
    o.c2 = (float)(kp1 * mp * Lh);
    o.c3 = (float)(J / Lh);
    o.c5 = (float)(kp1 * M);
    o.d1 = (float)(g / (kp1 * Lh));
    o.d2 = (float)(1.0 / (kp1 * Lh));
    o.d3 = (float)(J / (mp * Lh * kp1 * Lh));
    o.u_scale = (float)(kp1 * umax);
    o.h = (float)((double)h->cfg.dt / (double)h->cfg.substeps);
    {   // rotation substeps: the step folded into the angular-acceleration constants (ode_rhs_w) and the rotation (rotate_cs)
        const double hh = (double)h->cfg.dt / (double)h->cfg.substeps;
        const double hd2 = hh * (1.0 / (kp1 * Lh));
        o.yc1 = (float)(hd2 * (mp * g));
        o.yc2 = (float)(hd2 * (kp1 * mp * Lh));
        o.yc3 = (float)(hd2 * (J / Lh));
        o.yc5 = (float)(hd2 * (kp1 * M));
        o.yu_scale = (float)(hd2 * (kp1 * umax));
        o.v_y = (float)(kp1 * Lh);
        o.hd1 = (float)(hh * (g / (kp1 * Lh)));
        o.hd3 = (float)(hh * (J / (mp * Lh * kp1 * Lh)));
        o.rot_c2 = (float)(-hh * hh / 2.0);
        o.rot_s3 = (float)(-hh * hh * hh / 6.0);
        o.rot_c4 = (float)(hh * hh * hh * hh / 24.0);
        o.w_rot_max = (float)((double)CPS_ROT_MAX / hh);
    }
    o.thl = h->phys[CPS_PH_TRACK_HALF_LENGTH];
    o.bounce = (float)(2.0 / (0.5 * L));
    o.n = h->cfg.substeps;
}

static int fold_cost_into(cps_handle *h, float target_equilibrium, CostParams &c) {
    memset(&c, 0, sizeof(c));
    const float thl = h->phys[CPS_PH_TRACK_HALF_LENGTH];
    c.thl = thl;
    c.inv_2thl = 1.0f / (2.0f * thl);
    c.target_position = h->target_position;
    c.target_equilibrium = target_equilibrium;
    const float *w = h->cost_in;
    switch (h->cfg.cost_id) {
    case CPS_COST_NONE: break;
    case CPS_COST_DEFAULT:
    case CPS_COST_QUADRATIC_BOUNDARY: {
        // in: [dd_weight, ep_weight, cc_weight, ccrc_weight, R, MAX_COST]
        if (h->cost_in_n < 6) return fail(h, CPS_ERR_INVALID, "cost params: need 6 values for default/quadratic_boundary");
        const bool qb = h->cfg.cost_id == CPS_COST_QUADRATIC_BOUNDARY;
        c.w[0] = w[0]; c.w[1] = w[1] * 0.25f; c.w[2] = w[2] * w[4]; c.w[3] = qb ? w[3] : 0.0f;
        c.w[4] = (qb ? 0.95f : 0.90f) * thl;   // float32 product, as the plugin computes it
        c.w[5] = 1.0f / (0.05f * thl);
        c.max_cost = w[5];
        break;
    }
    case CPS_COST_QB_GRAD_MINIMAL: {
        // in: [dd_quadratic_w, db_w, ep_w, ekp_w, cc_w, R, permissible_track_fraction]
        if (h->cost_in_n < 7) return fail(h, CPS_ERR_INVALID, "cost params: need 7 values for quadratic_boundary_grad_minimal");
        c.w[0] = w[0]; c.w[1] = w[1]; c.w[2] = w[2]; c.w[3] = w[3]; c.w[4] = w[4] * w[5];
        c.w[5] = w[6] * thl;
        c.w[6] = 1.0f / ((1.0f - w[6]) * thl);
        break;
    }
    case CPS_COST_QB_GRAD: {
        // in (11): [dd_q, dd_lin, db, ep, ekp, cc, ccrc, R, permissible_track_fraction, corr, admissible_angle(rad)]
        // in (19): [dd_q, dd_lin, db, ep, ekp, cc, ccrc, corr]_up, [..]_down, R, fraction, admissible_angle(rad);
        //          the set is chosen by target_equilibrium == 1 (quadratic_boundary_grad.py:182-200)
        float v[11];
        if (h->cost_in_n == 11) {
            memcpy(v, w, sizeof(v));
        } else if (h->cost_in_n == 19) {
            const float *set = (target_equilibrium == 1.0f) ? w : w + 8;
            for (int i = 0; i < 7; ++i) v[i] = set[i];
            v[7] = w[16]; v[8] = w[17]; v[9] = set[7]; v[10] = w[18];
        } else {
            return fail(h, CPS_ERR_INVALID, "cost params: need 11 or 19 values for quadratic_boundary_grad");
        }
        const float e = target_equilibrium;
        c.w[0] = v[0]; c.w[1] = v[1]; c.w[2] = v[2]; c.w[3] = v[3]; c.w[4] = v[4]; c.w[5] = v[5] * v[7]; c.w[6] = v[6];
        c.w[7] = v[8] * thl;
        c.w[8] = 1.0f / ((1.0f - v[8]) * thl);
        c.w[9] = fabsf((120.0f * (1.0f + e)) / 2.0f + v[9]);
        c.w[10] = cosf(v[10]);
        break;
    }
    case CPS_COST_LEGACY_MPPI: {
        // in: [dd_weight, ep_weight, ekp_weight, ekc_weight, ccrc_weight] (controller_mppi_cartpole.py:245-257)
        if (h->cost_in_n < 5) return fail(h, CPS_ERR_INVALID, "cost params: need 5 values for the legacy controller_mppi_cartpole cost");
        c.w[0] = w[0]; c.w[1] = w[1] * 0.25f; c.w[2] = w[2]; c.w[3] = w[3]; c.w[4] = w[4];
        // |x| > 0.95 * TrackHalfLength is evaluated in double by numba (:142); for a float x that is x > RD(threshold)
        const double thr = 0.95 * (double)thl;
        float thr_f = (float)thr;
        if ((double)thr_f > thr) thr_f = nextafterf(thr_f, 0.0f);
        c.w[5] = thr_f;
        break;
    }
    default: return fail(h, CPS_ERR_UNSUPPORTED, "unknown cost id %d", h->cfg.cost_id);
    }
    return CPS_OK;
}

static int fold_cost(cps_handle *h) { return fold_cost_into(h, h->target_equilibrium, h->cost); }

int cps_fold_cost_for(cps_handle *h, float target_equilibrium, CostParams *out) {
    return fold_cost_into(h, target_equilibrium, *out);
}

static void fold_mppi(cps_handle *h) {
    MppiParams &m = h->mp;
    const float cc = h->mppi_in[0], R = h->mppi_in[1], LBD = h->mppi_in[2], NU = h->mppi_in[3];
    m.cc_half_nu = cc * ((0.5f * (1.0f - 1.0f / NU)) * R);
    m.cc_R = cc * R;
    m.cc_half_R = cc * (0.5f * R);
    m.inv_lambda = (float)(1.0 / (double)LBD);
    m.sigma = h->mppi_in[4];
    m.lo = h->mppi_in[5];
    m.hi = h->mppi_in[6];
    m.K = h->cfg.num_rollouts;
    m.T = h->cfg.horizon;
    m.p = h->cfg.interp_period;
    m.n_ind = h->n_ind;
    m.n_red = h->n_red;
    m.inv_T1 = 1.0f / (float)(m.T + 1);
    m.T1 = (float)(m.T + 1);
    m.rs_off = 0;
    m.inv_p = 1.0f / (float)m.p;
}

extern "C" int cps_abi_version(void) { return CPS_ABI_VERSION; }

extern "C" int cps_num_inducing_points(int horizon, int period) {
    if (horizon < 1 || period < 1) return -1;
    return (int)std::ceil((double)(horizon - 1) / (double)period) + 1;
}

extern "C" const char *cps_last_error(const cps_handle *h) { return h ? h->err.c_str() : g_create_err.c_str(); }

extern "C" int cps_create(const cps_config *cfg, cps_handle **out) {
    if (!cfg || !out) return fail(nullptr, CPS_ERR_INVALID, "cps_create: null argument");
    *out = nullptr;
    if (cfg->struct_size != (int)sizeof(cps_config))
        return fail(nullptr, CPS_ERR_INVALID, "cps_create: cps_config size mismatch (%d vs %d)", cfg->struct_size,
                    (int)sizeof(cps_config));
    if (cfg->num_rollouts < 1 || cfg->horizon < 1 || cfg->substeps < 1 || !(cfg->dt > 0.0f) || cfg->interp_period < 1)
        return fail(nullptr, CPS_ERR_INVALID, "cps_create: K, T, n, dt and period must be positive");
    if (cfg->integrator != CPS_EULER_V0 && cfg->integrator != CPS_EULER_CROMER && cfg->integrator != CPS_PREDICTOR_NEURAL)
        return fail(nullptr, CPS_ERR_UNSUPPORTED, "cps_create: unknown integrator %d", cfg->integrator);
    if (cfg->cost_id < CPS_COST_NONE || cfg->cost_id > CPS_COST_LEGACY_MPPI)
        return fail(nullptr, CPS_ERR_UNSUPPORTED, "cps_create: unknown cost id %d", cfg->cost_id);
    if (cfg->cost_id == CPS_COST_LEGACY_MPPI && (cfg->noise_mode != CPS_NOISE_DIRECT || cfg->integrator == CPS_PREDICTOR_NEURAL))
        return fail(nullptr, CPS_ERR_INVALID, "cps_create: CPS_COST_LEGACY_MPPI needs CPS_NOISE_DIRECT and an ODE integrator");
    if (cfg->noise_mode != CPS_NOISE_INDUCING && cfg->noise_mode != CPS_NOISE_DIRECT)
        return fail(nullptr, CPS_ERR_INVALID, "cps_create: unknown noise mode %d", cfg->noise_mode);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, CPS_ERR_CUDA, "cps_create: no CUDA device (%s); this library has no CPU fallback",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (cfg->device < 0 || cfg->device >= ndev)
        return fail(nullptr, CPS_ERR_INVALID, "cps_create: device %d out of range (%d devices)", cfg->device, ndev);
    cps_handle *h = new (std::nothrow) cps_handle();
    if (!h) return fail(nullptr, CPS_ERR_INVALID, "cps_create: out of host memory");
    h->cfg = *cfg;
    h->n_ind = cps_num_inducing_points(cfg->horizon, cfg->interp_period);
    h->n_red = (cfg->noise_mode == CPS_NOISE_INDUCING) ? h->n_ind : cfg->horizon;
    // defaults: cartpole_physical_parameters.yml:6-17,33-42
    const float ph[CPS_PH_COUNT] = {(float)(1.0 / 3.0), 0.230f, 0.087f, 9.81f, 5.0e-5f, 3.22f, 0.395f, 1.77f,
                                    (float)((44.0e-2 - 4.4e-2) / 2.0)};
    memcpy(h->phys, ph, sizeof(ph));
    h->L_var = ph[CPS_PH_L];
    h->m_pole_var = ph[CPS_PH_M_POLE];
    h->target_position = 0.0f;
    h->target_equilibrium = 1.0f;
    // defaults: config_cost_function.yml:5-58
    {
        const float d_def[6] = {600.0f, 20000.0f, 1.0f, 1.0f, 1.0f, 6000019968.0f};
        const float d_min[7] = {10.0f, 10000.0f, 40.0f, 1.0f, 5.0f, 1.0f, 0.85f};
        const float d_leg[5] = {120.0f, 50000.0f, 0.01f, 5.0f, 1.0f};  // config_controllers.yml:16-21
        const float d_grad[19] = {500.0f, 0.0f, 10000.0f, 6000.0f, 30.0f, 5.0f, 0.0f, 0.0f,
                                  500.0f, 0.0f, 10000.0f, 6000.0f, 30.0f, 5.0f, 0.0f, 100.0f, 1.0f, 0.85f, 0.0f};
        switch (cfg->cost_id) {
        case CPS_COST_DEFAULT: case CPS_COST_QUADRATIC_BOUNDARY: memcpy(h->cost_in, d_def, sizeof(d_def)); h->cost_in_n = 6; break;
        case CPS_COST_QB_GRAD_MINIMAL: memcpy(h->cost_in, d_min, sizeof(d_min)); h->cost_in_n = 7; break;
        case CPS_COST_QB_GRAD: memcpy(h->cost_in, d_grad, sizeof(d_grad)); h->cost_in_n = 19; break;
        case CPS_COST_LEGACY_MPPI: memcpy(h->cost_in, d_leg, sizeof(d_leg)); h->cost_in_n = 5; break;
        default: h->cost_in_n = 0; break;
        }
    }
    // defaults: config_optimizers.yml:87-97
    const float mp[7] = {1.0f, 1.0f, 100.0f, 1000.0f, (float)(0.03 / std::sqrt((double)cfg->dt)), -1.0f, 1.0f};
    memcpy(h->mppi_in, mp, sizeof(mp));
    if (cfg->cost_id == CPS_COST_LEGACY_MPPI) h->mppi_in[4] = (float)(0.02 / std::sqrt((double)cfg->dt));  // config_controllers.yml:27
    fold_ode(h);
    fold_mppi(h);
    int rc = fold_cost(h);
    if (rc != CPS_OK) { g_create_err = h->err; delete h; return rc; }

    // launch geometry of the MPPI kernel: small K is latency bound -> one warp per block spreads the warps over
    // the SMs; large K -> 128-thread blocks
    const int K = cfg->num_rollouts;
    h->block = (K <= 148 * 32 * 4) ? 32 : (K <= 148 * 64 * 8 ? 64 : 128);
    if (cfg->integrator == CPS_PREDICTOR_NEURAL) h->block = 16;  // rollouts per CTA of net_kernel (cps_net.cu)
    h->grid = (K + h->block - 1) / h->block;
    h->smem = sizeof(float) * mppi_smem_floats(h->mp, cfg->cost_id, h->block, 1);
    if (h->smem > 200 * 1024) {
        g_create_err = "cps_create: horizon too large for the shared-memory staging of this build";
        delete h;
        return CPS_ERR_UNSUPPORTED;
    }
#define CREATE_TRY(expr)                                                                                        \
    do {                                                                                                        \
        cudaError_t e2_ = (expr);                                                                               \
        if (e2_ != cudaSuccess) {                                                                               \
            fail(nullptr, CPS_ERR_CUDA, "cps_create: %s: %s", #expr, cudaGetErrorString(e2_));                  \
            cps_destroy(h);                                                                                     \
            return CPS_ERR_CUDA;                                                                                \
        }                                                                                                       \
    } while (0)
    CREATE_TRY(cudaSetDevice(cfg->device));
    CREATE_TRY(cudaMalloc(&h->d_partials, sizeof(float) * (size_t)h->grid * (h->n_red + 2)));
    CREATE_TRY(cudaMalloc(&h->d_ticket, sizeof(unsigned)));
    CREATE_TRY(cudaMalloc(&h->d_nonfinite, sizeof(int)));
    CREATE_TRY(cudaMalloc(&h->d_s, sizeof(float) * 8));
    CREATE_TRY(cudaMalloc(&h->d_unom, sizeof(float) * (size_t)cfg->horizon));
    CREATE_TRY(cudaMalloc(&h->d_u, sizeof(float) * 4));
    if (cfg->cost_id == CPS_COST_LEGACY_MPPI) {
        CREATE_TRY(cudaMalloc(&h->d_uprev, sizeof(float) * (size_t)cfg->horizon));
        CREATE_TRY(cudaMemset(h->d_uprev, 0, sizeof(float) * (size_t)cfg->horizon));
    }
    CREATE_TRY(cudaHostAlloc(&h->h_pin, sizeof(float) * 16, cudaHostAllocMapped));
    if (cudaHostGetDevicePointer((void **)&h->h_pin_dev, h->h_pin, 0) != cudaSuccess) { h->h_pin_dev = nullptr; cudaGetLastError(); }
    CREATE_TRY(cudaMemset(h->d_ticket, 0, sizeof(unsigned)));
    CREATE_TRY(cudaMemset(h->d_nonfinite, 0, sizeof(int)));
    CREATE_TRY(cudaMemset(h->d_unom, 0, sizeof(float) * (size_t)cfg->horizon));
    CREATE_TRY(cudaDeviceSynchronize());
#undef CREATE_TRY
    *out = h;
    return CPS_OK;
}

extern "C" void cps_destroy(cps_handle *h) {
    if (!h) return;
    cudaSetDevice(h->cfg.device);
    cps_net_free(h);
    cps_fleet_free(h);
    cps_rpgd_fleet_free(h);
    cps_cem_fleet_free(h);
    cps_plan_free(h);
    cps_gmm_free(h);
    cps_grad_free(h);
    cudaFree(h->d_partials); cudaFree(h->d_ticket); cudaFree(h->d_nonfinite); cudaFree(h->d_px_timeouts);
    cudaFree(h->d_s); cudaFree(h->d_unom); cudaFree(h->d_u); cudaFree(h->d_uprev); cudaFree(h->d_ldu); cudaFree(h->d_lknots);
    cudaFree(h->d_rs0); cudaFree(h->d_rQ); cudaFree(h->d_rtraj); cudaFree(h->d_rfinal);
    if (h->h_pin) cudaFreeHost(h->h_pin);
    if (h->pipe_ready) {
        cudaStreamDestroy(h->st_in); cudaStreamDestroy(h->st_out); cudaEventDestroy(h->ev_start);
        for (int i = 0; i < 16; ++i) { cudaEventDestroy(h->ev_in[i]); cudaEventDestroy(h->ev_k[i]); }
    }
    delete h;
}

extern "C" int cps_set_stream(cps_handle *h, void *s) {
    if (!h) return CPS_ERR_INVALID;
    h->stream = (cudaStream_t)s;
    return CPS_OK;
}

extern "C" int cps_set_physics(cps_handle *h, const float *p, int n) {
    if (!h) return CPS_ERR_INVALID;
    if (!p || n != CPS_PH_COUNT) return fail(h, CPS_ERR_INVALID, "cps_set_physics: need %d values", CPS_PH_COUNT);
    for (int i = 0; i < n; ++i)
        if (!std::isfinite(p[i])) return fail(h, CPS_ERR_INVALID, "cps_set_physics: value %d is not finite", i);
    memcpy(h->phys, p, sizeof(float) * n);
    h->L_var = p[CPS_PH_L];
    h->m_pole_var = p[CPS_PH_M_POLE];
    fold_ode(h);
    return fold_cost(h);
}

extern "C" int cps_set_cost_params(cps_handle *h, const float *w, int n) {
    if (!h) return CPS_ERR_INVALID;
    if (!w || n < 0 || n > 24) return fail(h, CPS_ERR_INVALID, "cps_set_cost_params: bad vector");
    float old[24];
    const int old_n = h->cost_in_n;
    memcpy(old, h->cost_in, sizeof(old));
    memcpy(h->cost_in, w, sizeof(float) * n);
    h->cost_in_n = n;
    const int rc = fold_cost(h);
    if (rc != CPS_OK) { memcpy(h->cost_in, old, sizeof(old)); h->cost_in_n = old_n; fold_cost(h); }
    return rc;
}

extern "C" int cps_set_mppi_params(cps_handle *h, float cc_weight, float R, float LBD, float NU, float sigma,
                                   float lo, float hi) {
    if (!h) return CPS_ERR_INVALID;
    if (!(LBD > 0.0f) || !(NU != 0.0f) || !(lo <= hi)) return fail(h, CPS_ERR_INVALID, "cps_set_mppi_params: need LBD > 0, NU != 0, lo <= hi");
    const float v[7] = {cc_weight, R, LBD, NU, sigma, lo, hi};
    memcpy(h->mppi_in, v, sizeof(v));
    fold_mppi(h);
    return CPS_OK;
}

extern "C" int cps_set_variable_parameters(cps_handle *h, float tp, float te, float L, float m_pole) {
    if (!h) return CPS_ERR_INVALID;
    if (!(L > 0.0f) || !(m_pole > 0.0f)) return fail(h, CPS_ERR_INVALID, "cps_set_variable_parameters: L and m_pole must be positive");
    h->target_position = tp; h->target_equilibrium = te; h->L_var = L; h->m_pole_var = m_pole;
    fold_ode(h);
    return fold_cost(h);
}

// ---- kernel dispatch --------------------------------------------------------------------------------
typedef void (*rollout_fn)(const RolloutArgs);
typedef void (*cost_fn)(const CostArgs);

// The MPPI solve kernels are instantiated in one translation unit per cost plugin (cps_mppi_*.cu, cps_mppi_inst.cuh).
#define CPS_DECL_MPPI(name) mppi_fn cps_pick_mppi_##name(int integ, int noise, unsigned flags, int n_sub); mppi_fn cps_pick_mppi_pair_##name(int integ, int n_sub);
CPS_DECL_MPPI(default) CPS_DECL_MPPI(qb) CPS_DECL_MPPI(gradmin) CPS_DECL_MPPI(grad) CPS_DECL_MPPI(none)
#undef CPS_DECL_MPPI
static mppi_fn pick_mppi_pair(const cps_config &c, int n_sub) {
    switch (c.cost_id) {
    case CPS_COST_DEFAULT: return cps_pick_mppi_pair_default(c.integrator, n_sub);
    case CPS_COST_QUADRATIC_BOUNDARY: return cps_pick_mppi_pair_qb(c.integrator, n_sub);
    case CPS_COST_QB_GRAD_MINIMAL: return cps_pick_mppi_pair_gradmin(c.integrator, n_sub);
    case CPS_COST_QB_GRAD: return cps_pick_mppi_pair_grad(c.integrator, n_sub);
    default: return cps_pick_mppi_pair_none(c.integrator, n_sub);
    }
}
static mppi_fn pick_mppi(const cps_config &c, int n_sub) {
    switch (c.cost_id) {
    case CPS_COST_DEFAULT: return cps_pick_mppi_default(c.integrator, c.noise_mode, c.flags, n_sub);
    case CPS_COST_QUADRATIC_BOUNDARY: return cps_pick_mppi_qb(c.integrator, c.noise_mode, c.flags, n_sub);
    case CPS_COST_QB_GRAD_MINIMAL: return cps_pick_mppi_gradmin(c.integrator, c.noise_mode, c.flags, n_sub);
    case CPS_COST_QB_GRAD: return cps_pick_mppi_grad(c.integrator, c.noise_mode, c.flags, n_sub);
    default: return cps_pick_mppi_none(c.integrator, c.noise_mode, c.flags, n_sub);
    }
}

template <int INTEG, int SC>
static rollout_fn pick_rollout2(unsigned flags) {
    const bool fd = flags & CPS_FLAG_FAST_DIV, ea = flags & CPS_FLAG_EXACT_ATAN2;
    if (fd) return ea ? rollout_kernel<INTEG, SC, true, true> : rollout_kernel<INTEG, SC, true, false>;
    return ea ? rollout_kernel<INTEG, SC, false, true> : rollout_kernel<INTEG, SC, false, false>;
}
template <int INTEG>
static rollout_fn pick_rollout1(unsigned flags) {
    switch (sc_mode(flags)) {
    case SC_ACCURATE: return pick_rollout2<INTEG, SC_ACCURATE>(flags);
    case SC_MUFU: return pick_rollout2<INTEG, SC_MUFU>(flags);
    default: return (flags & CPS_FLAG_FAST_DIV) ? rollout_kernel<INTEG, SC_ROTATE, true, false>
                                                : rollout_kernel<INTEG, SC_ROTATE, false, false>;
    }
}
static rollout_fn pick_rollout(const cps_config &c) {
    return c.integrator == CPS_EULER_V0 ? pick_rollout1<0>(c.flags) : pick_rollout1<1>(c.flags);
}
static cost_fn pick_cost(int cost) {
    switch (cost) {
    case CPS_COST_DEFAULT: return cost_kernel<COST_DEFAULT>;
    case CPS_COST_QUADRATIC_BOUNDARY: return cost_kernel<COST_QB>;
    case CPS_COST_QB_GRAD_MINIMAL: return cost_kernel<COST_GRADMIN>;
    case CPS_COST_QB_GRAD: return cost_kernel<COST_GRAD>;
    default: return nullptr;
    }
}

static void traj_strides(int layout, long long B, long long T, long long &ts_k, long long &ts_t, long long &ts_c) {
    if (layout == CPS_TIME_MAJOR) { ts_k = 1; ts_t = 6 * B; ts_c = B; }
    else { ts_k = (T + 1) * 6; ts_t = 6; ts_c = 1; }
}

// ---- MPPI ------------------------------------------------------------------------------------------
extern "C" int cps_mppi_step(cps_handle *h, const float *s_dev, const float *noise_dev, int noise_layout, float u_prev,
                             float *u_nom_dev, float *u_out_dev, float *J_out_dev, float *traj_out_dev, int traj_layout,
                             float *u_run_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    if (!s_dev || !noise_dev || !u_nom_dev || !u_out_dev) return fail(h, CPS_ERR_INVALID, "cps_mppi_step: null pointer");
    if (h->shard && !h->shard_out) return fail(h, CPS_ERR_INVALID, "cps_mppi_step: shard mode without an output buffer");
    if (h->cfg.cost_id == CPS_COST_LEGACY_MPPI) return fail(h, CPS_ERR_INVALID, "cps_mppi_step: this handle is a legacy controller_mppi_cartpole front-end; use cps_legacy_step");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (h->cfg.integrator == CPS_PREDICTOR_NEURAL)
        return cps_net_mppi_step(h, s_dev, noise_dev, noise_layout, u_prev, u_nom_dev, u_out_dev, J_out_dev, traj_out_dev,
                                 traj_layout, u_run_out_dev);
    MppiArgs a;
    a.ode = h->ode; a.cost = h->cost; a.mp = h->mp;
    a.use_inline = h->inline_s ? 1 : 0;
    for (int c = 0; c < 6; ++c) a.s_inline[c] = h->inline_s ? h->inline_s[c] : 0.0f;
    SolveIO &io = a.io;
    io.s = s_dev; io.noise = noise_dev;
    const long long K = h->cfg.num_rollouts;
    if (noise_layout == CPS_TIME_MAJOR) { io.ns_i = K; io.ns_k = 1; }
    else { io.ns_i = 1; io.ns_k = h->n_red; }
    io.u_prev = u_prev;
    io.u_nom = u_nom_dev; io.u_out = u_out_dev; io.J_out = J_out_dev; io.traj_out = traj_out_dev;
    traj_strides(traj_layout, K, h->cfg.horizon, io.ts_k, io.ts_t, io.ts_c);
    io.u_run_out = u_run_out_dev;
    io.partials = h->d_partials; io.ticket = h->d_ticket; io.nonfinite = h->d_nonfinite;
    io.shard_out = h->shard ? h->shard_out : nullptr;
    io.px = h->px;
    if (h->px.world > 1) io.px.epoch = ++h->px.epoch;
    // Large K is issue-bound, not latency-bound: two rollouts per thread in packed FP32 (same arithmetic per rollout; the
    // block sums associate pairs first).  Measured (tools/ab_pairs.py): 10 % faster at K = 65536, 10-15 % SLOWER at 16384
    // and 32768, where the solve is still bound by the latency of one rollout's dependence chain.  Needs the kernel's native noise order and no per-rollout logging outputs.
    const bool pairs = K >= CPS_MPPI_PAIR_MIN_ROLLOUTS && (K % 2) == 0 && sc_mode(h->cfg.flags) == SC_ROTATE &&
                       !(h->cfg.flags & (CPS_FLAG_FAST_DIV | CPS_FLAG_NO_PAIRS)) && h->cfg.noise_mode == CPS_NOISE_INDUCING &&
                       noise_layout == CPS_TIME_MAJOR && ((uintptr_t)noise_dev % 8) == 0 && !traj_out_dev && !u_run_out_dev;
    if (pairs) {
        const long long threads = K / 2;
        const int block = threads <= 148 * 32 * 4 ? 32 : (threads <= 148 * 64 * 8 ? 64 : 128);
        const int grid = (int)((threads + block - 1) / block);   // grid <= h->grid: the partial records fit
        const size_t smem = sizeof(float) * mppi_smem_floats(a.mp, h->cfg.cost_id, block, 2);
        if (smem > 200 * 1024) return fail(h, CPS_ERR_UNSUPPORTED, "cps_mppi_step: horizon too large for the shared-memory staging of this build");
        mppi_fn fn = pick_mppi_pair(h->cfg, a.ode.n);
        if (smem > 48 * 1024) CUDA_TRY(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        fn<<<grid, block, smem, h->stream>>>(a);
    } else {
        mppi_smem_floats(a.mp, h->cfg.cost_id, h->block, 1);   // a.mp.rs_off for this geometry
        mppi_fn fn = pick_mppi(h->cfg, a.ode.n);
        if (h->smem > 48 * 1024) CUDA_TRY(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem));
        fn<<<h->grid, h->block, h->smem, h->stream>>>(a);
    }
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

extern "C" int cps_mppi_step_host(cps_handle *h, const float *s_host, const float *noise_dev, int noise_layout,
                                  float u_prev, float *u_out_host) {
    if (!h) return CPS_ERR_INVALID;
    if (!s_host || !u_out_host) return fail(h, CPS_ERR_INVALID, "cps_mppi_step_host: null pointer");
    if (h->shard)   // a sharded solve ends with the merged partial record, not with a control: there is no u to return
        return fail(h, CPS_ERR_INVALID, "cps_mppi_step_host: the handle is in shard mode (cps_mppi_set_shard); use cps_mppi_step + cps_mppi_finalize");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (h->cfg.integrator != CPS_PREDICTOR_NEURAL && h->h_pin_dev) {
        // ODE predictors: ONE operation on the stream.  The state rides in the kernel's parameter block and the block that
        // finishes the update writes u straight into mapped pinned host memory; no copy in either direction.
        h->inline_s = s_host;
        int rc = cps_mppi_step(h, h->d_s, noise_dev, noise_layout, u_prev, h->d_unom, h->h_pin_dev + 8, nullptr, nullptr,
                               CPS_ROLLOUT_MAJOR, nullptr);
        h->inline_s = nullptr;
        if (rc != CPS_OK) return rc;
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        *u_out_host = h->h_pin[8];
        return CPS_OK;
    }
    memcpy(h->h_pin, s_host, sizeof(float) * 6);
    CUDA_TRY(h, cudaMemcpyAsync(h->d_s, h->h_pin, sizeof(float) * 6, cudaMemcpyHostToDevice, h->stream));
    int rc = cps_mppi_step(h, h->d_s, noise_dev, noise_layout, u_prev, h->d_unom, h->d_u, nullptr, nullptr,
                           CPS_ROLLOUT_MAJOR, nullptr);
    if (rc != CPS_OK) return rc;
    CUDA_TRY(h, cudaMemcpyAsync(h->h_pin + 8, h->d_u, sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    *u_out_host = h->h_pin[8];
    return CPS_OK;
}

__global__ void fill_kernel(float *p, int n, float v) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

extern "C" int cps_mppi_reset(cps_handle *h, float v) {
    if (!h) return CPS_ERR_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    fill_kernel<<<(h->cfg.horizon + 255) / 256, 256, 0, h->stream>>>(h->d_unom, h->cfg.horizon, v);   // stream-ordered, no allocation
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

extern "C" int cps_mppi_get_u_nom(cps_handle *h, float *out) {
    if (!h || !out) return CPS_ERR_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaMemcpyAsync(out, h->d_unom, sizeof(float) * h->cfg.horizon, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}

extern "C" int cps_mppi_set_u_nom(cps_handle *h, const float *in) {
    if (!h || !in) return CPS_ERR_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaMemcpyAsync(h->d_unom, in, sizeof(float) * h->cfg.horizon, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}

extern "C" float *cps_mppi_u_nom_dev(cps_handle *h) { return h ? h->d_unom : nullptr; }

extern "C" int cps_mppi_set_shard(cps_handle *h, int enabled, float *partial_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    if (enabled && !partial_out_dev) return fail(h, CPS_ERR_INVALID, "cps_mppi_set_shard: need an output buffer");
    if (enabled && h->px.world > 1) return fail(h, CPS_ERR_INVALID, "cps_mppi_set_shard: the handle exchanges over peer memory (cps_mppi_set_peers)");
    h->shard = enabled ? 1 : 0;
    h->shard_out = enabled ? partial_out_dev : nullptr;
    return CPS_OK;
}

extern "C" int cps_mppi_partial_size(const cps_handle *h) { return h ? h->n_red + 2 : -1; }

extern "C" long long cps_mppi_peer_buffer_floats(const cps_handle *h, int world) {
    if (!h || world < 1 || world > CPS_MAX_PEERS) return -1;
    return 2LL * world * (h->n_red + 2) + 2LL * world;   // 2 slots x world records, then 2 x world arrival flags
}

extern "C" int cps_mppi_set_peers(cps_handle *h, int world, int rank, float *const *peer_bufs_host) {
    if (!h) return CPS_ERR_INVALID;
    if (world <= 1 || !peer_bufs_host) {
        h->px.world = 0;
        return CPS_OK;
    }
    if (world > CPS_MAX_PEERS || rank < 0 || rank >= world)
        return fail(h, CPS_ERR_INVALID, "cps_mppi_set_peers: need 2 <= world <= CPS_MAX_PEERS and 0 <= rank < world");
    if (h->shard) return fail(h, CPS_ERR_INVALID, "cps_mppi_set_peers: the handle is in shard mode (cps_mppi_set_shard)");
    for (int r = 0; r < world; ++r)
        if (!peer_bufs_host[r]) return fail(h, CPS_ERR_INVALID, "cps_mppi_set_peers: null peer buffer");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (!h->d_px_timeouts) {
        CUDA_TRY(h, cudaMalloc(&h->d_px_timeouts, sizeof(int)));
        CUDA_TRY(h, cudaMemset(h->d_px_timeouts, 0, sizeof(int)));
    }
    for (int r = 0; r < CPS_MAX_PEERS; ++r) h->px.buf[r] = r < world ? peer_bufs_host[r] : nullptr;
    h->px.world = world; h->px.rank = rank; h->px.epoch = 0; h->px.timeouts = h->d_px_timeouts;
    return CPS_OK;
}

extern "C" int cps_mppi_peer_timeouts(cps_handle *h, int *count_out) {
    if (!h || !count_out) return CPS_ERR_INVALID;
    *count_out = 0;
    if (!h->d_px_timeouts) return CPS_OK;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaMemcpyAsync(count_out, h->d_px_timeouts, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}

extern "C" int cps_mppi_finalize(cps_handle *h, const float *partials_dev, int n_ranks, float *u_nom_dev,
                                 float *u_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    if (!partials_dev || n_ranks < 1 || !u_nom_dev || !u_out_dev) return fail(h, CPS_ERR_INVALID, "cps_mppi_finalize: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    FinalizeArgs a;
    a.mp = h->mp; a.partials = partials_dev; a.n_parts = n_ranks; a.u_nom = u_nom_dev; a.u_out = u_out_dev;
    a.shard_out = nullptr;
    const size_t smem = sizeof(float) * ((size_t)h->cfg.horizon + h->n_red + 2 + 4);  // + one float per warp
    finalize_kernel<<<1, 128, smem, h->stream>>>(a, h->cfg.noise_mode == CPS_NOISE_DIRECT);
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

// ---- open-loop rollouts -------------------------------------------------------------------------------
// B cartpoles starting at the given pointers; B_full is the batch size the time-major strides refer to (a chunk of a
// larger batch keeps the full batch's row pitch).
template <int INTEG, bool FAST>
static rollout_fn pick_pair2(bool n10, bool tr) {
    if (n10) return tr ? rollout_pair_kernel<INTEG, FAST, 10, true> : rollout_pair_kernel<INTEG, FAST, 10, false>;
    return tr ? rollout_pair_kernel<INTEG, FAST, 0, true> : rollout_pair_kernel<INTEG, FAST, 0, false>;
}
static rollout_fn pick_pair(bool v0, bool fast, bool n10, bool tr) {
    if (v0) return fast ? pick_pair2<0, true>(n10, tr) : pick_pair2<0, false>(n10, tr);
    return fast ? pick_pair2<1, true>(n10, tr) : pick_pair2<1, false>(n10, tr);
}

static int rollout_launch(cps_handle *h, const float *s0, int s0_batched, const float *Q, int q_layout, int B, int T,
                          float *traj, int traj_layout, float *fin, long long B_full = -1) {
    if (B_full < 0) B_full = B;
    RolloutArgs a;
    a.ode = h->ode;
    a.s0 = s0; a.ss_b = s0_batched ? 6 : 0;
    a.Q = Q;
    if (q_layout == CPS_TIME_MAJOR) { a.qs_b = 1; a.qs_t = B_full; }
    else { a.qs_b = T; a.qs_t = 1; }
    a.B = B; a.T = T;
    a.traj_out = traj;
    traj_strides(traj_layout, B_full, T, a.ts_k, a.ts_t, a.ts_c);
    a.final_out = fin;
    // Large time-major batches in rotation mode: two cartpoles per thread with packed FP32 (needs an even batch and
    // 8-byte aligned rows; below ~2 cartpoles per resident thread the one-per-thread kernel hides latency better).
    const bool pairs = sc_mode(h->cfg.flags) == SC_ROTATE && !(h->cfg.flags & CPS_FLAG_NO_PAIRS) && B >= CPS_PAIR_MIN_BATCH &&
                       (B % 2) == 0 && (B_full % 2) == 0 && q_layout == CPS_TIME_MAJOR &&
                       (!traj || traj_layout == CPS_TIME_MAJOR) && ((uintptr_t)Q % 8) == 0 && ((uintptr_t)traj % 8) == 0;
    if (pairs) {
        const int block = 128;
        long long grid = ((long long)(B / 2) + block - 1) / block;
        const long long max_grid = 148LL * 16 * 8;
        if (grid > max_grid) grid = max_grid;
        const bool v0 = h->cfg.integrator == CPS_EULER_V0, fast = (h->cfg.flags & CPS_FLAG_FAST_DIV) != 0;
        const bool n10 = a.ode.n == 10, tr = a.traj_out != nullptr;   // n = 10: the predictors' operating point
        rollout_fn fn = pick_pair(v0, fast, n10, tr);
        fn<<<(unsigned)grid, block, 0, h->stream>>>(a);
        h->rollout_last_kernel = 2;
    } else {
        h->rollout_last_kernel = 1;
        const int block = (B <= 148 * 32 * 4) ? 32 : 128;
        long long grid = ((long long)B + block - 1) / block;
        const long long max_grid = 148LL * 16 * 8;  // grid-stride beyond 8 full waves
        if (grid > max_grid) grid = max_grid;
        rollout_fn fn = pick_rollout(h->cfg);
        fn<<<(unsigned)grid, block, 0, h->stream>>>(a);
    }
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

extern "C" int cps_rollout(cps_handle *h, const float *s0_dev, int s0_batched, const float *Q_dev, int q_layout, int B,
                           int T, float *traj_out_dev, int traj_layout, float *final_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    if (B < 0 || T < 1) return fail(h, CPS_ERR_INVALID, "cps_rollout: need B >= 0 and T >= 1");
    if (B == 0) return CPS_OK;  // empty batch: nothing to do (pointers may be null)
    if (!s0_dev || !Q_dev) return fail(h, CPS_ERR_INVALID, "cps_rollout: null input pointer");
    if (!traj_out_dev && !final_out_dev) return fail(h, CPS_ERR_INVALID, "cps_rollout: no output requested");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (h->cfg.integrator == CPS_PREDICTOR_NEURAL) {
        if (final_out_dev) return fail(h, CPS_ERR_UNSUPPORTED, "cps_rollout: final_out is not available with the neural predictor");
        return cps_net_rollout(h, s0_dev, s0_batched, Q_dev, q_layout, B, T, nullptr, 0, traj_out_dev, traj_layout, nullptr);
    }
    return rollout_launch(h, s0_dev, s0_batched, Q_dev, q_layout, B, T, traj_out_dev, traj_layout, final_out_dev);
}

static int grow(cps_handle *h, float **p, size_t *cap, size_t need) {
    if (need <= *cap) return CPS_OK;
    if (*p) CUDA_TRY(h, cudaFree(*p));
    *p = nullptr; *cap = 0;
    CUDA_TRY(h, cudaMalloc(p, need));
    *cap = need;
    return CPS_OK;
}

extern "C" int cps_rollout_host(cps_handle *h, const float *s0_host, int s0_batched, const float *Q_host, int q_layout,
                                int B, int T, float *traj_out_host, int traj_layout, float *final_out_host) {
    if (!h) return CPS_ERR_INVALID;
    if (B < 0 || T < 1) return fail(h, CPS_ERR_INVALID, "cps_rollout_host: need B >= 0 and T >= 1");
    if (B == 0) return CPS_OK;
    if (!s0_host || !Q_host) return fail(h, CPS_ERR_INVALID, "cps_rollout_host: null input pointer");
    if (!traj_out_host && !final_out_host) return fail(h, CPS_ERR_INVALID, "cps_rollout_host: no output requested");
    if (h->cfg.integrator == CPS_PREDICTOR_NEURAL && final_out_host)
        return fail(h, CPS_ERR_UNSUPPORTED, "cps_rollout_host: final_out is not available with the neural predictor");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t n_s0 = sizeof(float) * 6 * (s0_batched ? (size_t)B : 1), n_Q = sizeof(float) * (size_t)B * T;
    const size_t n_traj = sizeof(float) * (size_t)B * (T + 1) * 6, n_fin = sizeof(float) * (size_t)B * 6;
    int rc;
    if ((rc = grow(h, &h->d_rs0, &h->cap_rs0, n_s0)) != CPS_OK) return rc;
    if ((rc = grow(h, &h->d_rQ, &h->cap_rQ, n_Q)) != CPS_OK) return rc;
    if (traj_out_host && (rc = grow(h, &h->d_rtraj, &h->cap_rtraj, n_traj)) != CPS_OK) return rc;
    if (final_out_host && (rc = grow(h, &h->d_rfinal, &h->cap_rfinal, n_fin)) != CPS_OK) return rc;
    // Large ODE batches: split into chunks and pipeline copy-in / kernel / copy-out on three streams, so that the
    // host->device copies of chunk c+1 and the kernel of chunk c run under the device->host copy of chunk c-1 (PCIe
    // is full duplex; the trajectory copy-out is the long pole).  Time-major arrays are copied as 2-D slabs.
    const int n_chunks = (h->cfg.integrator != CPS_PREDICTOR_NEURAL && B >= (1 << 16)) ? 8 : 1;
    if (n_chunks > 1) {
        if (!h->pipe_ready) {
            CUDA_TRY(h, cudaStreamCreateWithFlags(&h->st_in, cudaStreamNonBlocking));
            CUDA_TRY(h, cudaStreamCreateWithFlags(&h->st_out, cudaStreamNonBlocking));
            CUDA_TRY(h, cudaEventCreateWithFlags(&h->ev_start, cudaEventDisableTiming));
            for (int i = 0; i < 16; ++i) {
                CUDA_TRY(h, cudaEventCreateWithFlags(&h->ev_in[i], cudaEventDisableTiming));
                CUDA_TRY(h, cudaEventCreateWithFlags(&h->ev_k[i], cudaEventDisableTiming));
            }
            h->pipe_ready = 1;
        }
        // everything queued on the handle's stream so far happens before the pipeline starts
        CUDA_TRY(h, cudaEventRecord(h->ev_start, h->stream));
        CUDA_TRY(h, cudaStreamWaitEvent(h->st_in, h->ev_start, 0));
        CUDA_TRY(h, cudaStreamWaitEvent(h->st_out, h->ev_start, 0));
        const size_t rows = (size_t)(T + 1) * 6, pitch = sizeof(float) * (size_t)B;
        if (!s0_batched) CUDA_TRY(h, cudaMemcpyAsync(h->d_rs0, s0_host, n_s0, cudaMemcpyHostToDevice, h->st_in));
        for (int c = 0; c < n_chunks; ++c) {
            const long long b0 = (long long)B * c / n_chunks, b1 = (long long)B * (c + 1) / n_chunks, nb = b1 - b0;
            if (s0_batched)
                CUDA_TRY(h, cudaMemcpyAsync(h->d_rs0 + b0 * 6, s0_host + b0 * 6, sizeof(float) * 6 * nb, cudaMemcpyHostToDevice, h->st_in));
            if (q_layout == CPS_TIME_MAJOR)
                CUDA_TRY(h, cudaMemcpy2DAsync(h->d_rQ + b0, pitch, Q_host + b0, pitch, sizeof(float) * nb, T, cudaMemcpyHostToDevice, h->st_in));
            else
                CUDA_TRY(h, cudaMemcpyAsync(h->d_rQ + b0 * T, Q_host + b0 * T, sizeof(float) * nb * T, cudaMemcpyHostToDevice, h->st_in));
            CUDA_TRY(h, cudaEventRecord(h->ev_in[c], h->st_in));
            CUDA_TRY(h, cudaStreamWaitEvent(h->stream, h->ev_in[c], 0));
            const float *q_c = h->d_rQ + (q_layout == CPS_TIME_MAJOR ? b0 : b0 * T);
            float *traj_c = traj_out_host ? h->d_rtraj + (traj_layout == CPS_TIME_MAJOR ? b0 : b0 * (long long)rows) : nullptr;
            float *fin_c = final_out_host ? h->d_rfinal + b0 * 6 : nullptr;
            rc = rollout_launch(h, h->d_rs0 + (s0_batched ? b0 * 6 : 0), s0_batched, q_c, q_layout, (int)nb, T, traj_c,
                                traj_layout, fin_c, B);
            if (rc != CPS_OK) return rc;
            CUDA_TRY(h, cudaEventRecord(h->ev_k[c], h->stream));
            CUDA_TRY(h, cudaStreamWaitEvent(h->st_out, h->ev_k[c], 0));
            if (traj_out_host) {
                if (traj_layout == CPS_TIME_MAJOR)
                    CUDA_TRY(h, cudaMemcpy2DAsync(traj_out_host + b0, pitch, h->d_rtraj + b0, pitch, sizeof(float) * nb, rows, cudaMemcpyDeviceToHost, h->st_out));
                else
                    CUDA_TRY(h, cudaMemcpyAsync(traj_out_host + b0 * rows, h->d_rtraj + b0 * rows, sizeof(float) * nb * rows, cudaMemcpyDeviceToHost, h->st_out));
            }
            if (final_out_host)
                CUDA_TRY(h, cudaMemcpyAsync(final_out_host + b0 * 6, h->d_rfinal + b0 * 6, sizeof(float) * 6 * nb, cudaMemcpyDeviceToHost, h->st_out));
        }
        CUDA_TRY(h, cudaStreamSynchronize(h->st_out));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        return CPS_OK;
    }
    CUDA_TRY(h, cudaMemcpyAsync(h->d_rs0, s0_host, n_s0, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(h->d_rQ, Q_host, n_Q, cudaMemcpyHostToDevice, h->stream));
    if (h->cfg.integrator == CPS_PREDICTOR_NEURAL)
        rc = cps_net_rollout(h, h->d_rs0, s0_batched, h->d_rQ, q_layout, B, T, nullptr, 0, h->d_rtraj, traj_layout, nullptr);
    else
        rc = rollout_launch(h, h->d_rs0, s0_batched, h->d_rQ, q_layout, B, T, traj_out_host ? h->d_rtraj : nullptr,
                            traj_layout, final_out_host ? h->d_rfinal : nullptr);
    if (rc != CPS_OK) return rc;
    if (traj_out_host) CUDA_TRY(h, cudaMemcpyAsync(traj_out_host, h->d_rtraj, n_traj, cudaMemcpyDeviceToHost, h->stream));
    if (final_out_host) CUDA_TRY(h, cudaMemcpyAsync(final_out_host, h->d_rfinal, n_fin, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}

// ---- standalone cost ----------------------------------------------------------------------------------
static int cost_launch(cps_handle *h, const float *traj, int rows, const float *Q, float u_prev, int K, int T, float *J,
                       float *stage, int unshifted) {
    if (!traj || !Q) return fail(h, CPS_ERR_INVALID, "cost: null input pointer");
    if (K < 0 || T < 1) return fail(h, CPS_ERR_INVALID, "cost: need K >= 0 and T >= 1");
    cost_fn fn = pick_cost(h->cfg.cost_id);
    if (!fn) return fail(h, CPS_ERR_NOT_CONFIGURED, "cost: handle was created with CPS_COST_NONE");
    if (K == 0) return CPS_OK;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CostArgs a;
    a.cost = h->cost; a.traj = traj; a.Q = Q; a.u_prev = u_prev; a.K = K; a.T = T; a.rows = rows;
    a.inv_T1 = 1.0f / (float)(T + 1);
    a.J = J; a.stage = stage; a.unshifted = unshifted;
    const size_t smem = J ? sizeof(float) * (size_t)row_sum_slots(T + 1) * 128 : 0;
    if (smem > 48 * 1024) CUDA_TRY(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fn<<<(K + 127) / 128, 128, smem, h->stream>>>(a);
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

extern "C" int cps_trajectory_cost(cps_handle *h, const float *traj_dev, const float *Q_dev, float u_prev, int K, int T,
                                   float *J_dev) {
    if (!h) return CPS_ERR_INVALID;
    if (!J_dev) return fail(h, CPS_ERR_INVALID, "cps_trajectory_cost: null output");
    return cost_launch(h, traj_dev, T + 1, Q_dev, u_prev, K, T, J_dev, nullptr, 0);
}

extern "C" int cps_stage_cost(cps_handle *h, const float *states_dev, int rows, const float *Q_dev, float u_prev, int K,
                              int T, int unshifted, float *stage_dev) {
    if (!h) return CPS_ERR_INVALID;
    if (!stage_dev) return fail(h, CPS_ERR_INVALID, "cps_stage_cost: null output");
    if (rows != T && rows != T + 1) return fail(h, CPS_ERR_INVALID, "cps_stage_cost: rows must be T or T+1");
    return cost_launch(h, states_dev, rows, Q_dev, u_prev, K, T, nullptr, stage_dev, unshifted);
}

extern "C" int cps_terminal_cost(cps_handle *h, const float *states_dev, int K, float *out_dev) {
    if (!h) return CPS_ERR_INVALID;
    if (!states_dev || !out_dev || K < 0) return fail(h, CPS_ERR_INVALID, "cps_terminal_cost: bad argument");
    if (h->cfg.cost_id == CPS_COST_NONE) return fail(h, CPS_ERR_NOT_CONFIGURED, "cost: handle was created with CPS_COST_NONE");
    if (K == 0) return CPS_OK;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const int grid = (K + 127) / 128;
    switch (h->cfg.cost_id) {
    case CPS_COST_LEGACY_MPPI:  // phi() is default.py's terminal cost (controller_mppi_cartpole.py:271-298)
    case CPS_COST_DEFAULT: terminal_cost_kernel<COST_DEFAULT><<<grid, 128, 0, h->stream>>>(h->cost, states_dev, K, out_dev); break;
    case CPS_COST_QUADRATIC_BOUNDARY: terminal_cost_kernel<COST_QB><<<grid, 128, 0, h->stream>>>(h->cost, states_dev, K, out_dev); break;
    case CPS_COST_QB_GRAD_MINIMAL: terminal_cost_kernel<COST_GRADMIN><<<grid, 128, 0, h->stream>>>(h->cost, states_dev, K, out_dev); break;
    default: terminal_cost_kernel<COST_GRAD><<<grid, 128, 0, h->stream>>>(h->cost, states_dev, K, out_dev); break;
    }
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

// ---- roofline denominators, measured in place -------------------------------------------------------------
// FP32 FMA peak: 8 independent FFMA chains per thread, full occupancy.  2 flops per FFMA.  Unrolled 32 times: the
// constant-operand FFMA issues every cycle, so at the round-1 unroll of 4 the three loop instructions per 32 FFMAs capped
// the probe at 91 % of the pipe (66.9 TFLOP/s where the device does ~73).
__global__ void __launch_bounds__(256) fp32_peak_kernel(float *out, int iters, float a, float b) {
    float x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
#pragma unroll 32
    for (int i = 0; i < iters; ++i) {
        x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
        x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
    }
    const float r = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (r == 123.456f) out[0] = r;  // never true; keeps the chains alive
}
// MUFU peak: independent ex2.approx chains.
__global__ void __launch_bounds__(256) mufu_peak_kernel(float *out, int iters) {
    float x0 = threadIdx.x * 1e-3f, x1 = x0 + 0.1f, x2 = x0 + 0.2f, x3 = x0 + 0.3f;
#pragma unroll 4
    for (int i = 0; i < iters; ++i) {
        asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(x0));
        asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(x1));
        asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(x2));
        asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(x3));
    }
    const float r = (x0 + x1) + (x2 + x3);
    if (r == 123.456f) out[0] = r;
}

extern "C" int cps_measure_peaks(cps_handle *h, double *fp32_tflops, double *mufu_gops) {
    if (!h || !fp32_tflops || !mufu_gops) return CPS_ERR_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    cudaDeviceProp prop;
    CUDA_TRY(h, cudaGetDeviceProperties(&prop, h->cfg.device));
    const int grid = prop.multiProcessorCount * 8, block = 256, iters = 1 << 14;
    cudaEvent_t e0, e1;
    CUDA_TRY(h, cudaEventCreate(&e0));
    CUDA_TRY(h, cudaEventCreate(&e1));
    float ms = 0.0f;
    double best_f = 0.0, best_m = 0.0;
    for (int rep = 0; rep < 6; ++rep) {
        CUDA_TRY(h, cudaEventRecord(e0, h->stream));
        fp32_peak_kernel<<<grid, block, 0, h->stream>>>(h->d_u, iters, 1.000001f, 1e-7f);
        CUDA_TRY(h, cudaEventRecord(e1, h->stream));
        CUDA_TRY(h, cudaEventSynchronize(e1));
        CUDA_TRY(h, cudaEventElapsedTime(&ms, e0, e1));
        const double f = 2.0 * 8.0 * (double)iters * grid * block / (ms * 1e-3) / 1e12;
        if (rep > 0 && f > best_f) best_f = f;
        CUDA_TRY(h, cudaEventRecord(e0, h->stream));
        mufu_peak_kernel<<<grid, block, 0, h->stream>>>(h->d_u, iters);
        CUDA_TRY(h, cudaEventRecord(e1, h->stream));
        CUDA_TRY(h, cudaEventSynchronize(e1));
        CUDA_TRY(h, cudaEventElapsedTime(&ms, e0, e1));
        const double m = 4.0 * (double)iters * grid * block / (ms * 1e-3) / 1e9;
        if (rep > 0 && m > best_m) best_m = m;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    CUDA_TRY(h, cudaGetLastError());
    *fp32_tflops = best_f;
    *mufu_gops = best_m;
    return CPS_OK;
}

// ---- self-test of sincos_folded ---------------------------------------------------------------------------
// Every float of [-pi, pi] (both signs of every bit pattern up to fl32(pi)): sincos_folded against the math library's
// sincosf and cosf, bit for bit.
__global__ void __launch_bounds__(256) sincos_selftest_kernel(unsigned long long *mismatches) {
    const unsigned last = 0x40490fdbu;   // fl32(pi)
    unsigned long long bad = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i <= last;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        for (unsigned sign = 0; sign < 2; ++sign) {
            const float x = __uint_as_float((unsigned)i | (sign << 31));
            float s0, c0, s1, c1;
            sincosf(x, &s0, &c0);
            sincos_folded(x, s1, c1);
            bad += (__float_as_uint(s0) != __float_as_uint(s1)) + (__float_as_uint(c0) != __float_as_uint(c1)) +
                   (__float_as_uint(cosf(x)) != __float_as_uint(c1));
        }
    }
    if (bad) atomicAdd(mismatches, bad);
}

extern "C" int cps_selftest_sincos(cps_handle *h, long long *mismatches_out) {
    if (!h || !mismatches_out) return CPS_ERR_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    unsigned long long *d = nullptr, host = 0;
    CUDA_TRY(h, cudaMalloc(&d, sizeof(*d)));
    cudaMemsetAsync(d, 0, sizeof(*d), h->stream);
    sincos_selftest_kernel<<<148 * 8, 256, 0, h->stream>>>(d);
    h->launches += 1;
    cudaError_t e = cudaMemcpyAsync(&host, d, sizeof(host), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(d);
    CUDA_TRY(h, e);
    *mismatches_out = (long long)host;
    return CPS_OK;
}

// ---- diagnostics ---------------------------------------------------------------------------------------
extern "C" long long cps_launch_count(const cps_handle *h) { return h ? h->launches : -1; }
extern "C" int cps_net_last_kernel(const cps_handle *h) { return h ? h->net_last_kernel : -1; }
extern "C" int cps_rollout_last_kernel(const cps_handle *h) { return h ? h->rollout_last_kernel : -1; }

extern "C" int cps_nonfinite_costs(cps_handle *h, int *count_out) {
    if (!h || !count_out) return CPS_ERR_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaMemcpyAsync(count_out, h->d_nonfinite, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}
