// cps_legacy_fleet.cu -- E closed-loop experiments under the legacy controller_mppi_cartpole (SURVEY.md 8f, row f2;
// `mppi-cartpole` in Control_Toolkit_ASF/config_controllers.yml:9-30), advanced together.
//
// One controller period of EVERY experiment is one launch, whatever E:
//   solve periods (iteration % update_every == 0)
//     legacy_fleet_kernel      grid (h->grid, E), block h->block: each experiment's blocks are those of cps_legacy_step
//                              for K.  Rollout thread k stages its own T perturbations in shared memory (the SAMPLING_TYPE
//                              transform of its raw draws, Philox or supplied), then legacy_mppi_kernel's iteration
//                              (legacy_stage, control_step, block_partials, merge_partials) from the experiment's state,
//                              u, u_prev and target position; the experiment's last block updates and shifts u, applies
//                              the actuator noise and runs the plant period (plant_period_held) with the result;
//   other periods
//     legacy_fleet_advance_kernel  one thread per experiment: legacy_advance_kernel's shift, the actuator noise, the plant.
// Raw draws per rollout and period (controller_mppi_cartpole.py:392-457): T standard normals (iid, random_walk), T uniforms
// in [-1, 1) (uniform), 1 normal (repeated), ceil(T / 10) + 1 normals (interpolated, the knots 0, 10, 20, ...); Philox
// counter (rollout, LEGACY_DRAWS + group of four, period, experiment_offset + e).  The actuator uniform of a period:
// (0, LEGACY_ACT, period, experiment_offset + e).
#include <cuda_runtime.h>

#include <cmath>
#include <cstring>
#include <new>

#include "cps_internal.cuh"
#include "cps_legacy.cuh"
#include "cps_plant.cuh"

#define LEGACY_INTERP_STEP 10   // `step` of the interpolated sampler (:431)

// Dynamic shared memory (floats) of cps_legacy_step's block: [T] u, [T] u_prev, [nwarps][T + 2] reduction scratch reused
// by the merge (+ [nwarps])
__host__ __device__ inline size_t legacy_smem_floats(int T, int block) {
    const size_t nwarps = block / 32;
    return (size_t)2 * T + nwarps * (T + 2) + (size_t)T + 4 + nwarps;
}

// legacy_interp_kernel's value j = 1 .. step - 1 steps past the knot y_lo towards the next knot y_hi (scipy's interp1d in
// float64, rounded to float32)
__device__ __forceinline__ float legacy_interp_between(int j, int step, float y_lo, float y_hi) {
    const double w_hi = __ddiv_rn((double)j, (double)step), w_lo = __ddiv_rn((double)(step - j), (double)step);
    return __double2float_rn(__dadd_rn(__dmul_rn(w_hi, (double)y_hi), __dmul_rn(w_lo, (double)y_lo)));
}

static inline int legacy_fleet_n_draws(int sampling, int T) {
    switch (sampling) {
    case CPS_LEGACY_SAMPLING_REPEATED: return 1;
    case CPS_LEGACY_SAMPLING_INTERPOLATED: return (T + LEGACY_INTERP_STEP - 1) / LEGACY_INTERP_STEP + 1;
    default: return T;
    }
}

// One rollout's perturbations du[t * ds], t < T, from its raw draws raw[i * rs] (standard normals z, or uniforms v for
// "uniform"), in the reference's arithmetic: stdev is numpy's float64 scalar, so stdev * z and the random walk's sum are
// float64, rounded to float32 where the reference assigns them into its float32 array; the interpolated knots are
// fl32(stdev z_j) and the values between them legacy_interp_between's.  raw may alias du except for "interpolated".
__device__ __forceinline__ void legacy_perturb(int sampling, double stdev, const float *raw, long long rs, float *du,
                                               long long ds, int T) {
    switch (sampling) {
    case CPS_LEGACY_SAMPLING_RANDOM_WALK: {
        float prev = __double2float_rn(__dmul_rn(stdev, (double)raw[0]));
        du[0] = prev;
        for (int t = 1; t < T; ++t) {
            prev = __double2float_rn(__dadd_rn((double)prev, __dmul_rn(stdev, (double)raw[t * rs])));
            du[t * ds] = prev;
        }
        break;
    }
    case CPS_LEGACY_SAMPLING_UNIFORM:
        for (int t = 0; t < T; ++t) du[t * ds] = raw[t * rs];
        break;
    case CPS_LEGACY_SAMPLING_REPEATED: {
        const float v = __double2float_rn(__dmul_rn(stdev, (double)raw[0]));
        for (int t = 0; t < T; ++t) du[t * ds] = v;
        break;
    }
    case CPS_LEGACY_SAMPLING_INTERPOLATED: {
        float y_lo = __double2float_rn(__dmul_rn(stdev, (double)raw[0])), y_hi = y_lo;
        for (int t = 0; t < T; ++t) {
            const int lo = t / LEGACY_INTERP_STEP, j = t - lo * LEGACY_INTERP_STEP;
            if (j == 0) {
                y_lo = __double2float_rn(__dmul_rn(stdev, (double)raw[lo * rs]));
                y_hi = __double2float_rn(__dmul_rn(stdev, (double)raw[(lo + 1) * rs]));
                du[t * ds] = y_lo;
            } else {
                du[t * ds] = legacy_interp_between(j, LEGACY_INTERP_STEP, y_lo, y_hi);
            }
        }
        break;
    }
    default:   // iid, the reference's default branch
        for (int t = 0; t < T; ++t) du[t * ds] = __double2float_rn(__dmul_rn(stdev, (double)raw[t * rs]));
    }
}

// The raw draws of rollout k of global experiment e_global in `period`, n of them at dst[i * stride]
__device__ __forceinline__ void legacy_philox_draws(int sampling, unsigned long long seed, int k, unsigned period,
                                                    unsigned e_global, int n, float *dst, long long stride) {
    if (sampling == CPS_LEGACY_SAMPLING_UNIFORM)
        philox_uniforms(seed, (unsigned)k, LEGACY_DRAWS, period, e_global, n, dst, stride, -1.0f, 2.0f);
    else
        philox_normals(seed, (unsigned)k, LEGACY_DRAWS, period, e_global, n, dst, stride);
}

// Actuator noise and clipping of the mirror (controller_mppi_cartpole_b200.step): Q, p_Q and the uniform v are python
// floats there, so Q (1 + p_Q v) is float64, rounded to float32, then np.clip to [-1, 1] (NaN stays NaN).
__device__ __forceinline__ float legacy_actuate(float Q, double p_Q, float v) {
    const float q = __double2float_rn(__dmul_rn((double)Q, __dadd_rn(1.0, __dmul_rn(p_Q, (double)v))));
    return (q != q) ? q : fminf(fmaxf(q, -1.0f), 1.0f);
}

struct LegacyFleetArgs {
    OdeParams ode;
    CostParams cost;            // the handle's, folded at each cps_legacy_fleet_step; target_position per experiment
    MppiParams mp;
    PlantParams plant;
    int sampling, n_draws;
    double stdev, p_Q;
    float *s;                   // [E][8]
    float *u, *u_prev;          // [E][T] each
    float *Q;                   // [E] <- the period's control (after the actuator noise)
    const float *tp, *te;       // [E] targets of this period (null: 0 / +1)
    const float *draws;         // supplied raw draws [E][K][n_draws] of this period, or null: Philox
    const float *act;           // supplied actuator uniforms [E] of this period, or null: Philox
    unsigned long long seed;
    unsigned period, e_offset;
    float *partials;            // [E][grid][T + 2]
    unsigned *tickets;          // [E]
    int *nonfinite;
    float *record;              // [E][CPS_FLEET_RECORD] of this period, or null
    float *S_out;               // [E][K] or null
    double time;                // period * dt_control
};

// After the solve (or the shift) of experiment e, one thread: the actuator noise on the controller's Q, Q into a.Q[e], the
// plant period with Q held
__device__ __forceinline__ void legacy_fleet_finish(const LegacyFleetArgs &a, int e, float Qc) {
    float v;
    if (a.act) v = a.act[e];
    else philox_uniforms(a.seed, 0u, LEGACY_ACT, a.period, a.e_offset + (unsigned)e, 1, &v, 1, -1.0f, 2.0f);
    const float Q = legacy_actuate(Qc, a.p_Q, v);
    a.Q[e] = Q;
    plant_period_held(a.plant, a.s, e, Q, a.record, a.time, a.tp, a.te);
}

// smem: legacy_smem_floats, then (even offset) [T][blockDim.x] perturbations, then with Philox and "interpolated"
// [n_draws][blockDim.x] knot draws.
template <int INTEG, bool PHILOX>
__global__ void __launch_bounds__(256, 4) legacy_fleet_kernel(const __grid_constant__ LegacyFleetArgs a) {
    extern __shared__ float smem[];
    __shared__ CostParams s_cost;
    const MppiParams &mp = a.mp;
    const int T = mp.T, K = mp.K;
    const int e = blockIdx.y, tid = threadIdx.x, nb = blockDim.x;
    float *s_u = smem;
    float *s_up = s_u + T;
    float *s_red = s_up + T;
    float *s_du = smem + ((legacy_smem_floats(T, nb) + 1) & ~(size_t)1);
    float *u = a.u + (size_t)e * T, *u_prev = a.u_prev + (size_t)e * T;
    if (tid == 0) {
        s_cost = a.cost;
        s_cost.target_position = a.tp ? a.tp[e] : 0.0f;
    }
    for (int t = tid; t < T; t += nb) { s_u[t] = u[t]; s_up[t] = u_prev[t]; }
    // this rollout's perturbations into column tid (inactive threads of the last block: those of rollout K - 1)
    const int k = (int)(blockIdx.x * nb) + tid;
    const int kc = min(k, K - 1);
    float *col = s_du + tid;
    if (PHILOX) {
        float *raw = (a.sampling == CPS_LEGACY_SAMPLING_INTERPOLATED) ? s_du + (size_t)T * nb + tid : col;
        legacy_philox_draws(a.sampling, a.seed, kc, a.period, a.e_offset + (unsigned)e, a.n_draws, raw, nb);
        legacy_perturb(a.sampling, a.stdev, raw, nb, col, nb, T);
    } else {
        legacy_perturb(a.sampling, a.stdev, a.draws + ((size_t)e * K + kc) * a.n_draws, 1, col, nb, T);
    }
    __syncthreads();

    // legacy_mppi_kernel's iteration on this experiment (the same statements, in the same order)
    const bool active = k < K;
    const float *nz = s_du + tid;
    State z = load_state(a.s + (size_t)e * 8);
    const OdeParams ode = pin_params(a.ode, z.th);
    float c_cost = cosf(z.th);  // q() takes np.cos of the stored angle (:131-135)
    float S = 0.0f;
    float du_next = nz[0];
#pragma unroll 1
    for (int t = 0; t < T; ++t) {
        const float du = du_next;
        if (t + 1 < T) du_next = nz[(long long)(t + 1) * nb];  // prefetch under the integration
        const float un = s_u[t];
        S += legacy_stage(s_cost, mp, c_cost, z.w, z.x, z.v, un, du, s_up[t]);
        control_step<INTEG, SC_ROTATE, false, false>(ode, z, un + du);  // the rollout sees the UNCLIPPED input (:190-192)
        c_cost = z.c;
    }
    S += terminal_cost<COST_DEFAULT>(s_cost, z.th, z.x);  // phi() (:271-298) is default.py's terminal cost
    if (active) {
        if (a.S_out) a.S_out[(size_t)e * K + k] = S;
        if (!isfinite(S)) atomicAdd(a.nonfinite, 1);
    }
    unsigned *ticket = a.tickets + e;
    float *partials = a.partials + (size_t)e * gridDim.x * (mp.n_red + 2);
    if (!block_partials(mp, S, active, nz, nb, s_red, partials, ticket, blockIdx.x, gridDim.x)) return;
    merge_partials(mp, partials, gridDim.x, s_red);
    // update_inputs (:325-335): u += sum_k w_k du_k / sum_k w_k, no clipping
    const float invS = 1.0f / s_red[0];
    for (int t = tid; t < T; t += nb) s_u[t] = fmaf(s_red[1 + t], invS, s_u[t]);
    __syncthreads();
    // Q = u[0]; u_prev <- u; u <- [u[1:], 0]  (:521, :531-536)
    for (int t = tid; t < T; t += nb) {
        const float un = s_u[t];
        u_prev[t] = un;
        u[t] = (t + 1 < T) ? s_u[t + 1] : 0.0f;
    }
    if (tid == 0) {
        *ticket = 0u;
        legacy_fleet_finish(a, e, s_u[0]);
    }
}

// A period without a solve: legacy_advance_kernel's shift (Q = u[0], u_prev <- u, u <- [u[1:], 0]), then as above
__global__ void __launch_bounds__(128) legacy_fleet_advance_kernel(const __grid_constant__ LegacyFleetArgs a, int E) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    const int T = a.mp.T;
    float *u = a.u + (size_t)e * T, *u_prev = a.u_prev + (size_t)e * T;
    const float Qc = u[0];
    for (int t = 0; t < T; ++t) {
        u_prev[t] = u[t];
        u[t] = (t + 1 < T) ? u[t + 1] : 0.0f;
    }
    legacy_fleet_finish(a, e, Qc);
}

// Materialised perturbations [E][K][T] from raw draws [E][K][n_draws] (cps_legacy_fleet_perturbations), one thread per
// (rollout, experiment): legacy_perturb as the fleet's rollouts run it
__global__ void __launch_bounds__(256) legacy_fleet_perturb_kernel(const float *raw, float *out, int E, int K, int T,
                                                                   int n_draws, int sampling, double stdev) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)E * K) return;
    legacy_perturb(sampling, stdev, raw + i * n_draws, 1, out + i * T, 1, T);
}

struct LegacyFleetState {
    FleetCore core;             // d_uprev: each experiment's last control Q
    int sampling, update_every, n_draws;
    double stdev, p_Q;
    size_t smem;
    long long reset_period;     // the iteration counter is period - reset_period
    float *d_u, *d_up;          // [E][T] u, u_prev
    float *d_partials;          // [E][h->grid][T + 2]
    unsigned *d_tickets;        // [E]
    float *d_raw;               // [E][K][n_draws] scratch of cps_legacy_fleet_perturbations (allocated on first use)
};

void cps_legacy_fleet_free(cps_handle *h) {
    LegacyFleetState *F = h->lfleet;
    if (!F) return;
    fleet_core_free(F->core);
    cudaFree(F->d_u); cudaFree(F->d_up); cudaFree(F->d_partials); cudaFree(F->d_tickets); cudaFree(F->d_raw);
    delete F;
    h->lfleet = nullptr;
}

static LegacyFleetState *legacy_fleet(cps_handle *h, const char *who, bool ready) {
    if (legacy_check(h, who) != CPS_OK) return nullptr;
    LegacyFleetState *F = h->lfleet;
    if (!F || (ready && !F->core.ready)) {
        fail(h, CPS_ERR_NOT_CONFIGURED, "%s: no legacy fleet%s", who,
             ready ? " with states (cps_legacy_fleet_create, cps_legacy_fleet_set_states)" : " (cps_legacy_fleet_create)");
        return nullptr;
    }
    return F;
}

extern "C" int cps_legacy_fleet_create(cps_handle *h, const cps_legacy_fleet_config *cfg) {
    if (!h) return CPS_ERR_INVALID;
    const char *who = "cps_legacy_fleet_create";
    int rc;
    if ((rc = legacy_check(h, who)) != CPS_OK) return rc;
    if (!cfg || cfg->struct_size != (int)sizeof(cps_legacy_fleet_config))
        return fail(h, CPS_ERR_INVALID, "%s: cps_legacy_fleet_config size mismatch", who);
    FleetCore core;
    if ((rc = fleet_core_init(h, core, cfg->n_experiments, cfg->sim_substeps, cfg->draw_source, cfg->dt_simulation, cfg->seed,
                              cfg->experiment_offset, who)) != CPS_OK)
        return rc;
    if (core.E > 65535) return fail(h, CPS_ERR_INVALID, "%s: at most 65535 experiments per handle", who);
    if (cfg->sampling_type < CPS_LEGACY_SAMPLING_IID || cfg->sampling_type > CPS_LEGACY_SAMPLING_INTERPOLATED)
        return fail(h, CPS_ERR_INVALID, "%s: unknown sampling type %d", who, cfg->sampling_type);
    if (cfg->update_every < 1) return fail(h, CPS_ERR_INVALID, "%s: update_every must be >= 1", who);
    const int T = h->cfg.horizon;
    const int n_draws = legacy_fleet_n_draws(cfg->sampling_type, T);
    const size_t staged = (size_t)T + ((core.philox && cfg->sampling_type == CPS_LEGACY_SAMPLING_INTERPOLATED) ? n_draws : 0);
    const size_t smem = sizeof(float) * (((legacy_smem_floats(T, h->block) + 1) & ~(size_t)1) + staged * h->block);
    if (smem > 227 * 1024) return fail(h, CPS_ERR_UNSUPPORTED, "%s: horizon too large for shared memory", who);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    cps_legacy_fleet_free(h);
    LegacyFleetState *F = new (std::nothrow) LegacyFleetState();
    if (!F) return fail(h, CPS_ERR_INVALID, "%s: out of host memory", who);
    memset(F, 0, sizeof(*F));
    F->core = core;
    F->sampling = cfg->sampling_type; F->update_every = cfg->update_every; F->n_draws = n_draws;
    F->stdev = cfg->stdev; F->p_Q = cfg->p_Q;
    F->smem = smem;
    h->lfleet = F;
    const size_t E = core.E;
    if ((rc = fleet_core_alloc(h, F->core)) != CPS_OK) return rc;
    CUDA_TRY(h, cudaMalloc(&F->d_u, sizeof(float) * E * T));
    CUDA_TRY(h, cudaMalloc(&F->d_up, sizeof(float) * E * T));
    CUDA_TRY(h, cudaMalloc(&F->d_partials, sizeof(float) * E * h->grid * (T + 2)));
    CUDA_TRY(h, cudaMalloc(&F->d_tickets, sizeof(unsigned) * E));
    CUDA_TRY(h, cudaMemsetAsync(F->d_u, 0, sizeof(float) * E * T, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(F->d_up, 0, sizeof(float) * E * T, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(F->d_tickets, 0, sizeof(unsigned) * E, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}

extern "C" int cps_legacy_fleet_set_states(cps_handle *h, const float *s_host, long long period) {
    if (!h) return CPS_ERR_INVALID;
    const char *who = "cps_legacy_fleet_set_states";
    LegacyFleetState *F = legacy_fleet(h, who, false);
    if (!F) return CPS_ERR_NOT_CONFIGURED;
    int rc;
    if ((rc = fleet_core_set_states(h, F->core, s_host, period, who)) != CPS_OK) return rc;
    // every experiment as a freshly configured controller (configure, :351-391): u = u_prev = 0, iteration restarted
    const size_t n = sizeof(float) * (size_t)F->core.E * h->cfg.horizon;
    CUDA_TRY(h, cudaMemsetAsync(F->d_u, 0, n, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(F->d_up, 0, n, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    F->reset_period = period;
    F->core.ready = 1;
    return CPS_OK;
}

extern "C" int cps_legacy_fleet_get_states(cps_handle *h, float *s_host, float *Q_host) {
    if (!h) return CPS_ERR_INVALID;
    LegacyFleetState *F = legacy_fleet(h, "cps_legacy_fleet_get_states", true);
    return F ? fleet_core_get_states(h, F->core, s_host, Q_host, "cps_legacy_fleet_get_states") : CPS_ERR_NOT_CONFIGURED;
}

extern "C" int cps_legacy_fleet_get_inputs(cps_handle *h, float *u_host, float *u_prev_host) {
    if (!h) return CPS_ERR_INVALID;
    LegacyFleetState *F = legacy_fleet(h, "cps_legacy_fleet_get_inputs", true);
    if (!F) return CPS_ERR_NOT_CONFIGURED;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t n = sizeof(float) * (size_t)F->core.E * h->cfg.horizon;
    if (u_host) CUDA_TRY(h, cudaMemcpyAsync(u_host, F->d_u, n, cudaMemcpyDeviceToHost, h->stream));
    if (u_prev_host) CUDA_TRY(h, cudaMemcpyAsync(u_prev_host, F->d_up, n, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}

static bool legacy_fleet_solves(const LegacyFleetState *F, long long period) {
    return (period - F->reset_period) % F->update_every == 0;
}

extern "C" int cps_legacy_fleet_step(cps_handle *h, int n_periods, const float *tp_dev, const float *te_dev,
                                     const float *draws_dev, const float *act_draws_dev, float *record_dev, float *S_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    const char *who = "cps_legacy_fleet_step";
    LegacyFleetState *F = legacy_fleet(h, who, true);
    if (!F) return CPS_ERR_NOT_CONFIGURED;
    if (n_periods < 0) return fail(h, CPS_ERR_INVALID, "%s: negative number of periods", who);
    FleetCore &c = F->core;
    bool reads = false;
    for (int j = 0; j < n_periods && !reads; ++j) reads = legacy_fleet_solves(F, c.period + j);
    int rc;
    if ((rc = fleet_core_check_draws(h, c, draws_dev, reads, who)) != CPS_OK) return rc;
    if ((rc = fleet_core_check_draws(h, c, act_draws_dev, n_periods > 0, who)) != CPS_OK) return rc;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t E = c.E, K = h->cfg.num_rollouts;
    LegacyFleetArgs a;
    memset(&a, 0, sizeof(a));
    a.ode = h->ode; a.mp = h->mp;
    if ((rc = cps_fold_cost_for(h, 1.0f, &a.cost)) != CPS_OK) return rc;   // the legacy cost has no target equilibrium
    a.plant = plant_params(h, c.dt_sim, c.n_sim);
    a.sampling = F->sampling; a.n_draws = F->n_draws; a.stdev = F->stdev; a.p_Q = F->p_Q;
    a.s = c.d_s; a.u = F->d_u; a.u_prev = F->d_up; a.Q = c.d_uprev;
    a.seed = c.seed; a.e_offset = c.e_offset;
    a.partials = F->d_partials; a.tickets = F->d_tickets; a.nonfinite = h->d_nonfinite;
    void (*fn)(const LegacyFleetArgs) =
        (h->cfg.integrator == CPS_EULER_V0) ? (c.philox ? legacy_fleet_kernel<0, true> : legacy_fleet_kernel<0, false>)
                                            : (c.philox ? legacy_fleet_kernel<1, true> : legacy_fleet_kernel<1, false>);
    if (F->smem > 48 * 1024) CUDA_TRY(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)F->smem));
    for (int j = 0; j < n_periods; ++j) {
        const FleetRow row = fleet_core_row(c, j, tp_dev, te_dev, record_dev);
        a.tp = row.tp; a.te = row.te; a.record = row.record; a.period = row.period; a.time = row.time;
        a.act = act_draws_dev ? act_draws_dev + (size_t)j * E : nullptr;
        if (legacy_fleet_solves(F, c.period)) {
            a.draws = draws_dev ? draws_dev + (size_t)j * E * K * F->n_draws : nullptr;
            a.S_out = S_out_dev ? S_out_dev + (size_t)j * E * K : nullptr;
            fn<<<dim3(h->grid, c.E), h->block, F->smem, h->stream>>>(a);
        } else {
            legacy_fleet_advance_kernel<<<(c.E + 127) / 128, 128, 0, h->stream>>>(a, c.E);
        }
        h->launches += 1;
        c.period += 1;
    }
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

// The raw draws [E][K][n_draws] of `period` (counter: rollout, LEGACY_DRAWS + group, period, experiment)
static FleetDrawsArgs legacy_fleet_draws_args(const cps_handle *h, const LegacyFleetState *F, long long period, float *out) {
    const FleetCore &c = F->core;
    const int K = h->cfg.num_rollouts;
    return {c.seed, LEGACY_DRAWS, 0u, (unsigned)period, c.e_offset, c.E, K, F->n_draws, 0, (long long)K * F->n_draws,
            F->n_draws, 1, out};
}

static int legacy_fleet_raw(cps_handle *h, const LegacyFleetState *F, long long period, float *out) {
    const FleetDrawsArgs d = legacy_fleet_draws_args(h, F, period, out);
    return F->sampling == CPS_LEGACY_SAMPLING_UNIFORM ? fleet_uniforms_launch(h, d, 1, -1.0f, 2.0f) : fleet_draws_launch(h, d, 1);
}

extern "C" int cps_legacy_fleet_draws(cps_handle *h, long long period, float *out_dev) {
    if (!h) return CPS_ERR_INVALID;
    LegacyFleetState *F = legacy_fleet(h, "cps_legacy_fleet_draws", true);
    if (!F) return CPS_ERR_NOT_CONFIGURED;
    if (!out_dev || period < 0) return fail(h, CPS_ERR_INVALID, "cps_legacy_fleet_draws: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    return legacy_fleet_raw(h, F, period, out_dev);
}

extern "C" int cps_legacy_fleet_act_draws(cps_handle *h, long long period, float *out_dev) {
    if (!h) return CPS_ERR_INVALID;
    LegacyFleetState *F = legacy_fleet(h, "cps_legacy_fleet_act_draws", true);
    if (!F) return CPS_ERR_NOT_CONFIGURED;
    if (!out_dev || period < 0) return fail(h, CPS_ERR_INVALID, "cps_legacy_fleet_act_draws: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const FleetCore &c = F->core;
    const FleetDrawsArgs d = {c.seed, LEGACY_ACT, 0u, (unsigned)period, c.e_offset, c.E, 1, 1, 0, 1, 1, 1, out_dev};
    return fleet_uniforms_launch(h, d, 1, -1.0f, 2.0f);
}

extern "C" int cps_legacy_fleet_perturbations(cps_handle *h, long long period, float *out_dev) {
    if (!h) return CPS_ERR_INVALID;
    const char *who = "cps_legacy_fleet_perturbations";
    LegacyFleetState *F = legacy_fleet(h, who, true);
    if (!F) return CPS_ERR_NOT_CONFIGURED;
    if (!out_dev || period < 0) return fail(h, CPS_ERR_INVALID, "%s: bad argument", who);
    if (!F->core.philox) return fail(h, CPS_ERR_INVALID, "%s: a fleet with supplied draws has no draws of its own", who);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const int K = h->cfg.num_rollouts, T = h->cfg.horizon, E = F->core.E;
    if (!F->d_raw) CUDA_TRY(h, cudaMalloc(&F->d_raw, sizeof(float) * (size_t)E * K * F->n_draws));
    int rc;
    if ((rc = legacy_fleet_raw(h, F, period, F->d_raw)) != CPS_OK) return rc;
    const long long n = (long long)E * K;
    legacy_fleet_perturb_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(F->d_raw, out_dev, E, K, T, F->n_draws,
                                                                                    F->sampling, F->stdev);
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

extern "C" long long cps_legacy_fleet_period(const cps_handle *h) { return (h && h->lfleet) ? h->lfleet->core.period : -1; }
