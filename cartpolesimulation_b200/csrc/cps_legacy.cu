// cps_legacy.cu -- the legacy front-end: controller_mppi_cartpole (SURVEY.md 8f, row f2).
//
// Control_Toolkit_ASF/Controllers/controller_mppi_cartpole.py is the repository's original MPPI controller (what
// README.md:46 calls "MPPI with predictor_ODE_v0").  It runs the same K x T rollouts as optimizer_mppi but keeps its own
// books: host-drawn perturbations of five sampling types, no clipping of u + delta_u, a SUMMED cost with two extra
// kinetic-energy terms and an input-violation penalty, a per-step control-change term against the previous nominal
// SEQUENCE, an unclipped update and a zero-fill shift at the END of the iteration.
//
// Kernels
//   legacy_mppi_kernel   one update iteration in one launch: rollouts (the shared control_step code, rotation mode),
//                        q() + phi() accumulated in the same pass, block partials over the T perturbation channels, the
//                        last block merges them (online softmax), applies u += sum(w du)/sum(w), emits u[0], copies
//                        u -> u_prev and shifts u with a zero appended.
//   legacy_advance_kernel  an iteration without a solve (iteration % update_every != 0).
// The same for E closed-loop experiments: cps_legacy_fleet.cu.
#include <cuda_runtime.h>

#include <cmath>
#include <cstring>

#include "cps_internal.cuh"

struct LegacyArgs {
    OdeParams ode;
    CostParams cost;
    MppiParams mp;
    const float *s;           // [6]
    const float *du;          // K x T perturbations
    long long ns_t, ns_k;     // element strides along horizon step / rollout
    float *u;                 // [T] nominal inputs, in/out (shifted on exit)
    float *u_prev;            // [T] previous nominal inputs, in/out
    float *u_out;             // [1]
    float *S_out;             // [K] or null
    float *traj_out;          // K x (T+1) x 6 or null
    long long ts_k, ts_t, ts_c;
    float *u_upd_out;         // [T] or null
    float *partials;
    unsigned *ticket;
    int *nonfinite;
};

#include "cps_legacy.cuh"

// smem: [T] u, [T] u_prev, [nwarps][T + 2] reduction scratch reused by the merge (+ [nwarps]).
template <int INTEG>
__global__ void __launch_bounds__(256, 4) legacy_mppi_kernel(const __grid_constant__ LegacyArgs a) {
    extern __shared__ float smem[];
    const MppiParams &mp = a.mp;
    const int T = mp.T;
    float *s_u = smem;
    float *s_up = s_u + T;
    float *s_red = s_up + T;
    const int tid = threadIdx.x;
    const int k = blockIdx.x * blockDim.x + tid;
    const bool active = k < mp.K;
    const int kc = min(k, mp.K - 1);

    for (int t = tid; t < T; t += blockDim.x) { s_u[t] = a.u[t]; s_up[t] = a.u_prev[t]; }
    __syncthreads();

    State z = load_state(a.s);
    const OdeParams ode = pin_params(a.ode, z.th);
    float c_cost = cosf(z.th);  // q() takes np.cos of the stored angle (:131-135)
    const float *nz = a.du + (long long)kc * a.ns_k;
    float *traj = a.traj_out ? a.traj_out + (long long)kc * a.ts_k : nullptr;

    float S = 0.0f;
    float du_next = nz[0];
#pragma unroll 1
    for (int t = 0; t < T; ++t) {
        const float du = du_next;
        if (t + 1 < T) du_next = nz[(long long)(t + 1) * a.ns_t];  // prefetch under the integration
        const float un = s_u[t];
        S += legacy_stage(a.cost, mp, c_cost, z.w, z.x, z.v, un, du, s_up[t]);
        if (active && traj) store_state(traj + (long long)t * a.ts_t, a.ts_c, z);
        control_step<INTEG, SC_ROTATE, false, false>(ode, z, un + du);  // the rollout sees the UNCLIPPED input (:190-192)
        c_cost = z.c;
    }
    S += terminal_cost<COST_DEFAULT>(a.cost, z.th, z.x);  // phi() (:271-298) is default.py's terminal cost
    if (active) {
        if (traj) store_state(traj + (long long)T * a.ts_t, a.ts_c, z);
        if (a.S_out) a.S_out[k] = S;
        if (!isfinite(S)) atomicAdd(a.nonfinite, 1);
    }

    if (!block_partials(mp, S, active, nz, a.ns_t, s_red, a.partials, a.ticket, blockIdx.x, gridDim.x)) return;
    merge_partials(mp, a.partials, gridDim.x, s_red);
    // update_inputs (:325-335): u += sum_k w_k du_k / sum_k w_k, no clipping
    const float invS = 1.0f / s_red[0];
    for (int t = tid; t < T; t += blockDim.x) s_u[t] = fmaf(s_red[1 + t], invS, s_u[t]);
    __syncthreads();
    // Q = u[0]; u_prev <- u; u <- [u[1:], 0]  (:521, :531-536)
    for (int t = tid; t < T; t += blockDim.x) {
        const float un = s_u[t];
        a.u_prev[t] = un;
        if (a.u_upd_out) a.u_upd_out[t] = un;
        a.u[t] = (t + 1 < T) ? s_u[t + 1] : 0.0f;
        if (t == 0) *a.u_out = un;
    }
    if (tid == 0) *a.ticket = 0u;
}

__global__ void __launch_bounds__(128) legacy_advance_kernel(float *u, float *u_prev, float *u_out, int T) {
    extern __shared__ float s_u[];
    for (int t = threadIdx.x; t < T; t += blockDim.x) s_u[t] = u[t];
    __syncthreads();
    for (int t = threadIdx.x; t < T; t += blockDim.x) {
        u_prev[t] = s_u[t];
        u[t] = (t + 1 < T) ? s_u[t + 1] : 0.0f;
        if (t == 0) *u_out = s_u[0];
    }
}

extern "C" int cps_legacy_step(cps_handle *h, const float *s_dev, const float *delta_u_dev, int layout, float *u_out_dev,
                               float *S_out_dev, float *traj_out_dev, int traj_layout, float *u_upd_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    int rc = legacy_check(h, "cps_legacy_step");
    if (rc != CPS_OK) return rc;
    if (!s_dev || !delta_u_dev || !u_out_dev) return fail(h, CPS_ERR_INVALID, "cps_legacy_step: null pointer");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const long long K = h->cfg.num_rollouts, T = h->cfg.horizon;
    LegacyArgs a;
    a.ode = h->ode; a.cost = h->cost; a.mp = h->mp;
    a.s = s_dev; a.du = delta_u_dev;
    if (layout == CPS_TIME_MAJOR) { a.ns_t = K; a.ns_k = 1; }
    else { a.ns_t = 1; a.ns_k = T; }
    a.u = h->d_unom; a.u_prev = h->d_uprev; a.u_out = u_out_dev; a.S_out = S_out_dev; a.traj_out = traj_out_dev;
    if (traj_layout == CPS_TIME_MAJOR) { a.ts_k = 1; a.ts_t = 6 * K; a.ts_c = K; }
    else { a.ts_k = (T + 1) * 6; a.ts_t = 6; a.ts_c = 1; }
    a.u_upd_out = u_upd_out_dev;
    a.partials = h->d_partials; a.ticket = h->d_ticket; a.nonfinite = h->d_nonfinite;
    const int nwarps = h->block / 32;
    const size_t smem = sizeof(float) * ((size_t)2 * T + (size_t)nwarps * (T + 2) + (size_t)T + 4 + nwarps);
    void (*fn)(const LegacyArgs) = (h->cfg.integrator == CPS_EULER_V0) ? legacy_mppi_kernel<0> : legacy_mppi_kernel<1>;
    if (smem > 48 * 1024) CUDA_TRY(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fn<<<h->grid, h->block, smem, h->stream>>>(a);
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

extern "C" int cps_legacy_step_host(cps_handle *h, const float *s_host, const float *delta_u_host, int layout,
                                    float *u_out_host) {
    if (!h) return CPS_ERR_INVALID;
    int rc = legacy_check(h, "cps_legacy_step_host");
    if (rc != CPS_OK) return rc;
    if (!s_host || !delta_u_host || !u_out_host) return fail(h, CPS_ERR_INVALID, "cps_legacy_step_host: null pointer");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t n_du = sizeof(float) * (size_t)h->cfg.num_rollouts * h->cfg.horizon;
    if (!h->d_ldu) CUDA_TRY(h, cudaMalloc(&h->d_ldu, n_du));
    // stream order: state, delta_u, the solve, u
    return solve_host(h, s_host, u_out_host, false, [&](const float *s_dev, float *u_dev) {
        CUDA_TRY(h, cudaMemcpyAsync(h->d_ldu, delta_u_host, n_du, cudaMemcpyHostToDevice, h->stream));
        return cps_legacy_step(h, s_dev, h->d_ldu, layout, u_dev, nullptr, nullptr, CPS_ROLLOUT_MAJOR, nullptr);
    });
}

// SAMPLING_TYPE "interpolated" (controller_mppi_cartpole.py:430-451) on the device: the reference draws the perturbation at
// every `step`-th horizon index and fills the rest with scipy's linear interp1d, i.e. (scipy 1.18, _call_linear) in float64
//   y = ((x - x_lo) / (x_hi - x_lo)) * y_hi + ((x_hi - x) / (x_hi - x_lo)) * y_lo
// -- two products and a sum, each rounded, no contraction -- assigned into a float32 array.  Restated with the same
// operations so that the perturbations are bit-identical to the host path (tested against the recorded delta_u).
__global__ void __launch_bounds__(256) legacy_interp_kernel(const float *__restrict__ knots, float *__restrict__ du, int K, int T,
                                                            int n_knots, int step) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)K * T) return;
    const int k = (int)(i / T), t = (int)(i % T);
    const int lo = t / step, j = t - lo * step;
    const float *kn = knots + (long long)k * n_knots;
    float y = kn[lo];
    if (j != 0) {
        const double w_hi = __ddiv_rn((double)j, (double)step), w_lo = __ddiv_rn((double)(step - j), (double)step);
        y = __double2float_rn(__dadd_rn(__dmul_rn(w_hi, (double)kn[lo + 1]), __dmul_rn(w_lo, (double)kn[lo])));
    }
    du[i] = y;
}

extern "C" int cps_legacy_step_host_knots(cps_handle *h, const float *s_host, const float *knots_host, int n_knots, int knot_step,
                                          float *u_out_host) {
    if (!h) return CPS_ERR_INVALID;
    int rc = legacy_check(h, "cps_legacy_step_host_knots");
    if (rc != CPS_OK) return rc;
    if (!s_host || !knots_host || !u_out_host) return fail(h, CPS_ERR_INVALID, "cps_legacy_step_host_knots: null pointer");
    const int K = h->cfg.num_rollouts, T = h->cfg.horizon;
    if (knot_step < 1 || n_knots < 1 || (long long)(n_knots - 1) * knot_step < T - 1)
        return fail(h, CPS_ERR_INVALID, "cps_legacy_step_host_knots: the knots do not cover the horizon");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t n_du = sizeof(float) * (size_t)K * T, n_kn = sizeof(float) * (size_t)K * n_knots;
    if (!h->d_ldu) CUDA_TRY(h, cudaMalloc(&h->d_ldu, n_du));
    if (h->n_lknots < n_kn) {
        if (h->d_lknots) cudaFree(h->d_lknots);
        h->d_lknots = nullptr; h->n_lknots = 0;
        CUDA_TRY(h, cudaMalloc(&h->d_lknots, n_kn));
        h->n_lknots = n_kn;
    }
    // stream order: state, knots, interpolation, the solve, u
    return solve_host(h, s_host, u_out_host, false, [&](const float *s_dev, float *u_dev) {
        CUDA_TRY(h, cudaMemcpyAsync(h->d_lknots, knots_host, n_kn, cudaMemcpyHostToDevice, h->stream));
        const long long n = (long long)K * T;
        legacy_interp_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(h->d_lknots, h->d_ldu, K, T, n_knots, knot_step);
        h->launches += 1;
        return cps_legacy_step(h, s_dev, h->d_ldu, CPS_ROLLOUT_MAJOR, u_dev, nullptr, nullptr, CPS_ROLLOUT_MAJOR, nullptr);
    });
}

extern "C" int cps_legacy_get_perturbations(cps_handle *h, float *delta_u_host) {
    if (!h) return CPS_ERR_INVALID;
    int rc = legacy_check(h, "cps_legacy_get_perturbations");
    if (rc != CPS_OK) return rc;
    if (!delta_u_host) return fail(h, CPS_ERR_INVALID, "cps_legacy_get_perturbations: null pointer");
    if (!h->d_ldu) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_legacy_get_perturbations: no host-form step has run yet");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaMemcpyAsync(delta_u_host, h->d_ldu, sizeof(float) * (size_t)h->cfg.num_rollouts * h->cfg.horizon,
                                cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}

extern "C" int cps_legacy_advance(cps_handle *h, float *u_out_host) {
    if (!h) return CPS_ERR_INVALID;
    int rc = legacy_check(h, "cps_legacy_advance");
    if (rc != CPS_OK) return rc;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const int T = h->cfg.horizon;
    legacy_advance_kernel<<<1, 128, sizeof(float) * (size_t)T, h->stream>>>(h->d_unom, h->d_uprev, h->d_u, T);
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return u_out_host ? return_u_host(h, h->d_u, u_out_host) : CPS_OK;
}

extern "C" int cps_legacy_reset(cps_handle *h) {
    if (!h) return CPS_ERR_INVALID;
    int rc = legacy_check(h, "cps_legacy_reset");
    if (rc != CPS_OK) return rc;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t n = sizeof(float) * (size_t)h->cfg.horizon;
    CUDA_TRY(h, cudaMemsetAsync(h->d_unom, 0, n, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(h->d_uprev, 0, n, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}

extern "C" int cps_legacy_get_inputs(cps_handle *h, float *u_host, float *u_prev_host) {
    if (!h) return CPS_ERR_INVALID;
    int rc = legacy_check(h, "cps_legacy_get_inputs");
    if (rc != CPS_OK) return rc;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t n = sizeof(float) * (size_t)h->cfg.horizon;
    if (u_host) CUDA_TRY(h, cudaMemcpyAsync(u_host, h->d_unom, n, cudaMemcpyDeviceToHost, h->stream));
    if (u_prev_host) CUDA_TRY(h, cudaMemcpyAsync(u_prev_host, h->d_uprev, n, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}

extern "C" int cps_legacy_set_inputs(cps_handle *h, const float *u_host, const float *u_prev_host) {
    if (!h) return CPS_ERR_INVALID;
    int rc = legacy_check(h, "cps_legacy_set_inputs");
    if (rc != CPS_OK) return rc;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t n = sizeof(float) * (size_t)h->cfg.horizon;
    if (u_host) CUDA_TRY(h, cudaMemcpyAsync(h->d_unom, u_host, n, cudaMemcpyHostToDevice, h->stream));
    if (u_prev_host) CUDA_TRY(h, cudaMemcpyAsync(h->d_uprev, u_prev_host, n, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}
