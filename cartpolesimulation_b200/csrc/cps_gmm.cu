// cps_gmm.cu -- CEM with a two-component Gaussian-mixture sampling distribution (SURVEY.md 8f row f3, third
// forward-only optimizer): Control_Toolkit/Optimizers/optimizer_cem_gmm_tf.py:58-140.
//
// One outer iteration of the reference (update_distribution, :58-96):
//   Q = clip(sampling_dist.sample([K]))           MixtureSameFamily over the [T, 1] batch: every (rollout, step) picks
//                                                 its component independently, Q = loc[t, c] + scale[t, c] * eps
//   traj_cost = predict_and_cost(s, Q)            -> plan_kernel (cps_plan_cost), unchanged
//   elite_Q = Q[argsort(traj_cost)[:best_k]]      stable: ties keep index order
//   every elite but the two cheapest joins the cheaper / second-cheapest elite, whichever is nearer in the Euclidean norm
//   over the horizon (ties: the cheapest); the two clusters give the new components: per-step mean and population
//   standard deviation clipped to [stdev_min, 1e4]; mixture weight of the first = its share of the elites.
// After the last iteration (:107-119): u = elite_Q[0, 0]; loc and scale are shifted by one step, the last entry repeated
// (unlike optimizer_cem_tf, which refills the tail with the initial values).
//
// Three launches per outer iteration, nothing returns to the host in between:
//   gmm_sample_kernel   Q[T][K] from the supplied draws (standard normals for both components, one uniform per element)
//   plan_kernel         rollouts + cost (cps_plan_cost; with the neural predictor its net_grad_kernel pass)
//   gmm_update_kernel   ONE block: radix select of the best_k cheapest plans (ties in index order), the two cheapest of
//                       them, the distances, the cluster statistics, and after the last iteration u and the shift.
// The distribution lives on the device: loc[2][T], scale[2][T], p1.
#include <cuda_runtime.h>

#include <cmath>
#include <cstring>
#include <new>

#include "cps_internal.cuh"
#include "cps_plant.cuh"

struct GmmState {
    int best_k;
    float sd_init, sd_min;
    float *d_dist;    // loc[2][T], scale[2][T], p1
    float *d_Q;       // [T][K] sampled plans
    float *d_J;       // [K]
    int *d_elite;     // [K]: elite indices (ascending), then their cluster flags at [best_k ..)
};

struct GmmArgs {
    const float *eps, *u01;
    long long es_c, es_t, es_k;   // strides of the normal draws along component / step / rollout
    long long us_t, us_k;
    float *dist;                  // loc[2][T], scale[2][T], p1
    float *Q;                     // [T][K]
    const float *J;
    int K, T, best_k, last_iter;
    float lo, hi, sd_min;
    int *elite;
    float *u_out;
    float *Q_out;                 // or null: the last iteration's plans in the caller's layout
    long long qo_k, qo_t;
};

namespace {

__device__ __forceinline__ unsigned order_key(float J) {   // cost -> unsigned key with the same order; NaN sorts last
    if (J != J) return 0xFFFFFFFFu;
    const unsigned b = __float_as_uint(J);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__global__ void __launch_bounds__(256) gmm_sample_kernel(const __grid_constant__ GmmArgs a) {
    const long long n = (long long)a.K * a.T;
    const float p1 = a.dist[4 * a.T];
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int t = (int)(i / a.K), k = (int)(i - (long long)t * a.K);
        const int c = (a.u01[(long long)t * a.us_t + (long long)k * a.us_k] < p1) ? 0 : 1;
        const float e = a.eps[(long long)c * a.es_c + (long long)t * a.es_t + (long long)k * a.es_k];
        const float q = gmm_plan_value(a.dist[c * a.T + t], a.dist[(2 + c) * a.T + t], e, a.lo, a.hi);
        a.Q[i] = q;
        if (a.Q_out) a.Q_out[(long long)k * a.qo_k + (long long)t * a.qo_t] = q;
    }
}

__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// One CEM-GMM selection and update by one block of 256 threads (gmm_update_kernel, gmm_update_fleet_kernel): J [K] the
// costs, elite [2 K] scratch (elite indices ascending, then their cluster flags), dist loc[2][T], scale[2][T], p1 <- the
// update, *u_out <- u after the last iteration.  The plans are read through q_elite(t, e, k) (step t of elite e, plan k)
// and q_best(t, j, b) (step t of the j-th cheapest plan, plan b); rows(b0, b1) runs once the two cheapest are known.
template <class Rows, class QElite, class QBest>
__device__ __forceinline__ void gmm_update_block(const float *J, int K, int T, int bk, int last_iter, float sd_min, int *elite,
                                                 float *dist, float *u_out, Rows rows, QElite q_elite, QBest q_best) {
    __shared__ unsigned s_hist[256];
    __shared__ unsigned s_prefix, s_remaining;
    __shared__ int s_scan[8], s_base_eq, s_base_el;
    __shared__ unsigned long long s_best[8];
    __shared__ int s_b0, s_b1, s_n1;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nt = blockDim.x, nwarps = nt >> 5;

    // ---- the best_k-th smallest key: 8-bit radix select, most significant digit first ---------------------------------
    if (tid == 0) { s_prefix = 0u; s_remaining = (unsigned)bk; }
    __syncthreads();
    for (int shift = 24; shift >= 0; shift -= 8) {
        for (int b = tid; b < 256; b += nt) s_hist[b] = 0u;
        __syncthreads();
        const unsigned prefix = s_prefix, mask = (shift == 24) ? 0u : ~((1u << (shift + 8)) - 1u);
        for (int i = tid; i < K; i += nt) {
            const unsigned key = order_key(__ldcg(J + i));
            if ((key & mask) == prefix) atomicAdd(&s_hist[(key >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (tid == 0) {
            unsigned rem = s_remaining, cum = 0u;
            for (int b = 0; b < 256; ++b) {
                if (cum + s_hist[b] >= rem) { s_prefix = prefix | ((unsigned)b << shift); s_remaining = rem - cum; break; }
                cum += s_hist[b];
            }
        }
        __syncthreads();
    }
    const unsigned kth = s_prefix;
    const int ties_wanted = (int)s_remaining;   // plans with key == kth that belong to the elites (lowest indices first)

    // ---- elite indices, ascending (ordered compaction over chunks of nt plans) -------------------------------------------
    if (tid == 0) { s_base_eq = 0; s_base_el = 0; }
    __syncthreads();
    for (int base = 0; base < K; base += nt) {
        const int i = base + tid;
        const unsigned key = (i < K) ? order_key(__ldcg(J + i)) : 0xFFFFFFFFu;
        const bool is_eq = i < K && key == kth;
        // rank of this plan among the equal keys seen so far
        unsigned bal = __ballot_sync(0xffffffffu, is_eq);
        int eq_before = __popc(bal & ((1u << lane) - 1u));
        if (lane == 0) s_scan[warp] = __popc(bal);
        __syncthreads();
        int eq_base = s_base_eq;
        for (int w = 0; w < warp; ++w) eq_base += s_scan[w];
        int eq_total = 0;
        for (int w = 0; w < nwarps; ++w) eq_total += s_scan[w];
        __syncthreads();
        const bool take = i < K && (key < kth || (is_eq && eq_base + eq_before < ties_wanted));
        bal = __ballot_sync(0xffffffffu, take);
        const int el_before = __popc(bal & ((1u << lane) - 1u));
        if (lane == 0) s_scan[warp] = __popc(bal);
        __syncthreads();
        int el_base = s_base_el;
        for (int w = 0; w < warp; ++w) el_base += s_scan[w];
        int el_total = 0;
        for (int w = 0; w < nwarps; ++w) el_total += s_scan[w];
        if (take) elite[el_base + el_before] = i;
        __syncthreads();
        if (tid == 0) { s_base_eq += eq_total; s_base_el += el_total; }
        __syncthreads();
    }

    // ---- the cheapest and second-cheapest elite: sorted_cost[0], sorted_cost[1] (ties: lower index) -----------------------
    for (int pass = 0; pass < 2; ++pass) {
        unsigned long long best = ~0ull;
        for (int e = tid; e < bk; e += nt) {
            const int k = elite[e];
            if (pass == 1 && k == s_b0) continue;
            const unsigned long long c = ((unsigned long long)order_key(__ldcg(J + k)) << 32) | (unsigned)k;
            best = c < best ? c : best;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long n = __shfl_xor_sync(0xffffffffu, best, o);
            best = n < best ? n : best;
        }
        if (lane == 0) s_best[warp] = best;
        __syncthreads();
        if (tid == 0) {
            for (int w = 1; w < nwarps; ++w) best = s_best[w] < best ? s_best[w] : best;
            if (pass == 0) s_b0 = (int)(best & 0xFFFFFFFFull); else s_b1 = (int)(best & 0xFFFFFFFFull);
        }
        __syncthreads();
    }
    const int b0 = s_b0, b1 = s_b1;
    rows(b0, b1);

    // ---- cluster of every elite: nearer of the two in the Euclidean norm over the horizon (:72-77), one warp per elite ----
    int *flag = elite + bk;   // 0: first cluster, 1: second
    if (tid == 0) s_n1 = 0;
    __syncthreads();
    int n1_local = 0;
    for (int e = warp; e < bk; e += nwarps) {
        const int k = elite[e];
        int f;
        if (k == b0) f = 0;
        else if (k == b1) f = 1;
        else {
            float d0 = 0.0f, d1 = 0.0f;
            for (int t = lane; t < T; t += 32) {
                const float q = q_elite(t, e, k);
                const float x0 = q - q_best(t, 0, b0), x1 = q - q_best(t, 1, b1);
                d0 = fmaf(x0, x0, d0);
                d1 = fmaf(x1, x1, d1);
            }
            d0 = sqrtf(warp_sum_f(d0));
            d1 = sqrtf(warp_sum_f(d1));
            f = (d1 < d0) ? 1 : 0;   // tf.argmin: the first of equal distances
        }
        if (lane == 0) { flag[e] = f; n1_local += (f == 0) ? 1 : 0; }
    }
    if (lane == 0 && n1_local) atomicAdd(&s_n1, n1_local);
    __syncthreads();
    const int n1 = s_n1, n2 = bk - n1;

    // ---- per step: mean and population standard deviation of both clusters (:84-93), one warp per step -------------------
    for (int t = warp; t < T; t += nwarps) {
        float s0 = 0.0f, s1 = 0.0f;
        for (int e = lane; e < bk; e += 32) {
            const float q = q_elite(t, e, elite[e]);
            if (flag[e] == 0) s0 += q; else s1 += q;
        }
        const float m0 = __fdiv_rn(warp_sum_f(s0), (float)n1), m1 = __fdiv_rn(warp_sum_f(s1), (float)n2);
        float v0 = 0.0f, v1 = 0.0f;
        for (int e = lane; e < bk; e += 32) {
            const float q = q_elite(t, e, elite[e]);
            if (flag[e] == 0) { const float d = q - m0; v0 = fmaf(d, d, v0); }
            else { const float d = q - m1; v1 = fmaf(d, d, v1); }
        }
        v0 = sqrtf(__fdiv_rn(warp_sum_f(v0), (float)n1));
        v1 = sqrtf(__fdiv_rn(warp_sum_f(v1), (float)n2));
        if (lane == 0) {
            // written one step earlier after the last iteration: the shift of :111-118
            const int dst = last_iter ? t - 1 : t;
            const float sd0 = fminf(fmaxf(v0, sd_min), 1.0e4f), sd1 = fminf(fmaxf(v1, sd_min), 1.0e4f);
            if (dst >= 0) {
                dist[dst] = m0; dist[T + dst] = m1; dist[2 * T + dst] = sd0; dist[3 * T + dst] = sd1;
            }
            if (last_iter && t == T - 1) {   // the last entry is repeated
                dist[t] = m0; dist[T + t] = m1; dist[2 * T + t] = sd0; dist[3 * T + t] = sd1;
            }
        }
    }
    if (tid == 0) {
        dist[4 * T] = __fdiv_rn((float)n1, (float)bk);   // prob_Q_1 (:79-80)
        if (last_iter) *u_out = q_best(0, 0, b0);        // elite_Q[0, 0, :] (:108): step 0 of the cheapest plan
    }
}

// One block of 256 threads: the sampled plans are a.Q [T][K].
__global__ void __launch_bounds__(256) gmm_update_kernel(const __grid_constant__ GmmArgs a) {
    auto q = [&a](int t, int, int k) { return a.Q[(long long)t * a.K + k]; };
    gmm_update_block(a.J, a.K, a.T, a.best_k, a.last_iter, a.sd_min, a.elite, a.dist, a.u_out, [](int, int) {}, q, q);
}

// CEM-GMM fleets: block x runs gmm_update_block on experiment x.  The elites' plans are rebuilt into a.rows [best_k][T]
// from the mixture they were sampled from and their draws (supplied, or regenerated from Philox as the rollouts drew them).
template <bool PHILOX>
__global__ void __launch_bounds__(256) gmm_update_fleet_kernel(const __grid_constant__ GmmFleetUpdate a) {
    __shared__ int s_pos[2];   // positions of the two cheapest plans in the elite list
    const long long x = blockIdx.x;
    const int K = a.K, T = a.T, bk = a.best_k, G4 = (T + 3) / 4;
    const float *d = a.dist + x * (4 * T + 1);
    float *W = a.rows + x * bk * T;
    int *elite = a.elite + x * 2 * K;
    auto rows = [&](int b0, int b1) {
        const float p1 = d[4 * T];
        for (int i = threadIdx.x; i < bk * G4; i += blockDim.x) {
            const int pos = i / G4, g = i - pos * G4, k = elite[pos], n = min(4, T - 4 * g);
            float e0[4], e1[4], u[4];
            if (PHILOX) {
                const unsigned eg = a.e_offset + (unsigned)x;
                philox_normals(a.seed, (unsigned)k, a.w1 + (unsigned)g, a.period, eg, n, e0, 1);
                philox_normals(a.seed, (unsigned)k, a.w1 + (unsigned)(G4 + g), a.period, eg, n, e1, 1);
                philox_uniforms(a.seed, (unsigned)k, a.w1 + (unsigned)(2 * G4 + g), a.period, eg, n, u, 1, 0.0f, 1.0f);
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const long long t = min(4 * g + q, T - 1);
                    e0[q] = a.eps[(x * 2 * T + t) * K + k];
                    e1[q] = a.eps[(x * 2 * T + T + t) * K + k];
                    u[q] = a.u01[(x * T + t) * K + k];
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int t = 4 * g + q, c = (u[q] < p1) ? 0 : 1;
                if (q < n) W[pos * T + t] = gmm_plan_value(d[c * T + t], d[(2 + c) * T + t], c ? e1[q] : e0[q], a.lo, a.hi);
            }
            if (g == 0 && k == b0) s_pos[0] = pos;
            if (g == 0 && k == b1) s_pos[1] = pos;
        }
        __syncthreads();
    };
    gmm_update_block(a.J + x * K, K, T, bk, a.last_iter, a.sd_min, elite, a.dist_out + x * (4 * T + 1), a.u + x, rows,
                     [&](int t, int e, int) { return W[e * T + t]; },
                     [&](int t, int j, int) { return W[s_pos[j] * T + t]; });
}

}  // namespace

int cps_gmm_fleet_update(cps_handle *h, const GmmFleetUpdate &a) {
    if (a.eps) gmm_update_fleet_kernel<false><<<a.E, 256, 0, h->stream>>>(a);
    else gmm_update_fleet_kernel<true><<<a.E, 256, 0, h->stream>>>(a);
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

void cps_gmm_free(cps_handle *h) {
    GmmState *G = h->gmm;
    if (!G) return;
    cudaFree(G->d_dist); cudaFree(G->d_Q); cudaFree(G->d_J); cudaFree(G->d_elite);
    delete G;
    h->gmm = nullptr;
}

extern "C" int cps_cem_gmm_reset(cps_handle *h) {
    if (!h) return CPS_ERR_INVALID;
    GmmState *G = h->gmm;
    if (!G) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_cem_gmm_reset: cps_cem_gmm_configure first");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const int T = h->cfg.horizon;
    float *tmp = new (std::nothrow) float[4 * (size_t)T + 1];
    if (!tmp) return fail(h, CPS_ERR_INVALID, "cps_cem_gmm_reset: out of host memory");
    const float mid = (h->mppi_in[5] + h->mppi_in[6]) * 0.5f;   // optimizer_reset (cem_gmm_tf.py:133-139)
    for (int t = 0; t < 2 * T; ++t) { tmp[t] = mid; tmp[2 * T + t] = G->sd_init; }
    tmp[4 * T] = 0.5f;
    cudaError_t e = cudaMemcpyAsync(G->d_dist, tmp, sizeof(float) * (4 * (size_t)T + 1), cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    delete[] tmp;
    CUDA_TRY(h, e);
    return CPS_OK;
}

extern "C" int cps_cem_gmm_configure(cps_handle *h, int best_k, float initial_stdev, float stdev_min) {
    if (!h) return CPS_ERR_INVALID;
    const int rc = cps_plan_check(h, "cps_cem_gmm_configure");   // every solve runs cps_plan_cost (ODE or network)
    if (rc != CPS_OK) return rc;
    if (best_k < 2 || best_k > h->cfg.num_rollouts)   // the two cheapest elites seed the two clusters
        return fail(h, CPS_ERR_INVALID, "cps_cem_gmm_configure: cem_best_k must lie in [2, num_rollouts]");
    if (!(initial_stdev >= 0.0f) || !(stdev_min >= 0.0f)) return fail(h, CPS_ERR_INVALID, "cps_cem_gmm_configure: negative stdev");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    cps_gmm_free(h);
    GmmState *G = new (std::nothrow) GmmState();
    if (!G) return fail(h, CPS_ERR_INVALID, "cps_cem_gmm_configure: out of host memory");
    memset(G, 0, sizeof(*G));
    const size_t K = h->cfg.num_rollouts, T = h->cfg.horizon;
    cudaError_t e = cudaMalloc(&G->d_dist, sizeof(float) * (4 * T + 1));
    if (e == cudaSuccess) e = cudaMalloc(&G->d_Q, sizeof(float) * K * T);
    if (e == cudaSuccess) e = cudaMalloc(&G->d_J, sizeof(float) * K);
    if (e == cudaSuccess) e = cudaMalloc(&G->d_elite, sizeof(int) * 2 * K);
    if (e != cudaSuccess) {
        cudaFree(G->d_dist); cudaFree(G->d_Q); cudaFree(G->d_J); cudaFree(G->d_elite);
        delete G;
        return fail(h, CPS_ERR_CUDA, "cps_cem_gmm_configure: allocating the scratch: %s", cudaGetErrorString(e));
    }
    G->best_k = best_k; G->sd_init = initial_stdev; G->sd_min = stdev_min;
    h->gmm = G;
    return cps_cem_gmm_reset(h);
}

extern "C" int cps_cem_gmm_step(cps_handle *h, const float *s_dev, const float *eps_dev, const float *u01_dev, int layout,
                                int n_iterations, float u_prev, float *u_out_dev, float *Q_out_dev, float *J_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    GmmState *G = h->gmm;
    if (!G) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_cem_gmm_step: cps_cem_gmm_configure first");
    if (!s_dev || !eps_dev || !u01_dev || !u_out_dev) return fail(h, CPS_ERR_INVALID, "cps_cem_gmm_step: null pointer");
    if (n_iterations < 1) return fail(h, CPS_ERR_INVALID, "cps_cem_gmm_step: n_iterations < 1");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const int K = h->cfg.num_rollouts, T = h->cfg.horizon;
    GmmArgs a;
    memset(&a, 0, sizeof(a));
    if (layout == CPS_TIME_MAJOR) { a.es_c = (long long)T * K; a.es_t = K; a.es_k = 1; a.us_t = K; a.us_k = 1; a.qo_k = 1; a.qo_t = K; }
    else { a.es_c = 1; a.es_t = 2; a.es_k = 2LL * T; a.us_t = 1; a.us_k = T; a.qo_k = T; a.qo_t = 1; }
    a.dist = G->d_dist; a.Q = G->d_Q; a.J = J_out_dev ? J_out_dev : G->d_J;
    a.K = K; a.T = T; a.best_k = G->best_k;
    a.lo = h->mppi_in[5]; a.hi = h->mppi_in[6]; a.sd_min = G->sd_min;
    a.elite = G->d_elite; a.u_out = u_out_dev;
    const long long n = (long long)K * T;
    const int sgrid = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
    for (int it = 0; it < n_iterations; ++it) {
        a.eps = eps_dev + (size_t)it * 2 * K * T;
        a.u01 = u01_dev + (size_t)it * K * T;
        a.last_iter = (it == n_iterations - 1) ? 1 : 0;
        a.Q_out = a.last_iter ? Q_out_dev : nullptr;   // Q_logged is the last iteration's plans (:105)
        gmm_sample_kernel<<<sgrid, 256, 0, h->stream>>>(a);
        h->launches += 1;
        int rc = cps_plan_cost(h, s_dev, G->d_Q, CPS_TIME_MAJOR, K, T, u_prev, const_cast<float *>(a.J), nullptr, 0);
        if (rc != CPS_OK) return rc;
        gmm_update_kernel<<<1, 256, 0, h->stream>>>(a);
        h->launches += 1;
    }
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

extern "C" int cps_cem_gmm_step_host(cps_handle *h, const float *s_host, const float *eps_dev, const float *u01_dev, int layout,
                                     int n_iterations, float u_prev, float *u_out_host) {
    if (!h) return CPS_ERR_INVALID;
    if (!s_host || !u_out_host) return fail(h, CPS_ERR_INVALID, "cps_cem_gmm_step_host: null pointer");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    // ODE: the state travels in plan_kernel's parameter block; the network kernel reads it from device memory
    return solve_host(h, s_host, u_out_host, h->cfg.integrator != CPS_PREDICTOR_NEURAL, [&](const float *s_dev, float *u_dev) {
        return cps_cem_gmm_step(h, s_dev, eps_dev, u01_dev, layout, n_iterations, u_prev, u_dev, nullptr, nullptr);
    });
}

extern "C" int cps_cem_gmm_get_distribution(cps_handle *h, float *loc_host, float *scale_host, float *p1_host) {
    if (!h) return CPS_ERR_INVALID;
    GmmState *G = h->gmm;
    if (!G) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_cem_gmm_get_distribution: cps_cem_gmm_configure first");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t T = h->cfg.horizon;
    if (loc_host) CUDA_TRY(h, cudaMemcpyAsync(loc_host, G->d_dist, sizeof(float) * 2 * T, cudaMemcpyDeviceToHost, h->stream));
    if (scale_host) CUDA_TRY(h, cudaMemcpyAsync(scale_host, G->d_dist + 2 * T, sizeof(float) * 2 * T, cudaMemcpyDeviceToHost, h->stream));
    if (p1_host) CUDA_TRY(h, cudaMemcpyAsync(p1_host, G->d_dist + 4 * T, sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}

extern "C" int cps_cem_gmm_set_distribution(cps_handle *h, const float *loc_host, const float *scale_host, const float *p1_host) {
    if (!h) return CPS_ERR_INVALID;
    GmmState *G = h->gmm;
    if (!G) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_cem_gmm_set_distribution: cps_cem_gmm_configure first");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t T = h->cfg.horizon;
    if (loc_host) CUDA_TRY(h, cudaMemcpyAsync(G->d_dist, loc_host, sizeof(float) * 2 * T, cudaMemcpyHostToDevice, h->stream));
    if (scale_host) CUDA_TRY(h, cudaMemcpyAsync(G->d_dist + 2 * T, scale_host, sizeof(float) * 2 * T, cudaMemcpyHostToDevice, h->stream));
    if (p1_host) CUDA_TRY(h, cudaMemcpyAsync(G->d_dist + 4 * T, p1_host, sizeof(float), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}
