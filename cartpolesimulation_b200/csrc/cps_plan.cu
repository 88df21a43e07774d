// cps_plan.cu -- the forward-only optimizers' predict_and_cost and their selection step (SURVEY.md 8f row f3).
//
// optimizer_random_action_tf and optimizer_cem_tf (Control_Toolkit/Optimizers/optimizer_random_action_tf.py:42-49,
// optimizer_cem_tf.py:57-83) evaluate K candidate input plans Q[K][T] from one state:
//     rollout_trajectory = predictor.predict_core(s, Q);  traj_cost = cost_function.get_trajectory_cost(traj, Q, u)
// and then pick from the sorted costs: the best plan's first input (random action), or the cem_best_k elites whose
// per-step mean / standard deviation become the next sampling distribution (CEM).  In the reference these are three
// framework ops with the [K][T+1][6] trajectory tensor in between; here it is ONE launch per evaluation:
//   every thread integrates one plan (the same control_step / stage_cost device code as mppi_kernel) and keeps the
//   cost in a register; the block that finishes last (atomic ticket) selects on the K costs -- arg-min, or a radix
//   select of the best_k-th smallest cost with ties taken in index order -- and finishes the optimizer's update
//   (elite mean / population std per horizon step, and after the last CEM iteration the std clip, the shift of both
//   vectors and u = elite_Q[0, 0]).  CEM plans are built in the kernel from supplied standard-normal draws,
//   Q = clip(mu + eps * std) with separately rounded multiply and add (tf.multiply, then +), so they are bit-equal to
//   the reference's; nothing returns to the host between the outer iterations of one solve.
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>
#include <cstring>
#include <new>

#include "cps_internal.cuh"
#include "cps_plant.cuh"

enum { PLAN_Q = 0, PLAN_CEM = 1 };
enum { SELECT_NONE = 0, SELECT_ARGMIN = 1, SELECT_CEM = 2 };

struct PlanArgs {
    OdeParams ode;
    CostParams cost;
    const float *s;               // [6]
    float s_inline[6];            // *_host entry points: the state travels in the parameter block
    int use_inline;
    const float *Q;               // PLAN_Q: plans; PLAN_CEM: standard-normal draws
    long long qs_k, qs_t;         // element strides along plan / horizon step
    const float *mu, *sd;         // PLAN_CEM: sampling distribution [T]
    float lo, hi, inv_T1, u_prev;
    int K, T;
    int rs_off;                   // float offset (even) of the row-sum slots in dynamic shared memory (MAX_COST plugins)
    float *J;                     // [K]; required when select != SELECT_NONE
    float *Q_out;                 // PLAN_CEM: the sampled plans, same strides as Q, or null
    float *traj_out;
    long long ts_k, ts_t, ts_c;
    int select;
    int best_k, last_iter;
    float sd_min, sd_init, mid;
    unsigned *ticket;
    int *elite;                   // [K] scratch: indices of the elites, ascending (when they do not fit in shared memory)
    int elite_smem;               // capacity of the shared-memory elite list
    int defer_stats;              // CEM: stop after the elite list; cem_update_kernel computes the statistics
    // multi-block selection (cem_select_kernel, K > CPS_CEM_MULTIBLOCK_MIN): grid-wide scratch, zero between launches
    unsigned long long *g_best;   // [1] min over (key << 32 | index)
    unsigned *g_kmax;             // [1]
    unsigned *g_hist;             // [4][256]
    int *g_cnt;                   // [2][grid] per-block counts: keys below the threshold / equal to it
    float *mu_out, *sd_out;       // CEM: updated distribution [T]
    float *u_out;                 // [1]
    int *best_out;                // [1] or null: index of the cheapest plan
    int *nonfinite;
};

// CEM fleets (cps_cem_fleet.cu): the inputs of E experiments, read by plan_fleet_kernel / cem_update_fleet_kernel besides
// PlanArgs.  There PlanArgs' pointers are the fleet's bases and block (., e) offsets them to experiment e: J and elite
// [E][K], mu / sd / mu_out / sd_out [E][T], Q (supplied draws) and Q_out [E][T][K] (qs_k = 1, qs_t = K), u_out [E], ticket [E].
struct PlanFleetExt {
    const float *s;               // [E][8] states
    const float *tp, *te;         // [E] targets of this period (null: 0 / +1)
    CostParams cost_up, cost_dn;  // folded for target_equilibrium = +1 / -1
    unsigned long long seed;      // Philox draws: counter (plan, w1 + group, period, e_offset + e)
    unsigned w1, period, e_offset;
};

struct PlanState {
    int best_k;
    float sd_init, sd_min;
    float *d_J, *d_mu, *d_sd;     // d_mu / d_sd: two buffers of T floats each; `cur` is the live one
    int cur;
    int *d_elite, *d_best;
    unsigned *d_ticket;
    unsigned long long *d_gbest;
    unsigned *d_gkmax, *d_ghist;
    int *d_gcnt;
    int configured_cem;
};

// cost -> unsigned key with the same order; NaN sorts last
__device__ __forceinline__ unsigned order_key(float J) {
    if (J != J) return 0xFFFFFFFFu;
    const unsigned b = __float_as_uint(J);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__device__ __forceinline__ float cem_plan_value(float mu, float eps, float sd, float lo, float hi) {
    return clampf(__fadd_rn(mu, __fmul_rn(eps, sd)), lo, hi);  // tile(mu) + multiply(normal, stdev), then clip (:66-68)
}

// Costs 4g .. 4g+3 of the selecting block's pass over J: one 16-byte L2 load when the buffer is 16-byte aligned and K a
// multiple of 4 (vec), else four clamped 4-byte loads.  g must be a valid group (4g < K).
__device__ __forceinline__ float4 load_costs4(const float *J, int g, int K, bool vec) {
    if (vec) return __ldcg(reinterpret_cast<const float4 *>(J) + g);
    float4 v;
    v.x = __ldcg(J + min(4 * g, K - 1)); v.y = __ldcg(J + min(4 * g + 1, K - 1));
    v.z = __ldcg(J + min(4 * g + 2, K - 1)); v.w = __ldcg(J + min(4 * g + 3, K - 1));
    return v;
}

// Exclusive prefix of v over the block (thread order) and the block total.  s_w: [nwarps] shared scratch.
__device__ __forceinline__ int block_excl_scan(int v, int *s_w, int &total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += n;
    }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    int base = 0;
    total = 0;
    for (int w = 0; w < nwarps; ++w) {
        const int c = s_w[w];
        if (w < warp) base += c;
        total += c;
    }
    __syncthreads();
    return base + incl - v;
}

// Run by the block that finished last.  s_mu / s_sd: the distribution the plans were sampled from (PLAN_CEM);
// s_mu2 / s_sd2: [T] scratch for the updated one.
template <int MODE>
__device__ __forceinline__ void plan_select(const PlanArgs &a, const float *s_mu, const float *s_sd, float *s_mu2,
                                            float *s_sd2, int *s_elite) {
    __shared__ unsigned s_hist[256];
    __shared__ unsigned s_prefix, s_remaining;
    __shared__ int s_w[8];
    __shared__ unsigned long long s_bestw[8];
    __shared__ unsigned s_maxw[8];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nt = blockDim.x, nwarps = nt >> 5;
    const int K = a.K, T = a.T;

    // ---- cheapest plan, lowest index among equal costs (sorted_cost[0]); the largest key bounds the radix select ----------
    const bool vec = ((reinterpret_cast<unsigned long long>(a.J) & 15ull) == 0ull) && (K % 4 == 0);
    const int G = (K + 3) / 4;   // groups of four consecutive costs
    unsigned long long best = ~0ull;
    unsigned kmax = 0u;
#pragma unroll 4
    for (int g = tid; g < G; g += nt) {
        const float4 v = load_costs4(a.J, g, K, vec);
        const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int i = 4 * g + e;
            if (i < K) {
                const unsigned key = order_key(vv[e]);
                const unsigned long long c = ((unsigned long long)key << 32) | (unsigned)i;
                best = c < best ? c : best;
                kmax = max(kmax, key);
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long n = __shfl_xor_sync(0xffffffffu, best, o);
        best = n < best ? n : best;
        kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, o));
    }
    if (lane == 0) { s_bestw[warp] = best; s_maxw[warp] = kmax; }
    __syncthreads();
    for (int w = 0; w < nwarps; ++w) {
        best = s_bestw[w] < best ? s_bestw[w] : best;
        kmax = max(kmax, s_maxw[w]);
    }
    const int best_idx = (int)(best & 0xFFFFFFFFull);
    if (tid == 0 && a.best_out) *a.best_out = best_idx;
    if (a.select == SELECT_ARGMIN) {
        if (tid == 0) *a.u_out = a.Q[(long long)best_idx * a.qs_k];  // Q[best_idx, 0, :] (random_action_tf.py:69)
        return;
    }

    // ---- CEM: the best_k-th smallest key by an 8-bit radix select over the bits in which the keys differ -------------------
    // All keys lie in [kmin, kmax] and share the bits above the highest bit of kmin ^ kmax; starting below them spreads
    // the first digit over the bins (the costs of one solve share sign, exponent and often leading mantissa bits, which
    // would otherwise send every plan to one bin: tens of thousands of serialised same-address atomics).
    const int bk = min(a.best_k, K);
    const unsigned kmin = (unsigned)(best >> 32);
    int hi = 32 - __clz((int)(kmin ^ kmax));   // number of low bits that vary (0: all costs equal)
    if (tid == 0) { s_prefix = (hi >= 32) ? 0u : (kmin & ~((1u << hi) - 1u)); s_remaining = (unsigned)bk; }
    __syncthreads();
    while (hi > 0) {
        const int w = min(8, hi), shift = hi - w;
        const unsigned mask = (hi >= 32) ? 0u : ~((1u << hi) - 1u), digit = (1u << w) - 1u;
        for (int b = tid; b < 256; b += nt) s_hist[b] = 0u;
        __syncthreads();
        const unsigned prefix = s_prefix;
        for (int base = 0; base < G; base += nt * 8) {   // 8 independent 16-byte loads in flight per thread, then the atomics
            float4 v[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) v[q] = load_costs4(a.J, min(base + q * nt + tid, G - 1), K, vec);   // unconditional: the loads batch
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int g = base + q * nt + tid;
                const float vv[4] = {v[q].x, v[q].y, v[q].z, v[q].w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const unsigned key = order_key(vv[e]);
                    const bool in = g < G && 4 * g + e < K && (key & mask) == prefix;
                    const unsigned bin = (key >> shift) & digit;
                    // a few outliers stretch [kmin, kmax] and put the bulk into one bin again: when the whole warp agrees
                    // (one MATCH.ALL), lane 0 adds 32; otherwise every lane adds for itself
                    int uniform;
                    __match_all_sync(0xffffffffu, in ? bin : 0xFFFFFFFFu, &uniform);
                    if (uniform) {
                        if (lane == 0 && in) atomicAdd(&s_hist[bin], 32u);
                    } else if (in) {
                        atomicAdd(&s_hist[bin], 1u);
                    }
                }
            }
        }
        __syncthreads();
        if (warp == 0) {   // the bin that holds rank `rem`: each lane owns 8 consecutive bins, shuffle scan over the lanes
            const unsigned rem = s_remaining;
            unsigned c[8], mine = 0u;
#pragma unroll
            for (int j = 0; j < 8; ++j) { c[j] = s_hist[lane * 8 + j]; mine += c[j]; }
            unsigned incl = mine;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned n = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += n;
            }
            const unsigned before = incl - mine;
            const unsigned hit = __ballot_sync(0xffffffffu, incl >= rem);   // non-empty: the total is >= rem
            if (lane == __ffs(hit) - 1) {
                unsigned cum = before;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (cum + c[j] >= rem) { s_prefix = prefix | ((unsigned)(lane * 8 + j) << shift); s_remaining = rem - cum; break; }
                    cum += c[j];
                }
            }
        }
        hi = shift;
        __syncthreads();
    }
    const unsigned kth = s_prefix;
    const int ties_wanted = (int)s_remaining;  // how many plans with key == kth belong to the elites (lowest indices)

    // ---- elite indices in ascending order (ordered compaction); the list lives in shared memory when it fits ----------------
    int *elite = (bk <= a.elite_smem) ? s_elite : a.elite;
    int n_eq_before = 0, n_el_before = 0;
    for (int base = 0; base < K; base += nt * 8) {   // each thread owns 8 consecutive plans of the chunk
        const int i0 = base + tid * 8;
        unsigned key[8];
        int eq = 0;
        const float4 va = load_costs4(a.J, min(i0 / 4, G - 1), K, vec), vb = load_costs4(a.J, min(i0 / 4 + 1, G - 1), K, vec);
        const float v[8] = {va.x, va.y, va.z, va.w, vb.x, vb.y, vb.z, vb.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            key[j] = order_key(v[j]);
            eq += (i0 + j < K && key[j] == kth) ? 1 : 0;
        }
        int tot_eq, tot_el;
        int eq_rank = n_eq_before + block_excl_scan(eq, s_w, tot_eq);
        unsigned take = 0u;
        int el = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const bool in = i0 + j < K;
            const bool is_eq = in && key[j] == kth;
            if (in && (key[j] < kth || (is_eq && eq_rank < ties_wanted))) { take |= 1u << j; ++el; }
            eq_rank += is_eq ? 1 : 0;
        }
        int pos = n_el_before + block_excl_scan(el, s_w, tot_el);
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (take & (1u << j)) elite[pos++] = i0 + j;
        n_eq_before += tot_eq;
        n_el_before += tot_el;
    }
    __syncthreads();
    if (a.defer_stats) {
        if (a.last_iter && tid == 0) *a.u_out = cem_plan_value(s_mu[0], a.Q[(long long)best_idx * a.qs_k], s_sd[0], a.lo, a.hi);
        return;
    }

    // ---- per horizon step: mean and population standard deviation over the elites (cem_tf.py:79-81) ------------------------
    for (int t = warp; t < T; t += nwarps) {
        float sum = 0.0f;
        for (int e = lane; e < bk; e += 32) {
            const int k = elite[e];
            sum += cem_plan_value(s_mu[t], a.Q[(long long)k * a.qs_k + (long long)t * a.qs_t], s_sd[t], a.lo, a.hi);
        }
        const float mean = __fdiv_rn(warp_sum(sum), (float)bk);
        float ss = 0.0f;
        for (int e = lane; e < bk; e += 32) {
            const int k = elite[e];
            const float d = cem_plan_value(s_mu[t], a.Q[(long long)k * a.qs_k + (long long)t * a.qs_t], s_sd[t], a.lo, a.hi) - mean;
            ss = fmaf(d, d, ss);
        }
        const float var = __fdiv_rn(warp_sum(ss), (float)bk);
        if (lane == 0) { s_mu2[t] = mean; s_sd2[t] = sqrtf(var); }
    }
    __syncthreads();
    if (!a.last_iter) {
        for (int t = tid; t < T; t += nt) { a.mu_out[t] = s_mu2[t]; a.sd_out[t] = s_sd2[t]; }
        return;
    }
    // after the last outer iteration: clip the std from below, shift both vectors by one step and refill the tail
    // (cem_tf.py:96-99); u = elite_Q[0, 0] is the cheapest plan's first input
    for (int t = tid; t < T; t += nt) {
        if (t + 1 < T) {
            a.mu_out[t] = s_mu2[t + 1];
            a.sd_out[t] = clampf(s_sd2[t + 1], a.sd_min, 1.0e8f);
        } else {
            a.mu_out[t] = a.mid;
            a.sd_out[t] = a.sd_init;
        }
    }
    if (tid == 0) *a.u_out = cem_plan_value(s_mu[0], a.Q[(long long)best_idx * a.qs_k], s_sd[0], a.lo, a.hi);
}

// Selection over many plans (K > CPS_CEM_MULTIBLOCK_MIN) by the whole grid: one block per SM, launched cooperatively, each
// owning a contiguous slice of the costs; grid-wide steps are separated by grid.sync().  Same result as plan_select
// (cheapest plan with the lowest index; the best_k smallest costs with ties in index order; elite list ascending); the
// statistics follow in cem_update_kernel.  A single block needs ~125 us for 65 536 costs (instruction latency, 2 warps
// per scheduler); spread over 148 SMs every step is a few hundred keys per block.
#define CPS_CEM_MULTIBLOCK_MIN 8192
__global__ void __launch_bounds__(256) cem_select_kernel(const __grid_constant__ PlanArgs a) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ unsigned s_hist[256];
    __shared__ unsigned s_prefix, s_remaining;
    __shared__ int s_w[8];
    __shared__ unsigned long long s_bestw[8];
    __shared__ unsigned s_maxw[8];
    __shared__ int s_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nt = blockDim.x, nwarps = nt >> 5;
    const int K = a.K, G = gridDim.x, b = blockIdx.x;
    const int per = ((K + G - 1) / G + 7) & ~7;            // slice length, a multiple of 8
    const int lo = min(b * per, K), hi = min(lo + per, K);  // this block's costs [lo, hi)
    const int bk = min(a.best_k, K);

    // ---- grid minimum (with index) and maximum key ------------------------------------------------------------------------
    unsigned long long best = ~0ull;
    unsigned kmax = 0u;
    for (int i = lo + tid; i < hi; i += nt) {
        const unsigned key = order_key(__ldcg(a.J + i));
        const unsigned long long c = ((unsigned long long)key << 32) | (unsigned)i;
        best = c < best ? c : best;
        kmax = max(kmax, key);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long n = __shfl_xor_sync(0xffffffffu, best, o);
        best = n < best ? n : best;
        kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, o));
    }
    if (lane == 0) { s_bestw[warp] = best; s_maxw[warp] = kmax; }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < nwarps; ++w) { best = s_bestw[w] < best ? s_bestw[w] : best; kmax = max(kmax, s_maxw[w]); }
        if (lo < hi) { atomicMin(a.g_best, best); atomicMax(a.g_kmax, kmax); }
    }
    grid.sync();
    best = __ldcg(a.g_best);
    kmax = __ldcg(a.g_kmax);
    const int best_idx = (int)(best & 0xFFFFFFFFull);
    const unsigned kmin = (unsigned)(best >> 32);

    // ---- radix select over the bits in which the keys differ (every block reaches the same prefix) -----------------------------
    int hbits = 32 - __clz((int)(kmin ^ kmax));
    unsigned prefix = (hbits >= 32) ? 0u : (kmin & ~((1u << hbits) - 1u));
    unsigned remaining = (unsigned)bk;
    int pass = 0;
    while (hbits > 0) {
        const int w = min(8, hbits), shift = hbits - w;
        const unsigned mask = (hbits >= 32) ? 0u : ~((1u << hbits) - 1u), digit = (1u << w) - 1u;
        for (int q = tid; q < 256; q += nt) s_hist[q] = 0u;
        __syncthreads();
        for (int i = lo + tid; i < hi; i += nt) {
            const unsigned key = order_key(__ldcg(a.J + i));
            if ((key & mask) == prefix) atomicAdd(&s_hist[(key >> shift) & digit], 1u);
        }
        __syncthreads();
        unsigned *gh = a.g_hist + pass * 256;
        for (int q = tid; q < 256; q += nt)
            if (s_hist[q]) atomicAdd(gh + q, s_hist[q]);
        grid.sync();
        if (warp == 0) {   // every block finds the bin of rank `remaining` in the merged histogram
            unsigned c[8], mine = 0u;
#pragma unroll
            for (int j = 0; j < 8; ++j) { c[j] = __ldcg(gh + lane * 8 + j); mine += c[j]; }
            unsigned incl = mine;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned n = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += n;
            }
            const unsigned before = incl - mine;
            const unsigned hit = __ballot_sync(0xffffffffu, incl >= remaining);
            if (lane == __ffs(hit) - 1) {
                unsigned cum = before;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (cum + c[j] >= remaining) { s_prefix = prefix | ((unsigned)(lane * 8 + j) << shift); s_remaining = remaining - cum; break; }
                    cum += c[j];
                }
            }
        }
        __syncthreads();
        prefix = s_prefix;
        remaining = s_remaining;
        hbits = shift;
        ++pass;
        __syncthreads();
    }
    const unsigned kth = prefix;
    const int ties_wanted = (int)remaining;

    // ---- per-block counts, then the ordered compaction at the block's offset ------------------------------------------------
    int n_less = 0, n_eq = 0;
    for (int i = lo + tid; i < hi; i += nt) {
        const unsigned key = order_key(__ldcg(a.J + i));
        n_less += key < kth ? 1 : 0;
        n_eq += key == kth ? 1 : 0;
    }
    int tot_less, tot_eq;
    block_excl_scan(n_less, s_w, tot_less);
    block_excl_scan(n_eq, s_w, tot_eq);
    if (tid == 0) { a.g_cnt[b] = tot_less; a.g_cnt[G + b] = tot_eq; }
    grid.sync();
    if (tid == 0) {   // elites and ties in the blocks before this one
        int el = 0, eq = 0;
        for (int q = 0; q < b; ++q) {
            const int l = __ldcg(a.g_cnt + q), e = __ldcg(a.g_cnt + G + q);
            el += l + max(0, min(e, ties_wanted - eq));
            eq += e;
        }
        s_base = el;
        s_remaining = (unsigned)eq;
    }
    __syncthreads();
    int n_el_before = s_base, n_eq_before = (int)s_remaining;
    for (int base = lo; base < hi; base += nt * 8) {   // each thread owns 8 consecutive plans of the chunk
        const int i0 = base + tid * 8;
        unsigned key[8];
        int eq = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            key[j] = order_key(__ldcg(a.J + min(i0 + j, K - 1)));
            eq += (i0 + j < hi && key[j] == kth) ? 1 : 0;
        }
        int teq, tel;
        int eq_rank = n_eq_before + block_excl_scan(eq, s_w, teq);
        unsigned take = 0u;
        int el = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const bool in = i0 + j < hi;
            const bool is_eq = in && key[j] == kth;
            if (in && (key[j] < kth || (is_eq && eq_rank < ties_wanted))) { take |= 1u << j; ++el; }
            eq_rank += is_eq ? 1 : 0;
        }
        int pos = n_el_before + block_excl_scan(el, s_w, tel);
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (take & (1u << j)) a.elite[pos++] = i0 + j;
        n_eq_before += teq;
        n_el_before += tel;
    }
    if (b == 0) {   // outputs, and the scratch goes back to its resting state (all blocks are past their last read of it)
        if (tid == 0) {
            if (a.best_out) *a.best_out = best_idx;
            if (a.last_iter) *a.u_out = cem_plan_value(a.mu[0], a.Q[(long long)best_idx * a.qs_k], a.sd[0], a.lo, a.hi);
            *a.g_best = ~0ull;
            *a.g_kmax = 0u;
        }
        for (int q = tid; q < 4 * 256; q += nt) a.g_hist[q] = 0u;
    }
}

// CEM statistics for large elite sets: one block per horizon step (plan_select leaves the elite list in a.elite).  Reads
// the distribution the plans were sampled from (a.mu, a.sd) and writes the updated one to the OTHER buffer
// (a.mu_out, a.sd_out), so blocks do not race on the shifted write of the last iteration.
__global__ void __launch_bounds__(256) cem_update_kernel(const __grid_constant__ PlanArgs a) {
    __shared__ float s_part[8];
    __shared__ float s_bc;
    const int t = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int bk = min(a.best_k, a.K), T = a.T;
    const float mu = a.mu[t], sd = a.sd[t];
    const float *q = a.Q + (long long)t * a.qs_t;
    float sum = 0.0f;
#pragma unroll 4
    for (int e = tid; e < bk; e += 256) sum += cem_plan_value(mu, q[(long long)a.elite[e] * a.qs_k], sd, a.lo, a.hi);
    sum = warp_sum(sum);
    if (lane == 0) s_part[warp] = sum;
    __syncthreads();
    if (tid == 0) {
        float v = 0.0f;
        for (int w = 0; w < 8; ++w) v += s_part[w];
        s_bc = __fdiv_rn(v, (float)bk);
    }
    __syncthreads();
    const float mean = s_bc;
    float ss = 0.0f;
#pragma unroll 4
    for (int e = tid; e < bk; e += 256) {
        const float d = cem_plan_value(mu, q[(long long)a.elite[e] * a.qs_k], sd, a.lo, a.hi) - mean;
        ss = fmaf(d, d, ss);
    }
    ss = warp_sum(ss);
    __syncthreads();
    if (lane == 0) s_part[warp] = ss;
    __syncthreads();
    if (tid != 0) return;
    float v = 0.0f;
    for (int w = 0; w < 8; ++w) v += s_part[w];
    const float stdev = sqrtf(__fdiv_rn(v, (float)bk));
    if (!a.last_iter) {
        a.mu_out[t] = mean;
        a.sd_out[t] = stdev;
    } else {   // clip, shift by one step, refill the tail (cem_tf.py:96-99)
        if (t > 0) { a.mu_out[t - 1] = mean; a.sd_out[t - 1] = clampf(stdev, a.sd_min, 1.0e8f); }
        if (t == T - 1) { a.mu_out[t] = a.mid; a.sd_out[t] = a.sd_init; }
    }
}

// ---- CEM fleets: the selection and statistics of experiment x = blockIdx.y --------------------------------------------------
// Draw eps[k][t] of experiment x in the iteration `a` describes: supplied [E][T][K], or Philox (group t / 4 of plan k).
template <bool PHILOX>
__device__ __forceinline__ float fleet_draw(const PlanArgs &a, const PlanFleetExt &fx, long long x, int k, int t) {
    if (!PHILOX) return a.Q[(x * a.T + t) * a.K + k];
    float n[4];
    philox_normals(fx.seed, (unsigned)k, fx.w1 + (unsigned)(t >> 2), fx.period, fx.e_offset + (unsigned)x, 4, n, 1);
    const int c = t & 3;
    return c == 0 ? n[0] : (c == 1 ? n[1] : (c == 2 ? n[2] : n[3]));
}

// Run by the last block of experiment x: plan_select on the experiment's K costs (from a copy of the arguments pointed at
// the experiment, stopping after the elite list), then what plan_select does after it -- u after the last iteration, the
// statistics (deferred to cem_update_fleet_kernel above 2048 elite entries) -- with the same arithmetic in the same order.
// PHILOX: the elites' draws are regenerated into s_eps [best_k][T] first.
template <bool PHILOX>
__device__ __forceinline__ void cem_fleet_select(const PlanArgs &a, const PlanFleetExt &fx, const float *s_mu,
                                                 const float *s_sd, float *s_mu2, float *s_sd2, int *s_elite, float *s_eps) {
    __shared__ PlanArgs s_a;
    __shared__ int s_best;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nt = blockDim.x, nwarps = nt >> 5;
    const int K = a.K, T = a.T, bk = min(a.best_k, K);
    const long long x = blockIdx.y;
    if (tid == 0) {
        s_a = a;
        s_a.J = a.J + x * K;
        s_a.elite = a.elite + x * K;   // used when the list does not fit in shared memory (deferred statistics)
        s_a.best_out = &s_best;
        s_a.defer_stats = 1;   // stop after the elite list ...
        s_a.last_iter = 0;     // ... without reading the draws
    }
    __syncthreads();
    plan_select<PLAN_CEM>(s_a, s_mu, s_sd, s_mu2, s_sd2, s_elite);   // ends with the elite list visible to the block
    if (a.last_iter && tid == 0)   // u = elite_Q[0, 0]; thread 0 wrote s_best
        a.u_out[x] = cem_plan_value(s_mu[0], fleet_draw<PHILOX>(a, fx, x, s_best, 0), s_sd[0], a.lo, a.hi);
    if (a.defer_stats) return;
    const int *elite = s_elite;   // statistics here: best_k x T <= 2048, the list is in shared memory
    if (PHILOX) {
        const int G4 = (T + 3) / 4;
        for (int i = tid; i < bk * G4; i += nt) {
            const int pos = i / G4, g = i - pos * G4;
            philox_normals(fx.seed, (unsigned)elite[pos], fx.w1 + (unsigned)g, fx.period, fx.e_offset + (unsigned)x,
                           min(4, T - 4 * g), s_eps + pos * T + 4 * g, 1);
        }
        __syncthreads();
    }
    const float *Q = a.Q + x * T * K;   // supplied draws of the experiment, [T][K]
    for (int t = warp; t < T; t += nwarps) {   // as plan_select
        float sum = 0.0f;
        for (int e = lane; e < bk; e += 32)
            sum += cem_plan_value(s_mu[t], PHILOX ? s_eps[e * T + t] : Q[(long long)t * K + elite[e]], s_sd[t], a.lo, a.hi);
        const float mean = __fdiv_rn(warp_sum(sum), (float)bk);
        float ss = 0.0f;
        for (int e = lane; e < bk; e += 32) {
            const float d =
                cem_plan_value(s_mu[t], PHILOX ? s_eps[e * T + t] : Q[(long long)t * K + elite[e]], s_sd[t], a.lo, a.hi) - mean;
            ss = fmaf(d, d, ss);
        }
        const float var = __fdiv_rn(warp_sum(ss), (float)bk);
        if (lane == 0) { s_mu2[t] = mean; s_sd2[t] = sqrtf(var); }
    }
    __syncthreads();
    float *mu_out = a.mu_out + x * T, *sd_out = a.sd_out + x * T;
    for (int t = tid; t < T; t += nt) {
        if (!a.last_iter) {
            mu_out[t] = s_mu2[t];
            sd_out[t] = s_sd2[t];
        } else if (t + 1 < T) {
            mu_out[t] = s_mu2[t + 1];
            sd_out[t] = clampf(s_sd2[t + 1], a.sd_min, 1.0e8f);
        } else {
            mu_out[t] = a.mid;
            sd_out[t] = a.sd_init;
        }
    }
}

// cem_update_kernel for fleets: block (t, x) updates step t of experiment x, same arithmetic in the same order.
template <bool PHILOX>
__global__ void __launch_bounds__(256) cem_update_fleet_kernel(const __grid_constant__ PlanArgs a,
                                                               const __grid_constant__ PlanFleetExt fx) {
    __shared__ float s_part[8];
    __shared__ float s_bc;
    const int t = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int bk = min(a.best_k, a.K), T = a.T;
    const long long x = blockIdx.y;
    const float mu = a.mu[x * T + t], sd = a.sd[x * T + t];
    const int *elite = a.elite + x * a.K;
    float sum = 0.0f;
    for (int e = tid; e < bk; e += 256) sum += cem_plan_value(mu, fleet_draw<PHILOX>(a, fx, x, elite[e], t), sd, a.lo, a.hi);
    sum = warp_sum(sum);
    if (lane == 0) s_part[warp] = sum;
    __syncthreads();
    if (tid == 0) {
        float v = 0.0f;
        for (int w = 0; w < 8; ++w) v += s_part[w];
        s_bc = __fdiv_rn(v, (float)bk);
    }
    __syncthreads();
    const float mean = s_bc;
    float ss = 0.0f;
    for (int e = tid; e < bk; e += 256) {
        const float d = cem_plan_value(mu, fleet_draw<PHILOX>(a, fx, x, elite[e], t), sd, a.lo, a.hi) - mean;
        ss = fmaf(d, d, ss);
    }
    ss = warp_sum(ss);
    __syncthreads();
    if (lane == 0) s_part[warp] = ss;
    __syncthreads();
    if (tid != 0) return;
    float v = 0.0f;
    for (int w = 0; w < 8; ++w) v += s_part[w];
    const float stdev = sqrtf(__fdiv_rn(v, (float)bk));
    float *mu_out = a.mu_out + x * T, *sd_out = a.sd_out + x * T;
    if (!a.last_iter) {
        mu_out[t] = mean;
        sd_out[t] = stdev;
    } else {   // clip, shift by one step, refill the tail (cem_tf.py:96-99)
        if (t > 0) { mu_out[t - 1] = mean; sd_out[t - 1] = clampf(stdev, a.sd_min, 1.0e8f); }
        if (t == T - 1) { mu_out[t] = a.mid; sd_out[t] = a.sd_init; }
    }
}

// NSUB = 10: the substeps of the predictors' operating point unrolled (control_step); 0: a.ode.n substeps in a loop.
// FLEET (PLAN_CEM, plan_fleet_kernel): block (b, e) evaluates plans b * 256.. of experiment e from its state, distribution,
// u_prev and cost parameters `cost`; the last block of the experiment (its own ticket) selects on its K costs.  PHILOX:
// the draws come from Philox in the rollout thread, four per call as the horizon advances.  FLEET = false compiles to
// the code plan_kernel compiled to before the fleet existed.
template <int INTEG, int COST, int MODE, int NSUB, bool FLEET, bool PHILOX>
__device__ __forceinline__ void plan_body(const PlanArgs &a, const PlanFleetExt *fx, const CostParams &cost) {
    extern __shared__ float smem[];   // PLAN_CEM: mu[T], sd[T], mu2[T], sd2[T], elite list [elite_smem], PHILOX: elites' draws
    __shared__ unsigned s_ticket;
    const int tid = threadIdx.x, T = a.T;
    const long long x = FLEET ? blockIdx.y : 0;   // the experiment
    float *s_mu = smem, *s_sd = smem + T;
    if (MODE == PLAN_CEM) {
        for (int t = tid; t < T; t += blockDim.x) { s_mu[t] = a.mu[x * T + t]; s_sd[t] = a.sd[x * T + t]; }
        __syncthreads();
    }
    const int k = blockIdx.x * blockDim.x + tid;
    const bool active = k < a.K;
    const int kc = min(k, a.K - 1);

    State z = load_state(FLEET ? fx->s + x * 8 : (a.use_inline ? a.s_inline : a.s));
    const OdeParams ode = pin_params(a.ode, z.th);
    float c_cost = cosf(z.th);  // the plugins take cos(angle) of the stored angle (default.py:34)
    // FLEET: plan kc of experiment x in the [E][T][K] draws / plans, one offset for both (qs_k = 1, qs_t = K)
    const long long qoff = x * T * a.K + kc;
    const float *q = FLEET ? a.Q + qoff : a.Q + (long long)kc * a.qs_k;
    float *qo = (MODE == PLAN_CEM && a.Q_out) ? (FLEET ? a.Q_out + qoff : a.Q_out + (long long)kc * a.qs_k) : nullptr;
    float *traj = (!FLEET && a.traj_out) ? a.traj_out + (long long)kc * a.ts_k : nullptr;   // fleets write no trajectories
    float Jacc = 0.0f, up = FLEET ? a.u_out[x] : a.u_prev;
    float nr[4];   // PHILOX: the draws of the current group of four steps, consumed from nr[0]
    // default / quadratic_boundary: the T+1 entries are summed in the reference backend's order (cps_device.cuh RowSumPlan)
    constexpr bool ROWSUM = (COST == COST_DEFAULT || COST == COST_QB);
    const RowSumPlan rsp = row_sum_plan(T + 1);
    float *sl = smem + a.rs_off + tid;
    const int ss = blockDim.x;
    float rs_tail = 0.0f;
    if (ROWSUM) row_sum_init(rsp, sl, ss);
    float qn = PHILOX ? 0.0f : q[0];
#pragma unroll 1
    for (int t = 0; t < T; ++t) {
        float u = qn;
        if (PHILOX) {
            if ((t & 3) == 0)
                philox_normals(fx->seed, (unsigned)kc, fx->w1 + (unsigned)(t >> 2), fx->period, fx->e_offset + (unsigned)x, 4,
                               nr, 1);
            u = nr[0];
            nr[0] = nr[1]; nr[1] = nr[2]; nr[2] = nr[3];
        } else if (t + 1 < T) {
            qn = FLEET ? a.Q[qoff + (long long)(t + 1) * a.K] : q[(long long)(t + 1) * a.qs_t];  // prefetch under the integration
        }
        if (MODE == PLAN_CEM) {
            u = cem_plan_value(s_mu[t], u, s_sd[t], a.lo, a.hi);
            if (active && qo) (FLEET ? a.Q_out[qoff + (long long)t * a.K] : qo[(long long)t * a.qs_t]) = u;
        }
        if (COST != COST_NONE) {
            const float st = stage_cost<COST>(cost, c_cost, z.w, z.x, u, up);
            if (ROWSUM) row_sum_push(rsp, sl, ss, rs_tail, t, st - cost.max_cost);  // get_stage_cost shift
            else Jacc += st;
        }
        if (active && traj) store_state(traj + (long long)t * a.ts_t, a.ts_c, z);
        control_step<INTEG, SC_ROTATE, false, false, false, NSUB>(ode, z, u);
        c_cost = z.c;
        up = u;
    }
    if (COST != COST_NONE) {
        const float term = terminal_cost<COST>(cost, z.th, z.x);
        if (ROWSUM) {
            row_sum_push(rsp, sl, ss, rs_tail, T, term);
            Jacc = row_sum_finish(rsp, sl, ss, rs_tail);
        } else {
            Jacc += term;
        }
    }
    if (active && traj) store_state(traj + (long long)T * a.ts_t, a.ts_c, z);
    const float J = __fdiv_rn(Jacc, (float)(T + 1));  // mean over the T+1 entries (Cost_Functions/__init__.py:90-93)
    if (active) {
        if (a.J) a.J[(FLEET ? (long long)blockIdx.y : 0LL) * a.K + k] = J;   // blockIdx.y re-read: no register kept over the loop
        if (!isfinite(J)) atomicAdd(a.nonfinite, 1);
    }
    if (a.select == SELECT_NONE) return;

    __threadfence();
    __syncthreads();
    if (tid == 0) s_ticket = atomicAdd(a.ticket + (FLEET ? blockIdx.y : 0u), 1u);
    __syncthreads();
    if (s_ticket != gridDim.x - 1u) return;
    __threadfence();
    if (FLEET) {
        int *s_elite = reinterpret_cast<int *>(smem + 4 * T);
        cem_fleet_select<PHILOX>(a, *fx, s_mu, s_sd, smem + 2 * T, smem + 3 * T, s_elite,
                                 reinterpret_cast<float *>(s_elite + a.elite_smem));
    } else {
        plan_select<MODE>(a, s_mu, s_sd, smem + 2 * T, smem + 3 * T, reinterpret_cast<int *>(smem + 4 * T));
    }
    if (tid == 0) a.ticket[FLEET ? blockIdx.y : 0u] = 0u;  // re-arm
}
template <int INTEG, int COST, int MODE, int NSUB = 0>
__global__ void __launch_bounds__(256, 4) plan_kernel(const __grid_constant__ PlanArgs a) {
    plan_body<INTEG, COST, MODE, NSUB, false, false>(a, nullptr, a.cost);
}
// CEM fleets: grid (ceil(K / 256), E); experiment e's cost parameters are folded for its targets once per block
template <int INTEG, int COST, int NSUB, bool PHILOX>
__global__ void __launch_bounds__(256, 4) plan_fleet_kernel(const __grid_constant__ PlanArgs a,
                                                            const __grid_constant__ PlanFleetExt fx) {
    __shared__ CostParams s_cost;
    if (threadIdx.x == 0) s_cost = fold_cost_e(fx.cost_up, fx.cost_dn, fx.tp, fx.te, (int)blockIdx.y);
    __syncthreads();
    plan_body<INTEG, COST, PLAN_CEM, NSUB, true, PHILOX>(a, &fx, s_cost);
}

// Many plans, no selecting block, time-major plans: two plans per thread (k, k + 1) in packed FP32, as mppi_solve_block2
// does for the MPPI solve.  Per plan the arithmetic is that of plan_kernel, so the costs are bit-identical (tested).
#define CPS_PLAN_PAIR_MIN 65536   /* measured: at 16384 and 32768 plans one per thread is 10-25 % faster (latency regime) */
template <int INTEG, int COST, int MODE>
__global__ void __launch_bounds__(128, 4) plan_pair_kernel(const __grid_constant__ PlanArgs a) {
    extern __shared__ float smem[];   // PLAN_CEM: mu[T], sd[T]
    const int tid = threadIdx.x, T = a.T;
    float *s_mu = smem, *s_sd = smem + T;
    if (MODE == PLAN_CEM) {
        for (int t = tid; t < T; t += blockDim.x) { s_mu[t] = a.mu[t]; s_sd[t] = a.sd[t]; }
        __syncthreads();
    }
    const int k = 2 * (blockIdx.x * blockDim.x + tid);   // K is even: both plans active or both not
    if (k >= a.K) return;
    const State z1 = load_state(a.use_inline ? a.s_inline : a.s);
    State2 z = join_states(z1, z1);
    const OdeParams ode = pin_params(a.ode, z1.th);
    float cc0 = cosf(z1.th), cc1 = cc0;
    const float *q = a.Q + k;                            // qs_k == 1
    float *qo = (MODE == PLAN_CEM && a.Q_out) ? a.Q_out + k : nullptr;
    float Ja0 = 0.0f, Ja1 = 0.0f, up0 = a.u_prev, up1 = a.u_prev;
    constexpr bool ROWSUM = (COST == COST_DEFAULT || COST == COST_QB);   // see plan_kernel
    const RowSumPlan rsp = row_sum_plan(T + 1);
    float2 *sl = reinterpret_cast<float2 *>(smem + a.rs_off) + tid;
    const int ss = blockDim.x;
    float2 rs_tail = make_float2(0.0f, 0.0f);
    if (ROWSUM) row_sum_init(rsp, sl, ss);
    float2 qn = *reinterpret_cast<const float2 *>(q);
#pragma unroll 1
    for (int t = 0; t < T; ++t) {
        float u0 = qn.x, u1 = qn.y;
        if (t + 1 < T) qn = *reinterpret_cast<const float2 *>(q + (long long)(t + 1) * a.qs_t);
        if (MODE == PLAN_CEM) {
            u0 = cem_plan_value(s_mu[t], u0, s_sd[t], a.lo, a.hi);
            u1 = cem_plan_value(s_mu[t], u1, s_sd[t], a.lo, a.hi);
            if (qo) *reinterpret_cast<float2 *>(qo + (long long)t * a.qs_t) = make_float2(u0, u1);
        }
        if (COST != COST_NONE) {
            const float st0 = stage_cost<COST>(a.cost, cc0, lo(z.w), lo(z.x), u0, up0);
            const float st1 = stage_cost<COST>(a.cost, cc1, hi(z.w), hi(z.x), u1, up1);
            if (ROWSUM) row_sum_push(rsp, sl, ss, rs_tail, t, make_float2(st0 - a.cost.max_cost, st1 - a.cost.max_cost));
            else { Ja0 += st0; Ja1 += st1; }
        }
        control_step2<INTEG, false>(ode, z, f2(u0, u1));
        cc0 = lo(z.c); cc1 = hi(z.c);
        up0 = u0; up1 = u1;
    }
    if (COST != COST_NONE) {
        const float tm0 = terminal_cost<COST>(a.cost, lo(z.th), lo(z.x)), tm1 = terminal_cost<COST>(a.cost, hi(z.th), hi(z.x));
        if (ROWSUM) {
            row_sum_push(rsp, sl, ss, rs_tail, T, make_float2(tm0, tm1));
            const float2 r = row_sum_finish(rsp, sl, ss, rs_tail);
            Ja0 = r.x; Ja1 = r.y;
        } else {
            Ja0 += tm0; Ja1 += tm1;
        }
    }
    const float J0 = __fdiv_rn(Ja0, (float)(T + 1)), J1 = __fdiv_rn(Ja1, (float)(T + 1));
    a.J[k] = J0; a.J[k + 1] = J1;
    if (!isfinite(J0)) atomicAdd(a.nonfinite, 1);
    if (!isfinite(J1)) atomicAdd(a.nonfinite, 1);
}

template <int INTEG, int MODE>
static void (*pick_plan_pair2(int cost))(const PlanArgs) {
    switch (cost) {
    case CPS_COST_DEFAULT: return plan_pair_kernel<INTEG, COST_DEFAULT, MODE>;
    case CPS_COST_QUADRATIC_BOUNDARY: return plan_pair_kernel<INTEG, COST_QB, MODE>;
    case CPS_COST_QB_GRAD_MINIMAL: return plan_pair_kernel<INTEG, COST_GRADMIN, MODE>;
    case CPS_COST_QB_GRAD: return plan_pair_kernel<INTEG, COST_GRAD, MODE>;
    default: return nullptr;
    }
}
static void (*pick_plan_pair(int integ, int cost, int mode))(const PlanArgs) {
    if (integ == CPS_EULER_V0) return mode == PLAN_CEM ? pick_plan_pair2<0, PLAN_CEM>(cost) : pick_plan_pair2<0, PLAN_Q>(cost);
    return mode == PLAN_CEM ? pick_plan_pair2<1, PLAN_CEM>(cost) : pick_plan_pair2<1, PLAN_Q>(cost);
}
// Dynamic shared memory of a plan launch: `base` bytes of the kernel's own staging, then (MAX_COST plugins) the row-sum
// slots of the block's rollouts.  Sets a.rs_off.
static size_t plan_smem(const cps_handle *h, PlanArgs &a, size_t base, int block, int per_thread) {
    size_t fl = ((base + 3) / 4 + 1) & ~(size_t)1;
    a.rs_off = (int)fl;
    if (h->cfg.cost_id == CPS_COST_DEFAULT || h->cfg.cost_id == CPS_COST_QUADRATIC_BOUNDARY)
        fl += (size_t)row_sum_slots(a.T + 1) * block * per_thread;
    else if (base == 0) return 0;
    return fl * sizeof(float);
}
// true when a launch described by `a` (select == SELECT_NONE) can take the packed kernel
static bool plan_pair_ok(const cps_handle *h, const PlanArgs &a) {
    return a.K >= CPS_PLAN_PAIR_MIN && (a.K % 2) == 0 && a.qs_k == 1 && (a.qs_t % 2) == 0 && !a.traj_out && a.J &&
           !(h->cfg.flags & CPS_FLAG_NO_PAIRS) && ((uintptr_t)a.Q % 8) == 0 && (!a.Q_out || ((uintptr_t)a.Q_out % 8) == 0);
}
static void plan_pair_launch(cps_handle *h, PlanArgs &a, int mode) {
    const long long threads = a.K / 2;
    const int block = threads <= 148 * 32 * 4 ? 32 : (threads <= 148 * 64 * 8 ? 64 : 128);
    const int grid = (int)((threads + block - 1) / block);
    const size_t smem = plan_smem(h, a, mode == PLAN_CEM ? sizeof(float) * 2 * (size_t)a.T : 0, block, 2);
    auto fn = pick_plan_pair(h->cfg.integrator, h->cfg.cost_id, mode);
    if (smem > 48 * 1024) cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    fn<<<grid, block, smem, h->stream>>>(a);
}

// ---- host side ---------------------------------------------------------------------------------------------------------
typedef void (*plan_fn)(const PlanArgs);
template <int INTEG, int MODE, int NSUB>
static plan_fn pick_plan2(int cost) {
    switch (cost) {
    case CPS_COST_DEFAULT: return plan_kernel<INTEG, COST_DEFAULT, MODE, NSUB>;
    case CPS_COST_QUADRATIC_BOUNDARY: return plan_kernel<INTEG, COST_QB, MODE, NSUB>;
    case CPS_COST_QB_GRAD_MINIMAL: return plan_kernel<INTEG, COST_GRADMIN, MODE, NSUB>;
    case CPS_COST_QB_GRAD: return plan_kernel<INTEG, COST_GRAD, MODE, NSUB>;
    default: return nullptr;
    }
}
template <int INTEG, int MODE>
static plan_fn pick_plan1(int cost, int n_sub) {
    return n_sub == 10 ? pick_plan2<INTEG, MODE, 10>(cost) : pick_plan2<INTEG, MODE, 0>(cost);
}
static plan_fn pick_plan(int integ, int cost, int mode, int n_sub) {
    if (integ == CPS_EULER_V0) return mode == PLAN_CEM ? pick_plan1<0, PLAN_CEM>(cost, n_sub) : pick_plan1<0, PLAN_Q>(cost, n_sub);
    return mode == PLAN_CEM ? pick_plan1<1, PLAN_CEM>(cost, n_sub) : pick_plan1<1, PLAN_Q>(cost, n_sub);
}

void cps_plan_free(cps_handle *h) {
    PlanState *P = h->plan;
    if (!P) return;
    cudaFree(P->d_J); cudaFree(P->d_mu); cudaFree(P->d_sd); cudaFree(P->d_elite); cudaFree(P->d_best); cudaFree(P->d_ticket);
    cudaFree(P->d_gbest); cudaFree(P->d_gkmax); cudaFree(P->d_ghist); cudaFree(P->d_gcnt);
    delete P;
    h->plan = nullptr;
}

static int plan_state(cps_handle *h, PlanState **out) {
    if (h->plan) { *out = h->plan; return CPS_OK; }
    PlanState *P = new (std::nothrow) PlanState();
    if (!P) return fail(h, CPS_ERR_INVALID, "cps_plan: out of host memory");
    memset(P, 0, sizeof(*P));
    const size_t K = h->cfg.num_rollouts, T = h->cfg.horizon;
    cudaError_t e = cudaMalloc(&P->d_J, sizeof(float) * K);
    if (e == cudaSuccess) e = cudaMalloc(&P->d_mu, sizeof(float) * 2 * T);
    if (e == cudaSuccess) e = cudaMalloc(&P->d_sd, sizeof(float) * 2 * T);
    if (e == cudaSuccess) e = cudaMalloc(&P->d_elite, sizeof(int) * K);
    if (e == cudaSuccess) e = cudaMalloc(&P->d_best, sizeof(int));
    if (e == cudaSuccess) e = cudaMalloc(&P->d_ticket, sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMalloc(&P->d_gbest, sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMalloc(&P->d_gkmax, sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMalloc(&P->d_ghist, sizeof(unsigned) * 4 * 256);
    if (e == cudaSuccess) e = cudaMalloc(&P->d_gcnt, sizeof(int) * 2 * 1024);
    if (e == cudaSuccess) e = cudaMemset(P->d_gbest, 0xFF, sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemset(P->d_gkmax, 0, sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMemset(P->d_ghist, 0, sizeof(unsigned) * 4 * 256);
    if (e == cudaSuccess) e = cudaMemset(P->d_ticket, 0, sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMemset(P->d_mu, 0, sizeof(float) * 2 * T);
    if (e == cudaSuccess) e = cudaMemset(P->d_sd, 0, sizeof(float) * 2 * T);
    if (e != cudaSuccess) {   // nothing half-built stays attached to the handle
        cudaFree(P->d_J); cudaFree(P->d_mu); cudaFree(P->d_sd); cudaFree(P->d_elite); cudaFree(P->d_best); cudaFree(P->d_ticket);
        cudaFree(P->d_gbest); cudaFree(P->d_gkmax); cudaFree(P->d_ghist); cudaFree(P->d_gcnt);
        delete P;
        return fail(h, CPS_ERR_CUDA, "cps_plan: allocating the planner scratch: %s", cudaGetErrorString(e));
    }
    h->plan = P;
    *out = P;
    return CPS_OK;
}

static int plan_check(cps_handle *h, const char *who) {
    if (h->cfg.integrator == CPS_PREDICTOR_NEURAL)
        return fail(h, CPS_ERR_UNSUPPORTED, "%s: ODE predictors only (neural predictor: cps_plan_cost, or cps_net_rollout + cps_trajectory_cost)", who);
    if (h->cfg.cost_id == CPS_COST_NONE || h->cfg.cost_id == CPS_COST_LEGACY_MPPI)
        return fail(h, CPS_ERR_NOT_CONFIGURED, "%s: the handle has no cost-function plugin", who);
    if (h->cfg.flags & (CPS_FLAG_SUBSTEP_SINCOS | CPS_FLAG_FAST_DIV))
        return fail(h, CPS_ERR_UNSUPPORTED, "%s: built for the default (rotation) substeps only", who);
    return CPS_OK;
}

static void plan_common(cps_handle *h, PlanArgs &a, const float *s_dev, float u_prev, int K, int T) {
    memset(&a, 0, sizeof(a));
    a.ode = h->ode; a.cost = h->cost;
    a.s = s_dev;
    a.use_inline = h->inline_s ? 1 : 0;
    for (int c = 0; c < 6; ++c) a.s_inline[c] = h->inline_s ? h->inline_s[c] : 0.0f;
    a.lo = h->mppi_in[5]; a.hi = h->mppi_in[6];
    a.inv_T1 = 1.0f / (float)(T + 1);
    a.u_prev = u_prev;
    a.K = K; a.T = T;
    a.nonfinite = h->d_nonfinite;
}

// Without a selection step small K is latency bound: one warp per block spreads the warps over the SMs.  With one, the
// block that finishes last works alone on the K costs, so blocks are 256 wide (rollout latency is the same: the
// 10 x T substep dependence chain of one warp; 8 warps share an SM without slowing each other).
static void plan_geometry(int K, bool select, int &grid, int &block) {
    if (select) block = 256;
    else block = (K <= 148 * 32 * 4) ? 32 : (K <= 148 * 64 * 8 ? 64 : 128);
    grid = (K + block - 1) / block;
}

extern "C" int cps_plan_cost(cps_handle *h, const float *s_dev, const float *Q_dev, int q_layout, int K, int T, float u_prev,
                             float *J_out_dev, float *traj_out_dev, int traj_layout) {
    if (!h) return CPS_ERR_INVALID;
    if (!s_dev || !Q_dev || !J_out_dev) return fail(h, CPS_ERR_INVALID, "cps_plan_cost: null pointer");
    if (K < 1 || T < 1) return fail(h, CPS_ERR_INVALID, "cps_plan_cost: K and T must be positive");
    if (h->cfg.integrator == CPS_PREDICTOR_NEURAL)
        return cps_net_plan_cost(h, s_dev, Q_dev, q_layout, K, T, u_prev, J_out_dev, traj_out_dev, traj_layout);
    int rc = plan_check(h, "cps_plan_cost");
    if (rc != CPS_OK) return rc;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    PlanArgs a;
    plan_common(h, a, s_dev, u_prev, K, T);
    a.Q = Q_dev;
    if (q_layout == CPS_TIME_MAJOR) { a.qs_k = 1; a.qs_t = K; } else { a.qs_k = T; a.qs_t = 1; }
    a.J = J_out_dev;
    a.traj_out = traj_out_dev;
    if (traj_layout == CPS_TIME_MAJOR) { a.ts_k = 1; a.ts_t = 6LL * K; a.ts_c = K; }
    else { a.ts_k = (T + 1) * 6LL; a.ts_t = 6; a.ts_c = 1; }
    a.select = SELECT_NONE;
    if (plan_pair_ok(h, a)) {
        plan_pair_launch(h, a, PLAN_Q);
    } else {
        int grid, block;
        plan_geometry(K, false, grid, block);
        plan_fn fn = pick_plan(h->cfg.integrator, h->cfg.cost_id, PLAN_Q, h->ode.n);
        const size_t smem = plan_smem(h, a, 0, block, 1);
        if (smem > 48 * 1024) CUDA_TRY(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        fn<<<grid, block, smem, h->stream>>>(a);
    }
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

extern "C" int cps_plan_random_action(cps_handle *h, const float *s_dev, const float *Q_dev, int q_layout, float u_prev,
                                      float *u_out_dev, float *J_out_dev, int *best_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    if (!s_dev || !Q_dev || !u_out_dev) return fail(h, CPS_ERR_INVALID, "cps_plan_random_action: null pointer");
    int rc = plan_check(h, "cps_plan_random_action");
    if (rc != CPS_OK) return rc;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    PlanState *P;
    if ((rc = plan_state(h, &P)) != CPS_OK) return rc;
    const int K = h->cfg.num_rollouts, T = h->cfg.horizon;
    PlanArgs a;
    plan_common(h, a, s_dev, u_prev, K, T);
    a.Q = Q_dev;
    if (q_layout == CPS_TIME_MAJOR) { a.qs_k = 1; a.qs_t = K; } else { a.qs_k = T; a.qs_t = 1; }
    a.J = J_out_dev ? J_out_dev : P->d_J;
    a.select = SELECT_ARGMIN;
    a.ticket = P->d_ticket; a.elite = P->d_elite;
    a.u_out = u_out_dev;
    a.best_out = best_out_dev ? best_out_dev : P->d_best;
    int grid, block;
    plan_geometry(K, true, grid, block);
    plan_fn fn = pick_plan(h->cfg.integrator, h->cfg.cost_id, PLAN_Q, h->ode.n);
    const size_t smem = plan_smem(h, a, 0, block, 1);
    if (smem > 48 * 1024) CUDA_TRY(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fn<<<grid, block, smem, h->stream>>>(a);
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

extern "C" int cps_plan_random_action_host(cps_handle *h, const float *s_host, const float *Q_dev, int q_layout, float u_prev,
                                           float *u_out_host) {
    if (!h) return CPS_ERR_INVALID;
    if (!s_host || !u_out_host) return fail(h, CPS_ERR_INVALID, "cps_plan_random_action_host: null pointer");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    // one stream operation: state in the parameter block, control written into mapped pinned host memory
    float *u_dst = h->h_pin_dev ? h->h_pin_dev + 8 : h->d_u;
    h->inline_s = s_host;
    int rc = cps_plan_random_action(h, h->d_s, Q_dev, q_layout, u_prev, u_dst, nullptr, nullptr);
    h->inline_s = nullptr;
    if (rc != CPS_OK) return rc;
    if (!h->h_pin_dev) CUDA_TRY(h, cudaMemcpyAsync(h->h_pin + 8, h->d_u, sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    *u_out_host = h->h_pin[8];
    return CPS_OK;
}

// ---- CEM --------------------------------------------------------------------------------------------------------------
extern "C" int cps_cem_reset(cps_handle *h) {
    if (!h) return CPS_ERR_INVALID;
    PlanState *P = h->plan;
    if (!P || !P->configured_cem) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_cem_reset: cps_cem_configure first");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const int T = h->cfg.horizon;
    float *tmp = new (std::nothrow) float[2 * (size_t)T];
    if (!tmp) return fail(h, CPS_ERR_INVALID, "cps_cem_reset: out of host memory");
    const float mid = (h->mppi_in[5] + h->mppi_in[6]) * 0.5f;  // optimizer_reset (cem_tf.py:112-116)
    for (int t = 0; t < T; ++t) { tmp[t] = mid; tmp[T + t] = P->sd_init; }
    cudaError_t e = cudaMemcpyAsync(P->d_mu + (size_t)P->cur * T, tmp, sizeof(float) * T, cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(P->d_sd + (size_t)P->cur * T, tmp + T, sizeof(float) * T, cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    delete[] tmp;
    CUDA_TRY(h, e);
    return CPS_OK;
}

extern "C" int cps_cem_configure(cps_handle *h, int best_k, float initial_stdev, float stdev_min) {
    if (!h) return CPS_ERR_INVALID;
    int rc = plan_check(h, "cps_cem_configure");
    if (rc != CPS_OK) return rc;
    if (best_k < 1 || best_k > h->cfg.num_rollouts)
        return fail(h, CPS_ERR_INVALID, "cps_cem_configure: cem_best_k must lie in [1, num_rollouts]");
    if (!(initial_stdev >= 0.0f) || !(stdev_min >= 0.0f)) return fail(h, CPS_ERR_INVALID, "cps_cem_configure: negative stdev");
    if (sizeof(float) * 4 * (size_t)h->cfg.horizon + sizeof(int) * 2048 > 200 * 1024)
        return fail(h, CPS_ERR_UNSUPPORTED, "cps_cem_configure: horizon too large for shared memory");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    PlanState *P;
    if ((rc = plan_state(h, &P)) != CPS_OK) return rc;
    P->best_k = best_k; P->sd_init = initial_stdev; P->sd_min = stdev_min;
    P->configured_cem = 1;
    return cps_cem_reset(h);
}

extern "C" int cps_cem_step(cps_handle *h, const float *s_dev, const float *eps_dev, int eps_layout, int n_iterations,
                            float u_prev, float *u_out_dev, float *Q_out_dev, float *J_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    PlanState *P = h->plan;
    if (!P || !P->configured_cem) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_cem_step: cps_cem_configure first");
    if (!s_dev || !eps_dev || !u_out_dev) return fail(h, CPS_ERR_INVALID, "cps_cem_step: null pointer");
    if (n_iterations < 1) return fail(h, CPS_ERR_INVALID, "cps_cem_step: n_iterations < 1");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const int K = h->cfg.num_rollouts, T = h->cfg.horizon;
    PlanArgs a;
    plan_common(h, a, s_dev, u_prev, K, T);
    if (eps_layout == CPS_TIME_MAJOR) { a.qs_k = 1; a.qs_t = K; } else { a.qs_k = T; a.qs_t = 1; }
    a.J = J_out_dev ? J_out_dev : P->d_J;
    a.select = SELECT_CEM;
    a.best_k = P->best_k; a.sd_min = P->sd_min; a.sd_init = P->sd_init;
    a.mid = (a.lo + a.hi) * 0.5f;
    a.ticket = P->d_ticket; a.elite = P->d_elite;
    a.u_out = u_out_dev; a.best_out = P->d_best;
    int grid, block;
    plan_geometry(K, true, grid, block);
    a.elite_smem = 0;   // set below once defer_stats is known
    const size_t smem = sizeof(float) * 4 * (size_t)T + sizeof(int) * (size_t)(((long long)P->best_k * T > 2048) ? 0 : P->best_k);
    plan_fn fn = pick_plan(h->cfg.integrator, h->cfg.cost_id, PLAN_CEM, h->ode.n);
    // small elite sets: the selecting block also computes the T x best_k statistics; large ones: a second launch with
    // one block per horizon step
    a.defer_stats = ((long long)P->best_k * T > 2048) ? 1 : 0;
    a.elite_smem = a.defer_stats ? 0 : P->best_k;   // the update kernel reads the list from global memory
    // many plans: rollouts + costs without a selecting block (the latency geometry of cps_plan_cost), then the selection by
    // the whole grid (cem_select_kernel, cooperative launch, one block per SM) and the statistics kernel
    const bool multi = K > CPS_CEM_MULTIBLOCK_MIN;
    int sel_grid = 1;
    if (multi) {
        int dev = 0, sms = 148, coop = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
        if (!coop) return fail(h, CPS_ERR_UNSUPPORTED, "cps_cem_step: the device does not support cooperative launches");
        sel_grid = sms < 1024 ? sms : 1024;
        plan_geometry(K, false, grid, block);
        a.select = SELECT_NONE;
        a.defer_stats = 1;
        a.g_best = P->d_gbest; a.g_kmax = P->d_gkmax; a.g_hist = P->d_ghist; a.g_cnt = P->d_gcnt;
    }
    for (int it = 0; it < n_iterations; ++it) {
        a.Q = eps_dev + (size_t)it * K * T;
        a.last_iter = (it == n_iterations - 1) ? 1 : 0;
        a.Q_out = a.last_iter ? Q_out_dev : nullptr;   // Q_logged is the last iteration's plans (cem_tf.py:93)
        a.mu = P->d_mu + (size_t)P->cur * T; a.sd = P->d_sd + (size_t)P->cur * T;
        a.mu_out = P->d_mu + (size_t)(1 - P->cur) * T; a.sd_out = P->d_sd + (size_t)(1 - P->cur) * T;
        if (multi && plan_pair_ok(h, a) && sizeof(float) * 2 * (size_t)T <= 48 * 1024) {
            plan_pair_launch(h, a, PLAN_CEM);
        } else {
            const size_t sm = plan_smem(h, a, smem, block, 1);
            if (sm > 200 * 1024) return fail(h, CPS_ERR_UNSUPPORTED, "cps_cem_step: horizon too large for shared memory");
            if (sm > 48 * 1024) CUDA_TRY(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
            fn<<<grid, block, sm, h->stream>>>(a);
        }
        h->launches += 1;
        if (multi) {
            void *args[] = {(void *)&a};
            CUDA_TRY(h, cudaLaunchCooperativeKernel((const void *)cem_select_kernel, dim3(sel_grid), dim3(256), args, 0, h->stream));
            h->launches += 1;
        }
        if (a.defer_stats) {
            cem_update_kernel<<<T, 256, 0, h->stream>>>(a);
            h->launches += 1;
        }
        P->cur = 1 - P->cur;
    }
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

extern "C" int cps_cem_step_host(cps_handle *h, const float *s_host, const float *eps_dev, int eps_layout, int n_iterations,
                                 float u_prev, float *u_out_host) {
    if (!h) return CPS_ERR_INVALID;
    if (!s_host || !u_out_host) return fail(h, CPS_ERR_INVALID, "cps_cem_step_host: null pointer");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    float *u_dst = h->h_pin_dev ? h->h_pin_dev + 8 : h->d_u;
    h->inline_s = s_host;
    int rc = cps_cem_step(h, h->d_s, eps_dev, eps_layout, n_iterations, u_prev, u_dst, nullptr, nullptr);
    h->inline_s = nullptr;
    if (rc != CPS_OK) return rc;
    if (!h->h_pin_dev) CUDA_TRY(h, cudaMemcpyAsync(h->h_pin + 8, h->d_u, sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    *u_out_host = h->h_pin[8];
    return CPS_OK;
}

extern "C" int cps_cem_get_distribution(cps_handle *h, float *mu_host, float *stdev_host) {
    if (!h) return CPS_ERR_INVALID;
    PlanState *P = h->plan;
    if (!P || !P->configured_cem) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_cem_get_distribution: cps_cem_configure first");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t T = h->cfg.horizon;
    if (mu_host) CUDA_TRY(h, cudaMemcpyAsync(mu_host, P->d_mu + P->cur * T, sizeof(float) * T, cudaMemcpyDeviceToHost, h->stream));
    if (stdev_host) CUDA_TRY(h, cudaMemcpyAsync(stdev_host, P->d_sd + P->cur * T, sizeof(float) * T, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}

extern "C" int cps_cem_set_distribution(cps_handle *h, const float *mu_host, const float *stdev_host) {
    if (!h) return CPS_ERR_INVALID;
    PlanState *P = h->plan;
    if (!P || !P->configured_cem) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_cem_set_distribution: cps_cem_configure first");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t T = h->cfg.horizon;
    if (mu_host) CUDA_TRY(h, cudaMemcpyAsync(P->d_mu + P->cur * T, mu_host, sizeof(float) * T, cudaMemcpyHostToDevice, h->stream));
    if (stdev_host) CUDA_TRY(h, cudaMemcpyAsync(P->d_sd + P->cur * T, stdev_host, sizeof(float) * T, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}

// ---- CEM fleets (cps_cem_fleet.cu) ------------------------------------------------------------------------------------
typedef void (*plan_fleet_fn)(const PlanArgs, const PlanFleetExt);
template <int INTEG, int NSUB, bool PHILOX>
static plan_fleet_fn pick_plan_fleet3(int cost) {
    switch (cost) {
    case CPS_COST_DEFAULT: return plan_fleet_kernel<INTEG, COST_DEFAULT, NSUB, PHILOX>;
    case CPS_COST_QUADRATIC_BOUNDARY: return plan_fleet_kernel<INTEG, COST_QB, NSUB, PHILOX>;
    case CPS_COST_QB_GRAD_MINIMAL: return plan_fleet_kernel<INTEG, COST_GRADMIN, NSUB, PHILOX>;
    case CPS_COST_QB_GRAD: return plan_fleet_kernel<INTEG, COST_GRAD, NSUB, PHILOX>;
    default: return nullptr;
    }
}
template <int INTEG, int NSUB>
static plan_fleet_fn pick_plan_fleet2(int cost, bool philox) {
    return philox ? pick_plan_fleet3<INTEG, NSUB, true>(cost) : pick_plan_fleet3<INTEG, NSUB, false>(cost);
}
template <int INTEG>
static plan_fleet_fn pick_plan_fleet1(int cost, int n_sub, bool philox) {
    return n_sub == 10 ? pick_plan_fleet2<INTEG, 10>(cost, philox) : pick_plan_fleet2<INTEG, 0>(cost, philox);
}
static plan_fleet_fn pick_plan_fleet(int integ, int cost, int n_sub, bool philox) {
    return integ == CPS_EULER_V0 ? pick_plan_fleet1<0>(cost, n_sub, philox) : pick_plan_fleet1<1>(cost, n_sub, philox);
}

// Dynamic shared memory of plan_fleet_kernel (cps_cem_step's layout, plus the elites' regenerated draws with Philox); sets
// a.defer_stats, a.elite_smem and a.rs_off from a.best_k and a.T.
static size_t cem_fleet_smem(const cps_handle *h, PlanArgs &a, bool philox) {
    a.defer_stats = ((long long)a.best_k * a.T > 2048) ? 1 : 0;
    a.elite_smem = a.defer_stats ? 0 : a.best_k;
    const size_t base = sizeof(float) * 4 * (size_t)a.T + sizeof(int) * (size_t)a.elite_smem +
                        ((philox && !a.defer_stats) ? sizeof(float) * (size_t)a.best_k * a.T : 0);
    return plan_smem(h, a, base, 256, 1);
}

int cps_cem_fleet_check(cps_handle *h, int best_k, float initial_stdev, float stdev_min, int philox, const char *who) {
    if (plan_check(h, who) != CPS_OK) return CPS_ERR_UNSUPPORTED;   // the message plan_check left stands
    const int K = h->cfg.num_rollouts;
    if (K > CPS_CEM_MULTIBLOCK_MIN)
        return fail(h, CPS_ERR_UNSUPPORTED, "%s: at most %d plans (the multi-block selection is not built for fleets)", who,
                    CPS_CEM_MULTIBLOCK_MIN);
    if (best_k < 1 || best_k > K) return fail(h, CPS_ERR_INVALID, "%s: cem_best_k must lie in [1, num_rollouts]", who);
    if (!(initial_stdev >= 0.0f) || !(stdev_min >= 0.0f)) return fail(h, CPS_ERR_INVALID, "%s: negative stdev", who);
    PlanArgs a;
    memset(&a, 0, sizeof(a));
    a.best_k = best_k; a.T = h->cfg.horizon;
    if (cem_fleet_smem(h, a, philox != 0) > 200 * 1024)
        return fail(h, CPS_ERR_UNSUPPORTED, "%s: horizon too large for shared memory", who);
    return CPS_OK;
}

int cps_cem_fleet_iteration(cps_handle *h, const CemFleetIteration &c) {
    const int K = h->cfg.num_rollouts, T = h->cfg.horizon;
    const bool philox = c.eps == nullptr;
    PlanArgs a;
    plan_common(h, a, nullptr, 0.0f, K, T);
    a.Q = c.eps; a.qs_k = 1; a.qs_t = K;
    a.Q_out = c.Q_out;
    a.J = c.J;
    a.select = SELECT_CEM;
    a.best_k = c.best_k; a.sd_min = c.sd_min; a.sd_init = c.sd_init;
    a.mid = (a.lo + a.hi) * 0.5f;
    a.last_iter = c.last_iter;
    a.ticket = c.tickets; a.elite = c.elite; a.u_out = c.u;
    a.mu = c.mu; a.sd = c.sd; a.mu_out = c.mu_out; a.sd_out = c.sd_out;
    const size_t smem = cem_fleet_smem(h, a, philox);
    PlanFleetExt fx;
    memset(&fx, 0, sizeof(fx));
    fx.s = c.s; fx.tp = c.tp; fx.te = c.te;
    fx.cost_up = c.cost_up; fx.cost_dn = c.cost_dn;
    fx.seed = c.seed; fx.w1 = c.w1; fx.period = c.period; fx.e_offset = c.e_offset;
    plan_fleet_fn fn = pick_plan_fleet(h->cfg.integrator, h->cfg.cost_id, h->ode.n, philox);
    if (!fn) return fail(h, CPS_ERR_UNSUPPORTED, "cps_cem_fleet_step: no kernel for this configuration");
    if (smem > 48 * 1024) CUDA_TRY(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fn<<<dim3((unsigned)(K + 255) / 256, (unsigned)c.E), 256, smem, h->stream>>>(a, fx);
    h->launches += 1;
    if (a.defer_stats) {
        if (philox) cem_update_fleet_kernel<true><<<dim3((unsigned)T, (unsigned)c.E), 256, 0, h->stream>>>(a, fx);
        else cem_update_fleet_kernel<false><<<dim3((unsigned)T, (unsigned)c.E), 256, 0, h->stream>>>(a, fx);
        h->launches += 1;
    }
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}
