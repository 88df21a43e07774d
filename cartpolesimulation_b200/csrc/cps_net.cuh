// cps_net.cuh -- declarations shared by the two neural-predictor translation units (cps_net.cu: FP32 CUDA-core
// kernel + host side; cps_net_tc.cu: tcgen05 tensor-core kernel).
#pragma once
#include "cps_internal.cuh"

#define NET_RT 8            // rollouts per compute thread

typedef unsigned long long u64;

struct NetDev {
    int type, n_layers, n_in, n_state_in, n_out, htot, n_weights;
    int hsz[CPS_NET_MAX_LAYERS];
    int hoff[CPS_NET_MAX_LAYERS];   // offset of layer l inside the concatenated hidden state
    int in_idx[6], out_idx[6];
    float norm_a[7], norm_b[7], denorm_A[6], denorm_B[6];
    int differential;
    float p1[6], p2[6], on_a[6], on_b[6];
    int out_to_in[6];
    int has_angle, has_sin, has_cos;   // which of these the network outputs (the others are augmented)
    // offsets (in floats) into the device weight buffer
    int off_wih[CPS_NET_MAX_LAYERS], off_whh[CPS_NET_MAX_LAYERS], off_bih[CPS_NET_MAX_LAYERS], off_bhh[CPS_NET_MAX_LAYERS];
    int off_wout, off_bout;
};

struct NetState {
    NetDev dev;
    float *d_weights;   // device layout: per layer W_ih^T [in][G*H], W_hh^T [H][3H], b_ih, b_hh; W_out^T [H][n_out], b_out
    float *d_href;      // stored hidden state [htot] (memory_states_ref; rows are identical across the batch)
    int ht;             // common hidden size if the kernels have a specialisation for it (64, 32), else 0
    unsigned char *d_tc;  // tensor-core kernel image (fp16 hi/lo weights in UMMA core-matrix order + epilogue constants), or null
    float *d_gws;         // net_grad_kernel's records of the forward pass (cps_net_grad.cu), grown on demand
    size_t gws_bytes;
};

struct NetArgs {
    NetDev net;
    const float *weights;
    const unsigned char *tc;  // tensor-core image (net_tc_kernel)
    const float *s0;
    long long ss_b;
    const float *Q;           // plain rollouts: controls
    long long qs_b, qs_t;
    int B, T;
    const float *h0;
    long long hs_b;           // 0: one shared hidden state, htot: per rollout
    float *traj_out;
    long long ts_k, ts_t, ts_c;
    float *h_final;           // [B][htot] or null
    // MPPI mode
    int cost_id;
    CostParams cost;
    MppiParams mp;
    const float *noise;
    long long ns_i, ns_k;
    float u_prev;
    float *u_nom, *u_out, *J_out, *u_run_out, *partials;
    unsigned *ticket;
    int *nonfinite;
    float *shard_out;
    PeerExchange px;          // K sharded over GPUs, exchange inside the launch (cps_mppi_set_peers)
    float *h_ref;             // stored hidden state to advance after the solve (null: skip)
    int tc_rows;              // net_tc_kernel: live rollouts per CTA (32 | 64: the first 8 | 16 lanes of each tensor-memory lane quarter | 128)
};

// The MPPI fleet's per-experiment inputs (net_kernel / net_tc_kernel with FLEET = true; unused otherwise).  Grid
// (tiles, E): CTA (x, e = blockIdx.y) holds rollouts of experiment e only, and the experiment's gridDim.x tiles merge as the
// tiles of one cps_mppi_step do.  With FLEET, NetArgs' B is the rollouts per experiment K, noise the draws [E][n_ind][K]
// (ns_i = K, ns_k = 1), partials [E][gridDim.x][2 + n_red] and J_out [E][K] or null; s0, h0, u_nom, u_prev, u_out, cost,
// ticket and h_ref are taken from here instead.
struct NetFleetMppiExt {
    const float *s;               // [E][8] states
    float *u_nom;                 // [E][T] warm starts
    float *u_prev;                // [E] last controls; the solve's u replaces them (optimizer_mppi.py:210)
    float *h;                     // [E][htot] hidden states: the rollouts' h0, advanced on (u, s) by the experiment's last CTA
    const float *tp, *te;         // [E] targets of this period (null: 0 / +1)
    CostParams cost_up, cost_dn;  // folded for target_equilibrium = +1 / -1
    unsigned *tickets;            // [E]
};

// The experiment's cost parameters, as fleet_kernel selects them; staged once per CTA in shared memory.
__device__ __forceinline__ void fleet_cost_stage(const NetFleetMppiExt &fx, int e, CostParams *dst) {
    const float tp = fx.tp ? fx.tp[e] : 0.0f, te = fx.te ? fx.te[e] : 1.0f;
    CostParams c = (te == 1.0f) ? fx.cost_up : fx.cost_dn;
    c.target_position = tp;
    c.target_equilibrium = te;
    *dst = c;
}

// ---- small device helpers ---------------------------------------------------------------------------------------
__device__ __forceinline__ float sigmoid_f(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
// 1 - 2/(1 + e^{2x}): absolute error ~1e-7, saturates correctly for large |x|
__device__ __forceinline__ float tanh_f(float x) { return 1.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * x)); }

__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

// Packed FP32 pairs (Blackwell FFMA2: two IEEE fp32 FMAs per issue slot; same results as two fmaf).
__device__ __forceinline__ u64 pack2(float lo, float hi) {
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(u64 v, float &lo, float &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ u64 ffma2(u64 a, u64 b, u64 c) {
    u64 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}

// de-normalise, scatter into the 6-vector state, augment (predictors_customization.py:120-139)
__device__ __forceinline__ void compose_state(const NetDev &N, const float (&y)[6], float (&st)[6]) {
#pragma unroll
    for (int c = 0; c < 6; ++c) st[c] = 0.0f;
#pragma unroll
    for (int o = 0; o < 6; ++o) {
        if (o < N.n_out) {
            const float v = fmaf(N.denorm_A[o], y[o], N.denorm_B[o]);
            const int c = N.out_idx[o];
#pragma unroll
            for (int cc = 0; cc < 6; ++cc)
                if (cc == c) st[cc] = v;
        }
    }
    if (!N.has_angle && N.has_sin && N.has_cos) st[IDX_ANGLE] = atan2f(st[IDX_SIN], st[IDX_COS]);
    if (N.has_angle && !N.has_sin) st[IDX_SIN] = sinf(st[IDX_ANGLE]);
    if (N.has_angle && !N.has_cos) st[IDX_COS] = cosf(st[IDX_ANGLE]);
}

__device__ __forceinline__ float stage_cost_rt(int id, const CostParams &C, float ca, float w, float x, float u, float up) {
    switch (id) {
    case CPS_COST_DEFAULT: return stage_cost<COST_DEFAULT>(C, ca, w, x, u, up) - C.max_cost;  // get_stage_cost shift (:63-64)
    case CPS_COST_QUADRATIC_BOUNDARY: return stage_cost<COST_QB>(C, ca, w, x, u, up) - C.max_cost;
    case CPS_COST_QB_GRAD_MINIMAL: return stage_cost<COST_GRADMIN>(C, ca, w, x, u, up);
    case CPS_COST_QB_GRAD: return stage_cost<COST_GRAD>(C, ca, w, x, u, up);
    default: return 0.0f;
    }
}

