// cps_net_grad.cu -- cost and gradient of predict_and_cost with the autoregressive neural predictor (GRU / Dense).
//
// The reference's RPGD (Control_Toolkit/Optimizers/optimizer_rpgd_tf.py:167-175) takes d(traj_cost)/dQ with a GradientTape
// around predictor.predict_core + cost_function.get_trajectory_cost; with predictor_autoregressive_neural
// (SI_Toolkit/Predictors/predictor_autoregressive_neural.py:266-313) the tape holds T steps of the torch Sequence
// (Functions/Pytorch/Network.py:239-287), the normalised-output feedback (Predictors/autoregression.py:94-98), the
// de-normalisation and angle augmentation (predictors_customization.py:120-139) and the cost plugin.
//
// net_grad_kernel<R, HT, GRAD>: one CTA takes a tile of R (16 | 32) plans, with the tiling of net_kernel (cps_net.cu): all
// FP32 weights resident in shared memory (one bulk copy), R/4 compute warps, one row warp; plans are independent, so the
// CTA runs the forward pass over the horizon for its tile and then sweeps back over the same tile -- one launch, no
// grid-wide synchronisation.
//   forward  the device code of net_kernel (compute_step, out_layer_row, compose_state, stage_cost_rt): cps_net_rollout's
//            trajectory bit for bit, J = sum of the T stage costs / (T + 1) (the plugins' terminal cost is zero).  GRAD
//            keeps, per CTA and plans contiguous, each step's hidden states h_l(t) and network input x(t) and output y(t)
//            in a handle-owned workspace; the gates are recomputed in the reverse sweep rather than stored;
//   reverse  t = T-1 .. 0, the adjoint of exactly the forward arithmetic: the output y(t) receives adjoint from the next
//            step's input (the normalised output IS the next normalised input) and from the stage cost of step t+1
//            through de-normalisation, scatter and atan2(sin, cos) (cps_grad_partials.cuh: the same partials as the ODE
//            adjoint); then W_out^T, and per layer top-down the GRU cell (gate adjoints from recomputed gates, then W_hh^T
//            and W_ih^T products) or the tanh Dense layer; dJ/du_t = norm_a[0] dx(t)[0] + the plugin's direct control
//            terms.  No gradient flows into s0 or the stored hidden state h0, which these calls read and never write.
// Transposed products: the weights stay in net_kernel's [in][G*H] layout (the forward reads it conflict-free, lanes =
// consecutive output units).  W^T delta needs lanes = consecutive INPUT units, i.e. a stride of G*H words, which is a
// multiple of 32 for the 32 / 64-unit GRUs: every lane would hit the same bank.  Lane i therefore walks the columns
// starting at column i (c = (i + k) mod G*H): bank (i*G*H + i + k) mod 32 = (i + k) mod 32, conflict-free with no second,
// transposed copy of the weights (the 2 x 64 GRU image is 156 KB of the 227 KB).  The gate adjoints are kept [unit][R + 4]:
// the padding makes the 16-byte loads of eight consecutive units fall on distinct banks.
// FP32 on CUDA cores (FFMA2), no tensor cores: the shipped RPGD size is 16 plans, and the gradient wants fp32 accuracy.
//
// net_grad_kernel<R, HT, GRAD, FLEET = true> (cps_rpgd_fleet.cu): the plans of E experiments in one launch.  The tiles are
// laid per experiment (grid = E x ceil(K / R), R chosen from the per-experiment K as the single-experiment call chooses it),
// so every CTA holds plans of one experiment only and runs, per plan, exactly the arithmetic of cps_plan_cost_grad /
// cps_plan_cost for that experiment alone.  CTA b takes experiment e = b / ceil(K / R): its state s + 8 e, u_prev[e] and
// folded cost parameters costs[e]; Q, G [E][K][T] and J [E][K] are indexed by the global plan e K + k.  The weights and the
// stored hidden state h0 are shared and read-only.  FLEET = false compiles to the code it compiled to before FLEET existed.
#include <cuda_runtime.h>

#include <cmath>
#include <cstring>

#include "cps_grad_partials.cuh"
#include "cps_net_fp32.cuh"

struct NetGradArgs {
    NetDev net;
    const float *weights;
    const float *s;             // [6], shared by all plans
    const float *Q;
    long long qs_k, qs_t;
    int K, T, hmax;
    const float *h0;            // [htot]: the stored hidden state, shared by all plans
    int cost_id;
    CostParams cost;
    float u_prev, inv_T1;
    float *J;                   // [K]
    float *G;                   // gradient, layout of Q
    long long gs_k, gs_t;
    float *traj;                // optional trajectories
    long long ts_k, ts_t, ts_c;
    float *ws;                  // GRAD: per CTA [T+1][htot][R] hidden states, [T][8][R] inputs, [T][8][R] outputs
    long long ws_cta;           // floats per CTA
    int *nonfinite;
};

// FLEET's per-experiment inputs (unused otherwise): CTA b holds plans of experiment b / tiles.  With FLEET, NetGradArgs' K
// is the number of plans per experiment, s the fleet's states [E][8], Q and G [E][K][T], J [E][K].
struct NetFleetExt {
    const CostParams *costs;    // [E] folded for each experiment's targets of the period
    const float *u_prev;        // [E]
    int tiles;                  // CTAs per experiment, ceil(K / R)
};

namespace {

// acc[.] += sum_k W[i][c] d[c][g*8 .. g*8+8) over the ncol columns c of row i of a [in][ncol] weight image, starting at
// column c0 = i mod ncol (lane-rotated: conflict-free for ncol a multiple of 32).  Gate adjoint row of column c:
// c + (c >= split ? shift : 0).
template <int R>
__device__ __forceinline__ void tmatvec_acc2(const float *__restrict__ w, const float *__restrict__ d, int ncol, int c0, int split,
                                             int shift, int g, u64 (&acc)[4]) {
    constexpr int RP = R + 4;
    int c = c0;
#pragma unroll 4
    for (int k = 0; k < ncol; ++k) {
        const float wv = w[c];
        const float *dr = d + (c + (c >= split ? shift : 0)) * RP + g * NET_RT;
        const ulonglong2 d0 = *reinterpret_cast<const ulonglong2 *>(dr);
        const ulonglong2 d1 = *reinterpret_cast<const ulonglong2 *>(dr + 4);
        const u64 ww = pack2(wv, wv);
        acc[0] = ffma2(ww, d0.x, acc[0]);
        acc[1] = ffma2(ww, d0.y, acc[1]);
        acc[2] = ffma2(ww, d1.x, acc[2]);
        acc[3] = ffma2(ww, d1.y, acc[3]);
        if (++c == ncol) c = 0;
    }
}

__device__ __forceinline__ void load8(const float *p, u64 (&a)[4]) {
    const ulonglong2 x0 = *reinterpret_cast<const ulonglong2 *>(p), x1 = *reinterpret_cast<const ulonglong2 *>(p + 4);
    a[0] = x0.x; a[1] = x0.y; a[2] = x1.x; a[3] = x1.y;
}
__device__ __forceinline__ void store8(float *p, const u64 (&a)[4]) {
    *reinterpret_cast<ulonglong2 *>(p) = make_ulonglong2(a[0], a[1]);
    *reinterpret_cast<ulonglong2 *>(p + 4) = make_ulonglong2(a[2], a[3]);
}
__device__ __forceinline__ void store8f(float *p, const float (&v)[NET_RT]) {
    *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4 *>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void copy4(float *dst, const float *src, int n, int tid, int nt) {
    for (int i = 4 * tid; i < n; i += 4 * nt) *reinterpret_cast<float4 *>(dst + i) = *reinterpret_cast<const float4 *>(src + i);
}

template <int R, int HT, bool GRAD, bool FLEET>
__global__ void __launch_bounds__(R * 8 + 32, 1) net_grad_kernel(const __grid_constant__ NetGradArgs a,
                                                                 const __grid_constant__ NetFleetExt fx) {
    constexpr int NC = R * 8, NT = NC + 32, RP = R + 4, G8 = R / NET_RT;
    extern __shared__ __align__(16) float smem[];
    __shared__ __align__(8) unsigned long long s_bar;
    const NetDev &N = a.net;
    const int tid = threadIdx.x, lane = tid & 31;
    const bool row_warp = tid >= NC;
    const int T = a.T;
    const bool gru = N.type == CPS_NET_GRU;
    // FLEET: the CTA's experiment and its per-experiment inputs (read where the single-experiment call reads its own)
    const int e = FLEET ? (int)blockIdx.x / fx.tiles : 0;
    const CostParams &C = FLEET ? fx.costs[e] : a.cost;

    // ---- shared-memory carve-up (net_kernel's, then the adjoints) --------------------------------------------------
    float *wsm = smem;                              // [n_weights]
    float *hb = wsm + N.n_weights;                  // [2][htot][R]
    const int hstride = N.htot * R;
    float *xin = hb + 2 * hstride;                  // [8][R]
    float *dH = xin + 8 * R;                        // GRAD: [htot][R] adjoint of each layer's output of the step
    float *dA = dH + hstride;                       // GRAD: [4 hmax][R + 4] gate adjoints (r | z | n r | n) or Dense's
    float *dY = dA + 4 * a.hmax * RP;               // GRAD: [8][R] adjoint of the network output
    float *dX = dY + 8 * R;                         // GRAD: [8][R] adjoint of the network input
    float *wsH = a.ws + (long long)blockIdx.x * a.ws_cta;   // GRAD: [T+1][htot][R]
    float *wsX = wsH + (long long)(T + 1) * hstride;        // GRAD: [T][8][R]
    float *wsY = wsX + (long long)T * 8 * R;                // GRAD: [T][8][R]

    if (tid == 0) weights_copy_start(&s_bar, wsm, a.weights, N.n_weights);
    if (gru) {
        for (int idx = tid; idx < hstride; idx += NT) {
            const float v = a.h0[idx / R];
            hb[idx] = v;
            if (GRAD) wsH[idx] = v;
        }
    }
    __syncthreads();  // also publishes the mbarrier init

    const unsigned tile = FLEET ? blockIdx.x - (unsigned)(e * fx.tiles) : blockIdx.x;
    const long long pbase = FLEET ? (long long)e * a.K : 0;   // the experiment's first plan
    const int r_row = lane % R;
    const bool row_lead = row_warp && lane < R;
    const int k = tile * R + r_row;
    const bool active = row_lead && k < a.K;
    const int kc = min(k, a.K - 1);
    const float *qrow = a.Q + (pbase + kc) * a.qs_k;
    float *traj = (a.traj && active) ? a.traj + (long long)k * a.ts_k : nullptr;
    float Jacc = 0.0f, up = FLEET ? fx.u_prev[e] : a.u_prev, u_cur = 0.0f, u_nxt = row_warp ? qrow[0] : 0.0f;
    weights_copy_wait(&s_bar);
    __syncthreads();

    // ---- forward: net_kernel's horizon loop without the MPPI terms ---------------------------------------------------
    int p = 0;
    float st[6], y[6];
    const float *hlast_base = hb + N.hoff[N.n_layers - 1] * R;
#pragma unroll 1
    for (int t = 0; t < T; ++t) {
        if (row_warp) {
            if (t == 0) {
#pragma unroll
                for (int c = 0; c < 6; ++c) st[c] = (FLEET ? a.s + (long long)e * 8 : a.s)[c];
                if (row_lead)
                    for (int i = 0; i < N.n_state_in; ++i) xin[(1 + i) * R + r_row] = fmaf(N.norm_a[1 + i], (FLEET ? a.s + (long long)e * 8 : a.s)[N.in_idx[i]], N.norm_b[1 + i]);
            } else {
                out_layer_row<R>(N, wsm, hlast_base + (gru ? p * hstride : 0), lane, y);
                if (row_lead) {
#pragma unroll
                    for (int o = 0; o < 6; ++o) {
                        if (o < N.n_state_in) xin[(1 + o) * R + r_row] = y[o];
                        if (GRAD && o < N.n_out) wsY[((long long)(t - 1) * 8 + o) * R + r_row] = y[o];
                    }
                }
            }
            u_cur = u_nxt;
            if (row_lead) {
                xin[r_row] = fmaf(N.norm_a[0], u_cur, N.norm_b[0]);
                if (GRAD)
                    for (int i = 0; i < N.n_in; ++i) wsX[((long long)t * 8 + i) * R + r_row] = xin[i * R + r_row];
            }
            cta_sync();
            if (t > 0) compose_state(N, y, st);
            if (traj) {
#pragma unroll
                for (int c = 0; c < 6; ++c) traj[(long long)t * a.ts_t + c * a.ts_c] = st[c];
            }
            Jacc += stage_cost_rt(a.cost_id, C, cosf(st[IDX_ANGLE]), st[IDX_ANGLED], st[IDX_POS], u_cur, up);
            up = u_cur;
            if (t + 1 < T) u_nxt = qrow[(long long)(t + 1) * a.qs_t];
            for (int l = 0; l < N.n_layers; ++l) cta_sync();
        } else {
            compute_step<R, HT>(N, wsm, hb, hstride, p, xin, tid);
            if (GRAD) copy4(wsH + (long long)(t + 1) * hstride, hb + (gru ? (1 - p) * hstride : 0), hstride, tid, NC);
        }
        p ^= 1;
    }
    if (row_warp) {
        out_layer_row<R>(N, wsm, hlast_base + (gru ? p * hstride : 0), lane, y);
        compose_state(N, y, st);
        if (traj) {
#pragma unroll
            for (int c = 0; c < 6; ++c) traj[(long long)T * a.ts_t + c * a.ts_c] = st[c];
        }
        const float J = __fdiv_rn(Jacc, (float)(T + 1));   // mean over the T + 1 entries (true division, as torch.mean)
        if (active) {
            a.J[pbase + k] = J;
            if (!isfinite(J)) atomicAdd(a.nonfinite, 1);
        }
    }
    if (!GRAD) return;

    // ---- reverse sweep ---------------------------------------------------------------------------------------------
    __syncthreads();   // the workspace records of the whole tile are written
    for (int idx = tid; idx < hstride; idx += NT) dH[idx] = 0.0f;
    copy4(hb + (T & 1) * hstride, wsH + (long long)T * hstride, hstride, tid, NT);
    const bool full = a.cost_id == CPS_COST_QB_GRAD;
    const bool atan2_angle = !N.has_angle && N.has_sin && N.has_cos;
    float fb[6] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};   // row warp: adjoint of x(t+1)'s state features
#pragma unroll 1
    for (int t = T - 1; t >= 0; --t) {
        float *hA = hb + (t & 1) * hstride;             // h(t): the layers' input hidden states of step t
        const float *hB = hb + ((t + 1) & 1) * hstride; // h(t+1) (GRU) / the activations of step t (Dense)
        if (gru || t > 0) copy4(hA, wsH + (long long)t * hstride, hstride, tid, NT);
        copy4(xin, wsX + (long long)t * 8 * R, N.n_in * R, tid, NT);
        // (1) row warp: adjoint of y(t) -- the next step's input and the stage cost of step t+1
        if (row_lead) {
            float dy[6];
#pragma unroll
            for (int o = 0; o < 6; ++o) dy[o] = (o < N.n_state_in) ? fb[o] : 0.0f;
            if (t + 1 < T) {
                float yv[6];
#pragma unroll
                for (int o = 0; o < 6; ++o) yv[o] = (o < N.n_out) ? wsY[((long long)t * 8 + o) * R + r_row] : 0.0f;
                compose_state(N, yv, st);
                float d_th, d_w, d_x;
                if (full) grad_partials(C, st[IDX_ANGLE], st[IDX_ANGLED], st[IDX_POS], d_th, d_w, d_x);
                else gradmin_partials(C, st[IDX_ANGLE], st[IDX_ANGLED], st[IDX_POS], d_th, d_w, d_x);
                d_th *= a.inv_T1; d_w *= a.inv_T1; d_x *= a.inv_T1;
                float d_sin = 0.0f, d_cos = 0.0f;
                if (atan2_angle) {   // angle = atan2(sin, cos)
                    const float sn = st[IDX_SIN], cs = st[IDX_COS], ir2 = 1.0f / fmaf(sn, sn, cs * cs);
                    d_sin = d_th * cs * ir2;
                    d_cos = -d_th * sn * ir2;
                }
#pragma unroll
                for (int o = 0; o < 6; ++o) {
                    if (o < N.n_out) {
                        const int c = N.out_idx[o];
                        const float dv = (c == IDX_ANGLE) ? d_th : (c == IDX_ANGLED) ? d_w : (c == IDX_POS) ? d_x
                                       : (c == IDX_SIN) ? d_sin : (c == IDX_COS) ? d_cos : 0.0f;
                        dy[o] = fmaf(N.denorm_A[o], dv, dy[o]);
                    }
                }
            }
#pragma unroll
            for (int o = 0; o < 6; ++o)
                if (o < N.n_out) dY[o * R + r_row] = dy[o];
        }
        __syncthreads();
        // (2) output layer: the last layer's adjoint += W_out^T dy (Dense: =, nothing carries over from step t+1)
        if (!row_warp) {
            const int L1 = N.n_layers - 1, H = HT ? HT : N.hsz[L1];
            const float *Wo = wsm + N.off_wout;
            for (int item = tid; item < G8 * H; item += NC) {
                const int j = item % H, g = item / H;
                float *d = dH + (N.hoff[L1] + j) * R + g * NET_RT;
                float acc[NET_RT];
#pragma unroll
                for (int e = 0; e < NET_RT; ++e) acc[e] = gru ? d[e] : 0.0f;
                for (int o = 0; o < N.n_out; ++o) {
                    const float w = Wo[j * N.n_out + o];
#pragma unroll
                    for (int e = 0; e < NET_RT; ++e) acc[e] = fmaf(w, dY[o * R + g * NET_RT + e], acc[e]);
                }
                store8f(d, acc);
            }
        }
        __syncthreads();
        // (3) the hidden layers, top down
        for (int l = N.n_layers - 1; l >= 0; --l) {
            const int H = HT ? HT : N.hsz[l];
            const int in_len = l ? (HT ? HT : N.hsz[l - 1]) : N.n_in;
            const float *in = l ? hB + N.hoff[l - 1] * R : xin;
            float *dHl = dH + N.hoff[l] * R;
            float *dIn = l ? dH + N.hoff[l - 1] * R : dX;
            if (!row_warp) {
                for (int item = tid; item < G8 * H; item += NC) {
                    const int j = item % H, g = item / H;
                    float *dh = dHl + j * R + g * NET_RT;
                    float o0[NET_RT], o1[NET_RT], o2[NET_RT], o3[NET_RT];
                    if (gru) {
                        // the gates of step t, recomputed with the forward's code and inputs
                        u64 acc[3][4], ai[3][4];
                        gru_hh<R, HT>(N, wsm, l, hA + N.hoff[l] * R, j, g, acc);
                        gru_ih_acc<R, HT>(N, wsm, l, in, in_len, j, g, acc, ai);
                        const float *hp = hA + (N.hoff[l] + j) * R + g * NET_RT;
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            float ar[2], az[2], an[2], gn[2];
                            unpack2(ai[0][q], ar[0], ar[1]); unpack2(ai[1][q], az[0], az[1]);
                            unpack2(ai[2][q], an[0], an[1]); unpack2(acc[2][q], gn[0], gn[1]);
#pragma unroll
                            for (int h2 = 0; h2 < 2; ++h2) {
                                const int e = 2 * q + h2;
                                const float r = sigmoid_f(ar[h2]), z = sigmoid_f(az[h2]);
                                const float n = tanh_f(fmaf(r, gn[h2], an[h2]));
                                const float dhp = dh[e];
                                const float dan = dhp * (1.0f - z) * (1.0f - n * n);
                                o0[e] = dan * gn[h2] * r * (1.0f - r);             // a_r
                                o1[e] = dhp * (hp[e] - n) * z * (1.0f - z);        // a_z
                                o2[e] = dan * r;                                   // W_hn h + b_hn
                                o3[e] = dan;                                       // a_n (input part)
                                dh[e] = dhp * z;                                   // direct path of h' = (h - n) z + n
                            }
                        }
                        store8f(dA + j * RP + g * NET_RT, o0);
                        store8f(dA + (H + j) * RP + g * NET_RT, o1);
                        store8f(dA + (2 * H + j) * RP + g * NET_RT, o2);
                        store8f(dA + (3 * H + j) * RP + g * NET_RT, o3);
                    } else {
                        const float *act = hB + (N.hoff[l] + j) * R + g * NET_RT;
#pragma unroll
                        for (int e = 0; e < NET_RT; ++e) o0[e] = dh[e] * (1.0f - act[e] * act[e]);   // a = tanh(.)
                        store8f(dA + j * RP + g * NET_RT, o0);
                    }
                }
            }
            __syncthreads();
            if (!row_warp) {
                const int NG = gru ? 3 : 1;
                if (gru) {   // adjoint of h_l(t): dh' z + W_hh^T (a_r, a_z, a_n r)
                    for (int item = tid; item < G8 * H; item += NC) {
                        const int i = item % H, g = item / H;
                        u64 acc[4];
                        load8(dHl + i * R + g * NET_RT, acc);
                        tmatvec_acc2<R>(wsm + N.off_whh[l] + i * 3 * H, dA, 3 * H, i % (3 * H), 3 * H, 0, g, acc);
                        store8(dHl + i * R + g * NET_RT, acc);
                    }
                }
                // adjoint of the layer's input: W_ih^T (a_r, a_z, a_n); the layer below accumulates it on top of its
                // recurrent adjoint (GRU), the network input / a Dense layer's activation takes it as is
                for (int item = tid; item < G8 * in_len; item += NC) {
                    const int i = item % in_len, g = item / in_len;
                    float *d = dIn + i * R + g * NET_RT;
                    u64 acc[4];
                    if (l && gru) load8(d, acc);
                    else acc[0] = acc[1] = acc[2] = acc[3] = 0ull;
                    tmatvec_acc2<R>(wsm + N.off_wih[l] + i * NG * H, dA, NG * H, i % (NG * H), 2 * H, H, g, acc);
                    store8(d, acc);
                }
            }
            __syncthreads();
        }
        // (4) row warp: dJ/du_t = norm_a[0] dx(t)[0] + the plugin's direct control terms
        if (row_lead) {
#pragma unroll
            for (int o = 0; o < 6; ++o) fb[o] = (o < N.n_state_in) ? dX[(1 + o) * R + r_row] : 0.0f;
            const float u = qrow[(long long)t * a.qs_t];
            float du;
            if (full) {   // cc u_t^2 + ccrc (u_t - u_{t-1})^2 of this stage and ccrc (u_{t+1} - u_t)^2 of the next
                const float upv = (t > 0) ? qrow[(long long)(t - 1) * a.qs_t] : (FLEET ? fx.u_prev[e] : a.u_prev);
                du = 2.0f * C.w[5] * u + 2.0f * C.w[6] * (u - upv);
                if (t + 1 < T) du -= 2.0f * C.w[6] * (qrow[(long long)(t + 1) * a.qs_t] - u);
            } else {
                du = 2.0f * C.w[4] * u;
            }
            if (active) a.G[(pbase + k) * a.gs_k + (long long)t * a.gs_t] = fmaf(N.norm_a[0], dX[r_row], a.inv_T1 * du);
        }
    }
}

typedef void (*net_grad_fn)(const NetGradArgs, const NetFleetExt);

template <int R, bool GRAD, bool FLEET>
net_grad_fn pick2(int ht) {
    switch (ht) {
    case 64: return net_grad_kernel<R, 64, GRAD, FLEET>;
    case 32: return net_grad_kernel<R, 32, GRAD, FLEET>;
    default: return net_grad_kernel<R, 0, GRAD, FLEET>;
    }
}
template <bool FLEET>
net_grad_fn pick(int R, int ht, bool grad) {
    if (R == 32) return grad ? pick2<32, true, FLEET>(ht) : pick2<32, false, FLEET>(ht);
    return grad ? pick2<16, true, FLEET>(ht) : pick2<16, false, FLEET>(ht);
}

int hidden_max(const NetDev &N) {
    int m = 0;
    for (int l = 0; l < N.n_layers; ++l) m = N.hsz[l] > m ? N.hsz[l] : m;
    return m;
}

size_t smem_bytes(const NetDev &N, int R, bool grad) {
    size_t f = (size_t)N.n_weights + 2 * (size_t)N.htot * R + 8 * (size_t)R;
    if (grad) f += (size_t)N.htot * R + 4 * (size_t)hidden_max(N) * (R + 4) + 16 * (size_t)R;
    return f * sizeof(float);
}

// The configurations these calls cover (else an error that names what is missing)
int check(cps_handle *h, const char *who, bool grad) {
    if (!h->net) return fail(h, CPS_ERR_NOT_CONFIGURED, "%s: neural predictor without a network (cps_net_load)", who);
    const NetDev &N = h->net->dev;
    if (N.differential)
        return fail(h, CPS_ERR_UNSUPPORTED, "%s: differential (D_*) networks are not supported with the neural predictor", who);
    if (h->cfg.cost_id == CPS_COST_NONE || h->cfg.cost_id == CPS_COST_LEGACY_MPPI)
        return fail(h, CPS_ERR_NOT_CONFIGURED, "%s: the handle has no cost-function plugin", who);
    if (h->cfg.cost_id != CPS_COST_QB_GRAD_MINIMAL && h->cfg.cost_id != CPS_COST_QB_GRAD)
        return fail(h, CPS_ERR_UNSUPPORTED, "%s: with the neural predictor only the quadratic_boundary_grad_minimal and "
                    "quadratic_boundary_grad plugins are supported", who);
    if (h->cfg.flags & CPS_FLAG_NET_TENSOR_CORES)
        return fail(h, CPS_ERR_UNSUPPORTED, "%s: CPS_FLAG_NET_TENSOR_CORES forces the tensor-core kernel, which has no cost or "
                    "gradient pass; create the handle without it", who);
    const size_t smem = smem_bytes(N, 16, grad);
    if (smem > 227 * 1024)
        return fail(h, CPS_ERR_UNSUPPORTED, "%s: the network needs %zu bytes of shared memory per CTA here (limit 227 KB)", who, smem);
    return CPS_OK;
}

// Small batches: 16 plans per CTA spread the work over more SMs; large ones: 32 where the gradient's buffers leave room.
// The forward-only instantiation takes the same tile, so that both compute J with the same output-layer summation
// (out_layer_row splits it over two lanes at R = 16).
int tile_rows(const NetDev &N, int K) {
    return (K > 148 * 16 && smem_bytes(N, 32, true) <= 227 * 1024) ? 32 : 16;
}

// The forward records of the gradient: floats per CTA of R plans over T steps
long long ws_floats_per_cta(const NetDev &N, int R, int T) { return (long long)(T + 1) * N.htot * R + 16LL * T * R; }

// Makes the handle's workspace hold at least `need` bytes (grown on demand; K = 2000, T = 50, 2 x 64 GRU: 53 MB)
int grow_ws(cps_handle *h, size_t need) {
    NetState *S = h->net;
    if (need > S->gws_bytes) {
        cudaFree(S->d_gws);
        S->d_gws = nullptr;
        S->gws_bytes = 0;
        CUDA_TRY(h, cudaMalloc(&S->d_gws, need));
        S->gws_bytes = need;
    }
    return CPS_OK;
}

int launch(cps_handle *h, NetGradArgs &a, bool grad) {
    NetState *S = h->net;
    const int R = tile_rows(S->dev, a.K);
    const size_t smem = smem_bytes(S->dev, R, grad);
    const int grid = (a.K + R - 1) / R;
    if (grad) {
        a.ws_cta = ws_floats_per_cta(S->dev, R, a.T);
        const int rc = grow_ws(h, sizeof(float) * (size_t)a.ws_cta * grid);
        if (rc != CPS_OK) return rc;
        a.ws = S->d_gws;
    }
    net_grad_fn fn = pick<false>(R, S->ht, grad);
    CUDA_TRY(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fn<<<grid, R * 8 + 32, smem, h->stream>>>(a, NetFleetExt());
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

void common(cps_handle *h, NetGradArgs &a, const float *s_dev, const float *Q_dev, int q_layout, int K, int T, float u_prev) {
    memset(&a, 0, sizeof(a));
    a.net = h->net->dev;
    a.weights = h->net->d_weights;
    a.s = s_dev;
    a.Q = Q_dev;
    if (q_layout == CPS_TIME_MAJOR) { a.qs_k = 1; a.qs_t = K; } else { a.qs_k = T; a.qs_t = 1; }
    a.K = K; a.T = T; a.hmax = hidden_max(h->net->dev);
    a.h0 = h->net->d_href;
    a.cost_id = h->cfg.cost_id; a.cost = h->cost;
    a.u_prev = u_prev;
    a.inv_T1 = 1.0f / (float)(T + 1);
    a.nonfinite = h->d_nonfinite;
}

}  // namespace

int cps_net_plan_cost(cps_handle *h, const float *s_dev, const float *Q_dev, int q_layout, int K, int T, float u_prev,
                      float *J_out_dev, float *traj_out_dev, int traj_layout) {
    int rc = check(h, "cps_plan_cost", false);
    if (rc != CPS_OK) return rc;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    NetGradArgs a;
    common(h, a, s_dev, Q_dev, q_layout, K, T, u_prev);
    a.J = J_out_dev;
    a.traj = traj_out_dev;
    if (traj_layout == CPS_TIME_MAJOR) { a.ts_k = 1; a.ts_t = 6LL * K; a.ts_c = K; }
    else { a.ts_k = (T + 1) * 6LL; a.ts_t = 6; a.ts_c = 1; }
    return launch(h, a, false);
}

int cps_net_plan_cost_grad(cps_handle *h, const float *s_dev, const float *Q_dev, int q_layout, float u_prev, float *J_out_dev,
                           float *G_out_dev) {
    int rc = check(h, "cps_plan_cost_grad", true);
    if (rc != CPS_OK) return rc;
    const int K = h->cfg.num_rollouts, T = h->cfg.horizon;
    NetGradArgs a;
    common(h, a, s_dev, Q_dev, q_layout, K, T, u_prev);
    a.J = J_out_dev;
    a.G = G_out_dev;
    if (q_layout == CPS_TIME_MAJOR) { a.gs_k = 1; a.gs_t = K; } else { a.gs_k = T; a.gs_t = 1; }
    return launch(h, a, true);
}

// ---- cps_rpgd_fleet.cu: the plans of E experiments in one launch -----------------------------------------------------------
int cps_net_grad_fleet_prepare(cps_handle *h, int E, const char *who) {
    int rc = check(h, who, true);
    if (rc != CPS_OK) return rc;
    const NetDev &N = h->net->dev;
    const int K = h->cfg.num_rollouts, T = h->cfg.horizon, R = tile_rows(N, K);
    return grow_ws(h, sizeof(float) * (size_t)ws_floats_per_cta(N, R, T) * (size_t)E * (size_t)((K + R - 1) / R));
}

int cps_net_grad_fleet(cps_handle *h, int E, const float *s_dev, const float *Q_dev, const CostParams *costs_dev,
                       const float *u_prev_dev, float *J_dev, float *G_dev) {
    const bool grad = G_dev != nullptr;
    int rc = check(h, "cps_rpgd_fleet_step", grad);
    if (rc != CPS_OK) return rc;
    NetState *S = h->net;
    const int K = h->cfg.num_rollouts, T = h->cfg.horizon;
    const int R = tile_rows(S->dev, K), tiles = (K + R - 1) / R;   // the tile of the single-experiment call
    NetGradArgs a;
    NetFleetExt x;
    common(h, a, s_dev, Q_dev, CPS_ROLLOUT_MAJOR, K, T, 0.0f);
    a.J = J_dev;
    a.G = G_dev;
    a.gs_k = T; a.gs_t = 1;
    x.costs = costs_dev; x.u_prev = u_prev_dev; x.tiles = tiles;
    const long long grid = (long long)E * tiles;
    if (grad) {
        a.ws_cta = ws_floats_per_cta(S->dev, R, T);
        if ((rc = grow_ws(h, sizeof(float) * (size_t)a.ws_cta * (size_t)grid)) != CPS_OK) return rc;
        a.ws = S->d_gws;
    }
    const size_t smem = smem_bytes(S->dev, R, grad);
    net_grad_fn fn = pick<true>(R, S->ht, grad);
    CUDA_TRY(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fn<<<(unsigned)grid, R * 8 + 32, smem, h->stream>>>(a, x);
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}
