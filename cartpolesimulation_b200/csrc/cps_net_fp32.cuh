// cps_net_fp32.cuh -- device code of the FP32 CUDA-core network step, shared by net_kernel (cps_net.cu: rollouts and the
// MPPI solve) and net_grad_kernel (cps_net_grad.cu: cost and gradient of predict_and_cost), so that both evaluate the
// network with the same arithmetic.
#pragma once
#include "cps_net.cuh"

// All weights global -> shared with one bulk asynchronous copy (cp.async.bulk + mbarrier), issued by one thread; every
// thread waits with weights_copy_wait after a __syncthreads() that publishes the mbarrier's initialisation.
__device__ __forceinline__ void weights_copy_start(unsigned long long *s_bar, float *wsm, const float *weights, int n_weights) {
    const unsigned bar = smem_u32(s_bar);
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const unsigned bytes = (unsigned)n_weights * 4u;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
    unsigned done = 0;
    while (done < bytes) {
        const unsigned chunk = min(bytes - done, 32768u);
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(wsm) + done), "l"(reinterpret_cast<const char *>(weights) + done), "r"(chunk),
                     "r"(bar) : "memory");
        done += chunk;
    }
}
__device__ __forceinline__ void weights_copy_wait(unsigned long long *s_bar) {
    const unsigned bar = smem_u32(s_bar);
    unsigned ok = 0;
    while (!ok) {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok) : "r"(bar) : "memory");
    }
}

// Block-wide barrier for the warp-specialised part of net_kernel, where the row warp and the compute warps reach their
// matching barriers at DIFFERENT code locations: PTX's unaligned form (barrier.sync), which -- unlike __syncthreads()'s
// barrier.sync.aligned -- does not require all threads of the block to execute the same instruction (compute-sanitizer
// --tool synccheck flags the aligned form there; profiles/r02_sanitizer.txt).
__device__ __forceinline__ void cta_sync() { asm volatile("barrier.sync 0;" ::: "memory"); }

// acc[q][.] += sum_i Wt[i][q*H + j] * x[i][g*8 .. g*8+8), rows held as 4 packed pairs.
// Wt points at column j already; ws = row stride of Wt (NG*H); x points at the thread's row group.
template <int R, int NG, int HT>
__device__ __forceinline__ void matvec_acc2(const float *__restrict__ w, const float *__restrict__ xv, int in_len, int H,
                                            u64 (&acc)[NG][4]) {
    const int Hc = HT ? HT : H;
    const int ws = NG * Hc;
#pragma unroll 8
    for (int i = 0; i < in_len; ++i) {
        const ulonglong2 x0 = *reinterpret_cast<const ulonglong2 *>(xv + i * R);
        const ulonglong2 x1 = *reinterpret_cast<const ulonglong2 *>(xv + i * R + 4);
#pragma unroll
        for (int q = 0; q < NG; ++q) {
            const float wq = w[i * ws + q * Hc];
            const u64 ww = pack2(wq, wq);
            acc[q][0] = ffma2(ww, x0.x, acc[q][0]);
            acc[q][1] = ffma2(ww, x0.y, acc[q][1]);
            acc[q][2] = ffma2(ww, x1.x, acc[q][2]);
            acc[q][3] = ffma2(ww, x1.y, acc[q][3]);
        }
    }
}

// torch.nn.GRUCell (gate order r, z, n): r = s(W_ir x + b_ir + W_hr h + b_hr), z likewise,
// n = tanh(W_in x + b_in + r (W_hn h + b_hn)), h' = (h - n) z + n.
// The pre-activations of one hidden unit for 8 rollouts: acc[0] = r, acc[1] = z (both products summed), acc[2] = the
// hidden part of n; the input part of n is added by gru_ih_finish.
template <int R, int HT>
__device__ __forceinline__ void gru_hh(const NetDev &N, const float *W, int l, const float *hprev, int j, int g,
                                       u64 (&acc)[3][4]) {
    const int H = HT ? HT : N.hsz[l];
    const float *bih = W + N.off_bih[l], *bhh = W + N.off_bhh[l];
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        const float b = (q < 2) ? bih[q * H + j] + bhh[q * H + j] : bhh[q * H + j];
        const u64 bb = pack2(b, b);
#pragma unroll
        for (int r = 0; r < 4; ++r) acc[q][r] = bb;
    }
    matvec_acc2<R, 3, HT>(W + N.off_whh[l] + j, hprev + g * NET_RT, H, H, acc);
}

// The input products on top of gru_hh's: ai[0] = a_r, ai[1] = a_z (complete pre-activations), ai[2] = W_in x + b_in.
template <int R, int HT>
__device__ __forceinline__ void gru_ih_acc(const NetDev &N, const float *W, int l, const float *xin, int in_len, int j, int g,
                                           const u64 (&acc)[3][4], u64 (&ai)[3][4]) {
    const int H = HT ? HT : N.hsz[l];
    const float *Wih = W + N.off_wih[l] + j, *bih = W + N.off_bih[l];
    const float bn = bih[2 * H + j];
#pragma unroll
    for (int r = 0; r < 4; ++r) { ai[0][r] = acc[0][r]; ai[1][r] = acc[1][r]; ai[2][r] = pack2(bn, bn); }
    matvec_acc2<R, 3, HT>(Wih, xin + g * NET_RT, in_len, H, ai);
}

template <int R, int HT>
__device__ __forceinline__ void gru_ih_finish(const NetDev &N, const float *W, int l, const float *xin, int in_len,
                                              const float *hprev, float *hnew, int j, int g, u64 (&acc)[3][4]) {
    u64 ai[3][4];
    gru_ih_acc<R, HT>(N, W, l, xin, in_len, j, g, acc, ai);
    const float *ho = hprev + j * R + g * NET_RT;
    float *hn = hnew + j * R + g * NET_RT;
    float out[NET_RT];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        float r0, r1, z0, z1, ni0, ni1, nh0, nh1;
        unpack2(ai[0][r], r0, r1); unpack2(ai[1][r], z0, z1); unpack2(ai[2][r], ni0, ni1); unpack2(acc[2][r], nh0, nh1);
        const float n0 = tanh_f(fmaf(sigmoid_f(r0), nh0, ni0)), n1 = tanh_f(fmaf(sigmoid_f(r1), nh1, ni1));
        out[2 * r] = fmaf(ho[2 * r] - n0, sigmoid_f(z0), n0);
        out[2 * r + 1] = fmaf(ho[2 * r + 1] - n1, sigmoid_f(z1), n1);
    }
    *reinterpret_cast<float4 *>(hn) = make_float4(out[0], out[1], out[2], out[3]);
    *reinterpret_cast<float4 *>(hn + 4) = make_float4(out[4], out[5], out[6], out[7]);
}

// Dense layer: a = tanh(W x + b) (Functions/Pytorch/Network.py:255-260)
template <int R, int HT>
__device__ __forceinline__ void dense_unit(const NetDev &N, const float *W, int l, const float *xin, int in_len,
                                           float *act, int j, int g) {
    const int H = HT ? HT : N.hsz[l];
    const float b = (W + N.off_bih[l])[j];
    u64 a[1][4];
#pragma unroll
    for (int r = 0; r < 4; ++r) a[0][r] = pack2(b, b);
    matvec_acc2<R, 1, HT>(W + N.off_wih[l] + j, xin + g * NET_RT, in_len, H, a);
    float *o = act + j * R + g * NET_RT;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        float v0, v1;
        unpack2(a[0][r], v0, v1);
        o[2 * r] = tanh_f(v0);
        o[2 * r + 1] = tanh_f(v1);
    }
}

// One network step of the compute warps (threads 0 .. NC-1): hidden layers only.  GRU: reads h(t-1) from buffer p of
// every layer and writes h(t) into buffer 1-p.  The recurrent product of layer 0 does not depend on this step's
// input, so it runs BEFORE the first barrier, while the row warp is still producing that input (the previous
// step's output layer + feedback); the caller's row warp must execute 1 + n_layers matching barriers.
template <int R, int HT>
__device__ __forceinline__ void compute_step(const NetDev &N, const float *W, float *hb, int hstride, int p,
                                             const float *xin, int tid) {
    constexpr int NC = R * 8;
    const bool gru = N.type == CPS_NET_GRU;
    const int H0 = HT ? HT : N.hsz[0];
    const bool split = gru && (R / NET_RT) * H0 <= NC;   // one (unit, row group) item per thread
    const int j0 = tid % H0, g0 = tid / H0;
    const bool has0 = tid < (R / NET_RT) * H0;
    u64 acc[3][4];
    if (split && has0) gru_hh<R, HT>(N, W, 0, hb + p * hstride, j0, g0, acc);
    cta_sync();  // the row warp has written this step's network input
    const float *in = xin;
    int in_len = N.n_in;
    for (int l = 0; l < N.n_layers; ++l) {
        const int H = HT ? HT : N.hsz[l];
        float *hl = hb + N.hoff[l] * R;
        if (gru) {
            if (l == 0 && split) {
                if (has0) gru_ih_finish<R, HT>(N, W, 0, in, in_len, hl + p * hstride, hl + (1 - p) * hstride, j0, g0, acc);
            } else {
                for (int item = tid; item < (R / NET_RT) * H; item += NC) {
                    const int j = item % H, g = item / H;
                    u64 a2[3][4];
                    gru_hh<R, HT>(N, W, l, hl + p * hstride, j, g, a2);
                    gru_ih_finish<R, HT>(N, W, l, in, in_len, hl + p * hstride, hl + (1 - p) * hstride, j, g, a2);
                }
            }
            in = hl + (1 - p) * hstride;
        } else {
            for (int item = tid; item < (R / NET_RT) * H; item += NC) dense_unit<R, HT>(N, W, l, in, in_len, hl, item % H, item / H);
            in = hl;
        }
        in_len = H;
        cta_sync();
    }
}

// Linear output layer for one rollout, by the row warp: y = W_out h + b_out.  R = 16: lane = r + 16 * half, the two
// halves take alternate units and are combined with one shuffle; R = 32: lane = r.
template <int R>
__device__ __forceinline__ void out_layer_row(const NetDev &N, const float *W, const float *hlast, int lane, float (&y)[6]) {
    const int H = N.hsz[N.n_layers - 1];
    const float *Wo = W + N.off_wout, *bo = W + N.off_bout;
    constexpr int NS = 32 / R;          // lanes per rollout
    const int r = lane % R, part = lane / R;
#pragma unroll
    for (int o = 0; o < 6; ++o) y[o] = (o < N.n_out && part == 0) ? bo[o] : 0.0f;
    for (int j = part; j < H; j += NS) {
        const float hv = hlast[j * R + r];
#pragma unroll
        for (int o = 0; o < 6; ++o)
            if (o < N.n_out) y[o] = fmaf(Wo[j * N.n_out + o], hv, y[o]);
    }
    if (NS == 2) {
#pragma unroll
        for (int o = 0; o < 6; ++o) y[o] += __shfl_xor_sync(0xffffffffu, y[o], 16);
    }
}
