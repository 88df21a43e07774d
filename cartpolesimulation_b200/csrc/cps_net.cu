// cps_net.cu -- autoregressive neural predictor (GRU / Dense) of libcps_b200.so, FP32 CUDA-core path.
//
// Reference: SI_Toolkit/src/SI_Toolkit/Predictors/predictor_autoregressive_neural.py:266-313 (_predict_core),
// :332-352 (_update_internal_state_tf); Functions/Pytorch/Network.py:239-287 (Sequence.forward, GRUCell / Linear
// stack); Predictors/autoregression.py:33-158 (feedback loop, differential variant);
// Functions/General/Normalising.py:15-186; ToolkitCustomization/predictors_customization.py:71-139 (augmentation).
//
// net_kernel<R, HT, MPPI>: one CTA advances a tile of R (16 | 32) rollouts through the whole horizon.
//   * all weights live in shared memory for the whole launch (2x64 GRU: 156 KB), fetched once with one bulk
//     asynchronous copy (cp.async.bulk + mbarrier);
//   * R/4 compute warps: thread (row group g, unit j) keeps the gate pre-activations of 8 rollouts for one hidden
//     unit in registers as 4 packed pairs and accumulates them with FFMA2 (fma.rn.f32x2: two IEEE fp32 FMAs per
//     issue slot); weights are read conflict-free ([in][3H] layout, consecutive lanes = consecutive units),
//     activations as broadcast 16-byte loads ([unit][R] layout) -> 24 FMAs per 5 shared-memory loads and 12 issue
//     slots; HT = compile-time hidden size (64, 32; 0 = any) turns the address arithmetic into immediates;
//   * 1 "row" warp (lane = rollout): the linear output layer, the feedback into the next network input,
//     de-normalisation, angle augmentation, trajectory store, stage / terminal cost, MPPI perturbation interpolation
//     and the next control.  The recurrent product W_hh h of the first layer does not depend on the fed-back output,
//     so the compute warps run it while the row warp produces the input: the output layer is off the critical path;
//   * MPPI = true additionally does what mppi_kernel does after the rollout (block partials, last-block merge,
//     clipped u_nom / u) and then advances the stored hidden state by one step on (u, s)
//     (optimizer_mppi.py:191,194-196) -- one launch per solve.
#include <cuda_runtime.h>

#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include "cps_net_fp32.cuh"

template <int R, int HT, bool MPPI, bool FLEET>
__global__ void __launch_bounds__(R * 8 + 32, 1) net_kernel(const __grid_constant__ NetArgs a,
                                                            const __grid_constant__ NetFleetMppiExt fx) {
    constexpr int NC = R * 8, NT = NC + 32;
    extern __shared__ __align__(16) float smem[];
    __shared__ __align__(8) unsigned long long s_bar;
    __shared__ unsigned s_ticket;
    const NetDev &N = a.net;
    const int tid = threadIdx.x, lane = tid & 31;
    const bool row_warp = tid >= NC;
    const int T = a.T;
    const int row0 = blockIdx.x * R;
    // differential networks: autoregression_loop.run takes the integrating helper only in its general loop; with
    // horizon == 1 the "0th iteration" branch hands out the raw network output (autoregression.py:49-70)
    const bool diff = N.differential && T > 1;
    const int e = FLEET ? (int)blockIdx.y : 0;   // FLEET: the CTA's experiment

    // ---- shared-memory carve-up ------------------------------------------------------------------------------
    float *wsm = smem;                              // [n_weights]
    float *hb = wsm + N.n_weights;                  // GRU: [2][htot][R]; Dense: [htot][R] activations
    const int hstride = N.htot * R;
    float *xin = hb + 2 * hstride;                  // [n_in][R]
    float *snorm = xin + 8 * R;                     // [n_out][R] (differential nets: integrated normalised state)
    float *s_unom = snorm + 8 * R;                  // MPPI: [T] shifted nominal inputs, then [p] w0, [p] w1, scratch
    float *s_w0 = s_unom + (MPPI ? a.mp.T : 0);
    float *s_w1 = s_w0 + (MPPI ? a.mp.p : 0);
    float *s_red = s_w1 + (MPPI ? a.mp.p : 0);      // [n_red + 2 + 16]
    float *s_rs = s_red + (MPPI ? a.mp.n_red + 2 + 16 : 0);   // MAX_COST plugins: row-sum slots [32][R] (RowSumPlan)
    CostParams *s_cost = reinterpret_cast<CostParams *>(s_rs + 32 * R);   // FLEET: the experiment's cost parameters

    // ---- weights: one bulk asynchronous copy global -> shared ---------------------------------------------------
    if (tid == 0) weights_copy_start(&s_bar, wsm, a.weights, N.n_weights);

    // ---- prologue: hidden state, MPPI tables ------------------------------------------------------------------------
    if (N.type == CPS_NET_GRU) {
        for (int idx = tid; idx < N.htot * R; idx += NT) {
            const int j = idx / R, r = idx % R;
            const int b = min(row0 + r, a.B - 1);
            hb[idx] = FLEET ? fx.h[(long long)e * N.htot + j] : a.h0[(long long)b * a.hs_b + j];
        }
    }
    if (MPPI) {
        // warm-start shift at the START of the solve (optimizer_mppi.py:183)
        for (int t = tid; t < T; t += NT) s_unom[t] = (FLEET ? fx.u_nom + (long long)e * T : a.u_nom)[min(t + 1, T - 1)];
        for (int j = tid; j < a.mp.p; j += NT) {
            s_w0[j] = (float)(a.mp.p - j) / (float)a.mp.p;
            s_w1[j] = (float)j / (float)a.mp.p;
        }
        if (FLEET && tid == 0) fleet_cost_stage(fx, e, s_cost);
    }
    __syncthreads();  // also publishes the mbarrier init

    // ---- row-warp state --------------------------------------------------------------------------------------
    const int r_row = lane % R;                    // rollout handled by this lane of the row warp
    const bool row_lead = row_warp && lane < R;    // the lane that owns the rollout's bookkeeping
    const int k = row0 + r_row;
    const bool active = row_lead && k < a.B;
    const int kc = min(k, a.B - 1);
    float Jacc = 0.0f, corr = 0.0f, up = FLEET ? fx.u_prev[e] : a.u_prev, u_cur = 0.0f, du_cur = 0.0f, u_nxt = 0.0f, du_nxt = 0.0f;
    // default / quadratic_boundary: the T+1 cost entries are summed in the reference backend's order (cps_device.cuh)
    const bool rowsum = MPPI && (a.cost_id == CPS_COST_DEFAULT || a.cost_id == CPS_COST_QUADRATIC_BOUNDARY);
    const RowSumPlan rsp = row_sum_plan(T + 1);
    float *sl = s_rs + r_row;
    float rs_tail = 0.0f;
    if (rowsum && row_lead) row_sum_init(rsp, sl, R);
    int seg = 0, jj = 0;
    float na = 0.0f, nb = 0.0f;
    const float *nz = nullptr;
    const float *qrow = nullptr;
    float *traj = nullptr;
    if (row_warp) {
        traj = (a.traj_out && active) ? a.traj_out + (long long)k * a.ts_k : nullptr;
        if (MPPI) {
            nz = (FLEET ? a.noise + (long long)e * a.mp.n_ind * a.B : a.noise) + (long long)kc * a.ns_k;
            na = nz[0] * a.mp.sigma;
            nb = (a.mp.n_ind > 1) ? nz[a.ns_i] * a.mp.sigma : 0.0f;
        } else {
            qrow = a.Q + (long long)kc * a.qs_b;
        }
    }
    // control of step t (row warp): MPPI: clip(u_nom[t] + delta_u[t]) with delta_u interpolated from the inducing
    // points (Interpolator.py:53-77); else Q[k][t]
    auto next_control = [&](int t) {
        if (MPPI) {
            const MppiParams &mp = a.mp;
            du_nxt = (seg == mp.n_ind - 1) ? na * mp.inv_p : fmaf(na, s_w0[jj], nb * s_w1[jj]);
            if (++jj == mp.p) {
                jj = 0; ++seg; na = nb;
                nb = (seg + 1 < mp.n_ind) ? nz[(long long)(seg + 1) * a.ns_i] * mp.sigma : 0.0f;
            }
            u_nxt = clampf(s_unom[t] + du_nxt, mp.lo, mp.hi);
        } else {
            u_nxt = qrow[(long long)t * a.qs_t];
        }
    };
    if (row_warp) next_control(0);
    // all threads: wait for the weights
    weights_copy_wait(&s_bar);
    __syncthreads();

    // ---- the horizon ------------------------------------------------------------------------------------------
    int p = 0;  // hidden-state buffer holding h(t-1)
    float st[6], y[6];
    const float *hlast_base = hb + N.hoff[N.n_layers - 1] * R;
#pragma unroll 1
    for (int t = 0; t < T; ++t) {
        if (row_warp) {
            // (1) this step's network input: control + state features (the initial state, or the previous output)
            if (t == 0) {
#pragma unroll
                for (int c = 0; c < 6; ++c) st[c] = (FLEET ? fx.s + (long long)e * 8 : a.s0)[(long long)kc * a.ss_b + c];
                if (row_lead) {
                    for (int i = 0; i < N.n_state_in; ++i)
                        xin[(1 + i) * R + r_row] = fmaf(N.norm_a[1 + i], (FLEET ? fx.s + (long long)e * 8 : a.s0)[(long long)kc * a.ss_b + N.in_idx[i]], N.norm_b[1 + i]);
                    if (diff)  // dmah.set_starting_point (autoregression.py:145-146)
                        for (int o = 0; o < N.n_out; ++o)
                            snorm[o * R + r_row] = fmaf(N.on_a[o], (FLEET ? fx.s + (long long)e * 8 : a.s0)[(long long)kc * a.ss_b + N.out_idx[o]], N.on_b[o]);
                }
            } else {
                out_layer_row<R>(N, wsm, hlast_base + (N.type == CPS_NET_GRU ? p * hstride : 0), lane, y);
                if (row_lead) {
                    if (diff) {  // autoregression.py:149-154
#pragma unroll
                        for (int o = 0; o < 6; ++o) {
                            if (o < N.n_out) {
                                y[o] = snorm[o * R + r_row] + fmaf(N.p1[o], y[o], N.p2[o]);
                                snorm[o * R + r_row] = y[o];
                            }
                        }
                        for (int i = 0; i < N.n_state_in; ++i) xin[(1 + i) * R + r_row] = snorm[N.out_to_in[i] * R + r_row];
                    } else {
#pragma unroll
                        for (int o = 0; o < 6; ++o)  // autoregression.py:94-98: the output is the next input
                            if (o < N.n_state_in) xin[(1 + o) * R + r_row] = y[o];
                    }
                }
            }
            u_cur = u_nxt; du_cur = du_nxt;
            if (row_lead) xin[r_row] = fmaf(N.norm_a[0], u_cur, N.norm_b[0]);
            cta_sync();
            // (2) behind the compute warps: state s_t -> trajectory row, stage cost, next control
            if (t > 0) compose_state(N, y, st);
            if (traj) {
#pragma unroll
                for (int c = 0; c < 6; ++c) traj[(long long)t * a.ts_t + c * a.ts_c] = st[c];
            }
            if (MPPI) {
                const float stc = stage_cost_rt(a.cost_id, FLEET ? *s_cost : a.cost, cosf(st[IDX_ANGLE]), st[IDX_ANGLED], st[IDX_POS], u_cur, up);
                if (rowsum) { if (row_lead) row_sum_push(rsp, sl, R, rs_tail, t, stc); }
                else Jacc += stc;
                corr = fmaf(a.mp.cc_half_nu * du_cur, du_cur,
                            fmaf(a.mp.cc_R * u_cur, du_cur, fmaf(a.mp.cc_half_R * u_cur, u_cur, corr)));
                if (a.u_run_out && active) a.u_run_out[(long long)k * T + t] = u_cur;
                up = u_cur;
            }
            if (t + 1 < T) next_control(t + 1);
            for (int l = 0; l < N.n_layers; ++l) cta_sync();
        } else {
            compute_step<R, HT>(N, wsm, hb, hstride, p, xin, tid);
        }
        p ^= 1;
    }

    // ---- last state, costs, hidden state out ---------------------------------------------------------------------
    float J = 0.0f;
    if (row_warp) {
        out_layer_row<R>(N, wsm, hlast_base + (N.type == CPS_NET_GRU ? p * hstride : 0), lane, y);
        if (diff && row_lead) {
#pragma unroll
            for (int o = 0; o < 6; ++o)
                if (o < N.n_out) y[o] = snorm[o * R + r_row] + fmaf(N.p1[o], y[o], N.p2[o]);
        }
        compose_state(N, y, st);
        if (traj) {
#pragma unroll
            for (int c = 0; c < 6; ++c) traj[(long long)T * a.ts_t + c * a.ts_c] = st[c];
        }
        if (MPPI) {
            if (rowsum) {
                if (row_lead) {
                    row_sum_push(rsp, sl, R, rs_tail, T, terminal_cost<COST_DEFAULT>(FLEET ? *s_cost : a.cost, st[IDX_ANGLE], st[IDX_POS]));
                    Jacc = row_sum_finish(rsp, sl, R, rs_tail);
                }
            }
            J = __fdiv_rn(Jacc, a.mp.T1) + corr;   // mean over T+1 entries (true division, as torch.mean) + correction
            if (active) {
                if (a.J_out) (FLEET ? a.J_out + (long long)e * a.B : a.J_out)[k] = J;
                if (!isfinite(J)) atomicAdd(a.nonfinite, 1);
            }
        }
    }
    if (a.h_final && N.type == CPS_NET_GRU) {
        for (int idx = tid; idx < N.htot * R; idx += NT) {
            const int j = idx / R, r = idx % R;
            if (row0 + r < a.B) a.h_final[(long long)(row0 + r) * N.htot + j] = hb[p * hstride + idx];
        }
    }
    if (!MPPI) return;

    // ---- MPPI: block partial (row warp), last block merges and finishes -------------------------------------------
    const MppiParams &mp = a.mp;
    const int rec = 2 + mp.n_red;
    if (row_warp) {
        const float m = warp_min(active ? J : INFINITY);
        const float wgt = active ? expf(-(J - m) * mp.inv_lambda) : 0.0f;
        float *part = (FLEET ? a.partials + (size_t)e * gridDim.x * rec : a.partials) + (size_t)blockIdx.x * rec;
        const float S = warp_sum(wgt);
        if (lane == 0) { part[0] = m; part[1] = S; }
        for (int i = 0; i < mp.n_red; ++i) {
            const float e = active ? nz[(long long)i * a.ns_i] : 0.0f;
            const float v = warp_sum(wgt * e);
            if (lane == 0) part[2 + i] = v;
        }
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) s_ticket = atomicAdd(FLEET ? fx.tickets + e : a.ticket, 1u);
    __syncthreads();
    if (s_ticket != gridDim.x - 1) return;
    __threadfence();
    // FLEET: the experiment's tiles, warm start and last control
    merge_and_finish(mp, FLEET ? a.partials + (size_t)e * gridDim.x * rec : a.partials, gridDim.x, s_red, s_unom,
                     FLEET ? fx.u_nom + (long long)e * T : a.u_nom, FLEET ? fx.u_prev + e : a.u_out, a.shard_out, false, &a.px);
    if (tid == 0) *(FLEET ? fx.tickets + e : a.ticket) = 0u;
    if (a.shard_out || !(FLEET ? fx.h : a.h_ref) || N.type != CPS_NET_GRU) return;

    // ---- advance the stored hidden state by one step on (u, s) (optimizer_mppi.py:191,194-196) --------------------
    __syncthreads();
    float *const h_ref = FLEET ? fx.h + (long long)e * N.htot : a.h_ref;
    const float u_sel = __ldcg(FLEET ? fx.u_prev + e : a.u_out);
    for (int idx = tid; idx < N.htot * R; idx += NT) hb[idx] = h_ref[idx / R];
    for (int idx = tid; idx < N.n_in * R; idx += NT) {
        const int i = idx / R;
        const float v = (i == 0) ? u_sel : (FLEET ? fx.s + (long long)e * 8 : a.s0)[N.in_idx[i - 1]];
        xin[idx] = fmaf(N.norm_a[i], v, N.norm_b[i]);
    }
    __syncthreads();
    if (row_warp) {
        for (int l = 0; l <= N.n_layers; ++l) cta_sync();
    } else {
        compute_step<R, HT>(N, wsm, hb, hstride, 0, xin, tid);
    }
    for (int j = tid; j < N.htot; j += NT) h_ref[j] = hb[hstride + j * R];
}

// =====================================================================================================
// host side
// =====================================================================================================
static size_t net_smem_bytes(const NetDev &N, int R, bool mppi, const MppiParams *mp) {
    size_t f = (size_t)N.n_weights + 2 * (size_t)N.htot * R + 16 * (size_t)R;
    if (mppi) f += (size_t)mp->T + 2 * (size_t)mp->p + (size_t)mp->n_red + 2 + 16;  // + one float per warp (merge)
    if (mppi) f += 32 * (size_t)R;   // row-sum slots of the MAX_COST plugins (T + 1 < 512: one accumulator level)
    return f * sizeof(float);
}

typedef void (*net_fn)(const NetArgs, const NetFleetMppiExt);

template <int R, bool MPPI, bool FLEET = false>
static net_fn pick_net2(int ht) {
    switch (ht) {
    case 64: return net_kernel<R, 64, MPPI, FLEET>;
    case 32: return net_kernel<R, 32, MPPI, FLEET>;
    default: return net_kernel<R, 0, MPPI, FLEET>;
    }
}
static net_fn pick_net(int R, int ht, bool mppi) {
    if (R == 32) return mppi ? pick_net2<32, true>(ht) : pick_net2<32, false>(ht);
    return mppi ? pick_net2<16, true>(ht) : pick_net2<16, false>(ht);
}

// cps_net_tc.cu
bool cps_net_tc_eligible(const NetDev &N);
void cps_net_tc_build_image(const NetDev &N, const float *w, std::vector<unsigned char> &img);
int cps_net_tc_launch(cps_handle *h, NetArgs &a, bool mppi, int n_rows);
size_t cps_net_tc_smem(const MppiParams *mp, bool mppi);
int cps_net_tc_rows(cps_handle *h, long long n_rows);
int cps_net_tc_fleet_launch(cps_handle *h, NetArgs &a, const NetFleetMppiExt &x, int E);

void cps_net_free(cps_handle *h) {
    if (!h || !h->net) return;
    cudaFree(h->net->d_tc);
    cudaFree(h->net->d_gws);
    cudaFree(h->net->d_weights);
    cudaFree(h->net->d_href);
    delete h->net;
    h->net = nullptr;
}

extern "C" int cps_net_load(cps_handle *h, const cps_net_desc *d, const float *w, long long n_weights) {
    if (!h) return CPS_ERR_INVALID;
    if (!d || !w) return fail(h, CPS_ERR_INVALID, "cps_net_load: null argument");
    if (d->struct_size != (int)sizeof(cps_net_desc))
        return fail(h, CPS_ERR_INVALID, "cps_net_load: cps_net_desc size mismatch (%d vs %d)", d->struct_size,
                    (int)sizeof(cps_net_desc));
    if (d->net_type != CPS_NET_GRU && d->net_type != CPS_NET_DENSE)
        return fail(h, CPS_ERR_UNSUPPORTED, "cps_net_load: network type %d is not supported (GRU and Dense are)", d->net_type);
    if (d->n_layers < 1 || d->n_layers > CPS_NET_MAX_LAYERS)
        return fail(h, CPS_ERR_UNSUPPORTED, "cps_net_load: 1..%d hidden layers supported", CPS_NET_MAX_LAYERS);
    if (d->n_state_in < 0 || d->n_state_in > 6 || d->n_out < 1 || d->n_out > 6)
        return fail(h, CPS_ERR_INVALID, "cps_net_load: need 0..6 state inputs and 1..6 outputs");
    if (!d->differential && d->n_state_in > d->n_out)
        return fail(h, CPS_ERR_INVALID, "cps_net_load: the outputs feed back as the next inputs, so n_out >= n_state_in is required");
    NetDev N;
    memset(&N, 0, sizeof(N));
    N.type = d->net_type; N.n_layers = d->n_layers; N.n_state_in = d->n_state_in; N.n_in = 1 + d->n_state_in;
    N.n_out = d->n_out; N.differential = d->differential ? 1 : 0;
    for (int i = 0; i < d->n_state_in; ++i) {
        if (d->in_idx[i] < 0 || d->in_idx[i] > 5) return fail(h, CPS_ERR_INVALID, "cps_net_load: in_idx out of range");
        N.in_idx[i] = d->in_idx[i];
        if (d->differential && (d->out_to_in[i] < 0 || d->out_to_in[i] >= d->n_out))
            return fail(h, CPS_ERR_INVALID, "cps_net_load: out_to_in out of range");
        N.out_to_in[i] = d->out_to_in[i];
    }
    for (int o = 0; o < d->n_out; ++o) {
        if (d->out_idx[o] < 0 || d->out_idx[o] > 5) return fail(h, CPS_ERR_INVALID, "cps_net_load: out_idx out of range");
        N.out_idx[o] = d->out_idx[o];
        if (d->out_idx[o] == IDX_ANGLE) N.has_angle = 1;
        if (d->out_idx[o] == IDX_SIN) N.has_sin = 1;
        if (d->out_idx[o] == IDX_COS) N.has_cos = 1;
        N.denorm_A[o] = d->denorm_A[o]; N.denorm_B[o] = d->denorm_B[o];
        N.p1[o] = d->diff_p1[o]; N.p2[o] = d->diff_p2[o]; N.on_a[o] = d->out_norm_a[o]; N.on_b[o] = d->out_norm_b[o];
    }
    for (int i = 0; i < N.n_in; ++i) { N.norm_a[i] = d->norm_a[i]; N.norm_b[i] = d->norm_b[i]; }
    // device image: transposed weights, every block 16-byte aligned
    const int G = (N.type == CPS_NET_GRU) ? 3 : 1;
    std::vector<float> img;
    auto align4 = [&]() { while (img.size() % 4) img.push_back(0.0f); };
    long long need = 0;
    int in_len = N.n_in, htot = 0;
    for (int l = 0; l < N.n_layers; ++l) {
        const int H = d->hidden[l];
        if (H < 1 || H > 128) return fail(h, CPS_ERR_UNSUPPORTED, "cps_net_load: hidden sizes 1..128 supported, got %d", H);
        need += (long long)G * H * in_len + (N.type == CPS_NET_GRU ? 3LL * H * H + 6LL * H : H);
        in_len = H;
    }
    need += (long long)N.n_out * in_len + N.n_out;
    if (need != n_weights)
        return fail(h, CPS_ERR_INVALID, "cps_net_load: expected %lld weights for this architecture, got %lld", need, n_weights);
    for (long long i = 0; i < n_weights; ++i)
        if (!std::isfinite(w[i])) return fail(h, CPS_ERR_INVALID, "cps_net_load: weight %lld is not finite", i);
    const float *p = w;
    in_len = N.n_in;
    auto put_T = [&](const float *src, int rows, int cols) {  // src [rows][cols] -> image [cols][rows]
        const int off = (int)img.size();
        img.resize(off + (size_t)rows * cols);
        for (int r = 0; r < rows; ++r)
            for (int c = 0; c < cols; ++c) img[off + (size_t)c * rows + r] = src[(size_t)r * cols + c];
        align4();
        return off;
    };
    auto put = [&](const float *src, int n) {
        const int off = (int)img.size();
        img.insert(img.end(), src, src + n);
        align4();
        return off;
    };
    for (int l = 0; l < N.n_layers; ++l) {
        const int H = d->hidden[l];
        N.hsz[l] = H; N.hoff[l] = htot; htot += H;
        N.off_wih[l] = put_T(p, G * H, in_len); p += (size_t)G * H * in_len;
        if (N.type == CPS_NET_GRU) {
            N.off_whh[l] = put_T(p, 3 * H, H); p += (size_t)3 * H * H;
            N.off_bih[l] = put(p, 3 * H); p += 3 * H;
            N.off_bhh[l] = put(p, 3 * H); p += 3 * H;
        } else {
            N.off_bih[l] = put(p, H); p += H;
        }
        in_len = H;
    }
    N.off_wout = put_T(p, N.n_out, in_len); p += (size_t)N.n_out * in_len;
    N.off_bout = put(p, N.n_out);
    N.htot = htot;
    N.n_weights = (int)img.size();
    const size_t smem = net_smem_bytes(N, 16, true, &h->mp);
    int ht = N.hsz[0];
    for (int l = 1; l < N.n_layers; ++l)
        if (N.hsz[l] != ht) ht = 0;
    if (ht != 64 && ht != 32) ht = 0;
    if (smem > 227 * 1024)
        return fail(h, CPS_ERR_UNSUPPORTED, "cps_net_load: the network needs %zu bytes of shared memory per CTA (limit 227 KB); "
                    "larger networks are not supported by this build", smem);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    cps_net_free(h);
    NetState *S = new (std::nothrow) NetState();
    if (!S) return fail(h, CPS_ERR_INVALID, "cps_net_load: out of host memory");
    S->dev = N; S->d_weights = nullptr; S->d_href = nullptr; S->ht = ht; S->d_tc = nullptr;
    h->net = S;
    CUDA_TRY(h, cudaMalloc(&S->d_weights, img.size() * sizeof(float)));
    CUDA_TRY(h, cudaMalloc(&S->d_href, sizeof(float) * (size_t)(htot > 0 ? htot : 1)));
    CUDA_TRY(h, cudaMemcpy(S->d_weights, img.data(), img.size() * sizeof(float), cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemset(S->d_href, 0, sizeof(float) * (size_t)(htot > 0 ? htot : 1)));
    if (cps_net_tc_eligible(N)) {  // 2 x 64 GRU: also prepare the tensor-core kernel's image
        std::vector<unsigned char> tc;
        cps_net_tc_build_image(N, w, tc);
        CUDA_TRY(h, cudaMalloc(&S->d_tc, tc.size()));
        CUDA_TRY(h, cudaMemcpy(S->d_tc, tc.data(), tc.size(), cudaMemcpyHostToDevice));
    }
    return CPS_OK;
}

static int net_launch(cps_handle *h, NetArgs &a, bool mppi, int n_rows) {
    NetState *S = h->net;
    a.net = S->dev;
    a.weights = S->d_weights;
    a.tc = S->d_tc;
    // 2 x 64 GRU: the tensor-core kernel (tcgen05; 64 or 128 rollouts per CTA) at every batch size -- a T = 50 solve takes
    // 0.21 ms up to 64 x 148 rollouts (per-step latency bound) and 1.0 ms at 65536, against 0.39 ms / 8.0 ms of the FP32
    // kernel (profiles/r02_net_timing.txt).  CPS_FLAG_NET_FP32 forces the CUDA-core kernel.
    const unsigned fl = h->cfg.flags;
    if ((fl & CPS_FLAG_NET_TENSOR_CORES) && !S->d_tc)
        return fail(h, CPS_ERR_UNSUPPORTED, "CPS_FLAG_NET_TENSOR_CORES: the tensor-core kernel supports plain (not differential, D_*) 2 x 64 GRU networks only");
    if (S->d_tc && !(fl & CPS_FLAG_NET_FP32) && ((fl & CPS_FLAG_NET_TENSOR_CORES) || cps_net_tc_smem(&h->mp, mppi) <= 227 * 1024))
        return cps_net_tc_launch(h, a, mppi, n_rows);
    // small batches: 16 rollouts per CTA spread the work over more SMs; large ones: 32 (two warps per scheduler)
    int R = (n_rows > 148 * 16) ? 32 : 16;
    if (net_smem_bytes(S->dev, R, mppi, &h->mp) > 227 * 1024) R = 16;
    const size_t smem = net_smem_bytes(S->dev, R, mppi, &h->mp);
    net_fn fn = pick_net(R, S->ht, mppi);
    CUDA_TRY(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int grid = (n_rows + R - 1) / R;
    fn<<<grid, R * 8 + 32, smem, h->stream>>>(a, NetFleetMppiExt());
    h->launches += 1;
    h->net_last_kernel = 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

extern "C" int cps_net_rollout(cps_handle *h, const float *s0_dev, int s0_batched, const float *Q_dev, int q_layout, int B,
                               int T, const float *h0_dev, int h0_batched, float *traj_out_dev, int traj_layout,
                               float *h_final_dev) {
    if (!h) return CPS_ERR_INVALID;
    if (!h->net) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_net_rollout: no network loaded (cps_net_load)");
    if (B < 0 || T < 1) return fail(h, CPS_ERR_INVALID, "cps_net_rollout: need B >= 0 and T >= 1");
    if (B == 0) return CPS_OK;
    if (!s0_dev || !Q_dev) return fail(h, CPS_ERR_INVALID, "cps_net_rollout: null input pointer");
    if (!traj_out_dev && !h_final_dev) return fail(h, CPS_ERR_INVALID, "cps_net_rollout: no output requested");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    NetArgs a;
    memset(&a, 0, sizeof(a));
    a.s0 = s0_dev; a.ss_b = s0_batched ? 6 : 0;
    a.Q = Q_dev;
    if (q_layout == CPS_TIME_MAJOR) { a.qs_b = 1; a.qs_t = B; } else { a.qs_b = T; a.qs_t = 1; }
    a.B = B; a.T = T;
    a.h0 = h0_dev ? h0_dev : h->net->d_href;
    a.hs_b = (h0_dev && h0_batched) ? h->net->dev.htot : 0;
    a.traj_out = traj_out_dev;
    if (traj_layout == CPS_TIME_MAJOR) { a.ts_k = 1; a.ts_t = 6LL * B; a.ts_c = B; }
    else { a.ts_k = (T + 1) * 6LL; a.ts_t = 6; a.ts_c = 1; }
    a.h_final = h_final_dev;
    return net_launch(h, a, false, B);
}

extern "C" int cps_net_update(cps_handle *h, const float *s_dev, const float *q0_dev) {
    if (!h) return CPS_ERR_INVALID;
    if (!h->net) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_net_update: no network loaded (cps_net_load)");
    if (!s_dev || !q0_dev) return fail(h, CPS_ERR_INVALID, "cps_net_update: null pointer");
    if (h->net->dev.type != CPS_NET_GRU) return CPS_OK;  // Dense: nothing to update (:334-335)
    return cps_net_rollout(h, s_dev, 0, q0_dev, CPS_ROLLOUT_MAJOR, 1, 1, nullptr, 0, nullptr, CPS_ROLLOUT_MAJOR,
                           h->net->d_href);
}

extern "C" int cps_net_state_size(const cps_handle *h) { return (h && h->net) ? h->net->dev.htot : -1; }

extern "C" int cps_net_reset_state(cps_handle *h) {
    if (!h) return CPS_ERR_INVALID;
    if (!h->net) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_net_reset_state: no network loaded");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (h->net->dev.htot > 0) CUDA_TRY(h, cudaMemsetAsync(h->net->d_href, 0, sizeof(float) * h->net->dev.htot, h->stream));
    return CPS_OK;
}

extern "C" int cps_net_get_state(cps_handle *h, float *out) {
    if (!h || !out) return CPS_ERR_INVALID;
    if (!h->net) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_net_get_state: no network loaded");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (h->net->dev.htot > 0) {
        CUDA_TRY(h, cudaMemcpyAsync(out, h->net->d_href, sizeof(float) * h->net->dev.htot, cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    }
    return CPS_OK;
}

extern "C" int cps_net_set_state(cps_handle *h, const float *in) {
    if (!h || !in) return CPS_ERR_INVALID;
    if (!h->net) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_net_set_state: no network loaded");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (h->net->dev.htot > 0) {
        CUDA_TRY(h, cudaMemcpyAsync(h->net->d_href, in, sizeof(float) * h->net->dev.htot, cudaMemcpyHostToDevice, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    }
    return CPS_OK;
}

// cps_mppi_step with CPS_PREDICTOR_NEURAL (called from cps_lib.cu)
int cps_net_mppi_step(cps_handle *h, const float *s_dev, const float *noise_dev, int noise_layout, float u_prev,
                      float *u_nom_dev, float *u_out_dev, float *J_out_dev, float *traj_out_dev, int traj_layout,
                      float *u_run_out_dev) {
    if (!h->net) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_mppi_step: neural predictor without a network (cps_net_load)");
    if (h->cfg.noise_mode != CPS_NOISE_INDUCING)
        return fail(h, CPS_ERR_UNSUPPORTED, "cps_mppi_step: the neural predictor supports CPS_NOISE_INDUCING only");
    if ((h->cfg.cost_id == CPS_COST_DEFAULT || h->cfg.cost_id == CPS_COST_QUADRATIC_BOUNDARY) && row_sum_slots(h->cfg.horizon + 1) > 32)
        return fail(h, CPS_ERR_UNSUPPORTED, "cps_mppi_step: default / quadratic_boundary with the neural predictor support horizons below 511");
    NetArgs a;
    memset(&a, 0, sizeof(a));
    const long long K = h->cfg.num_rollouts;
    const int T = h->cfg.horizon;
    a.s0 = s_dev; a.ss_b = 0;
    a.B = (int)K; a.T = T;
    a.h0 = h->net->d_href; a.hs_b = 0;
    a.traj_out = traj_out_dev;
    if (traj_layout == CPS_TIME_MAJOR) { a.ts_k = 1; a.ts_t = 6LL * K; a.ts_c = K; }
    else { a.ts_k = (T + 1) * 6LL; a.ts_t = 6; a.ts_c = 1; }
    a.cost_id = h->cfg.cost_id; a.cost = h->cost; a.mp = h->mp;
    a.noise = noise_dev;
    if (noise_layout == CPS_TIME_MAJOR) { a.ns_i = K; a.ns_k = 1; } else { a.ns_i = 1; a.ns_k = h->n_red; }
    a.u_prev = u_prev;
    a.u_nom = u_nom_dev; a.u_out = u_out_dev; a.J_out = J_out_dev; a.u_run_out = u_run_out_dev;
    a.partials = h->d_partials; a.ticket = h->d_ticket; a.nonfinite = h->d_nonfinite;
    a.shard_out = h->shard ? h->shard_out : nullptr;
    a.px = h->px;
    if (h->px.world > 1) a.px.epoch = ++h->px.epoch;
    a.h_ref = h->net->d_href;
    return net_launch(h, a, true, (int)K);
}

// ---- cps_fleet.cu: MPPI fleets on the neural predictor ----------------------------------------------------------------
// The kernel an MPPI fleet of E experiments runs, chosen as net_launch chooses it for a single solve: the tensor-core kernel
// for the GRUs it takes (live rollouts per CTA from the fleet's E x K rollouts by cps_net_tc_launch's rule), else the FP32
// kernel with R from the per-experiment K, so that every experiment runs the arithmetic of one cps_mppi_step.  Both stage
// the experiment's cost parameters in shared memory behind the single solve's carve-up.
int cps_net_mppi_fleet_plan(cps_handle *h, int E, const char *who, NetFleetPlan *p) {
    if (!h->net) return fail(h, CPS_ERR_NOT_CONFIGURED, "%s: neural predictor without a network (cps_net_load)", who);
    if (h->cfg.noise_mode != CPS_NOISE_INDUCING)
        return fail(h, CPS_ERR_UNSUPPORTED, "%s: the neural predictor supports CPS_NOISE_INDUCING only", who);
    if ((h->cfg.cost_id == CPS_COST_DEFAULT || h->cfg.cost_id == CPS_COST_QUADRATIC_BOUNDARY) && row_sum_slots(h->cfg.horizon + 1) > 32)
        return fail(h, CPS_ERR_UNSUPPORTED, "%s: default / quadratic_boundary with the neural predictor support horizons below 511", who);
    NetState *S = h->net;
    const unsigned fl = h->cfg.flags;
    const int K = h->cfg.num_rollouts;
    if ((fl & CPS_FLAG_NET_TENSOR_CORES) && !S->d_tc)
        return fail(h, CPS_ERR_UNSUPPORTED, "CPS_FLAG_NET_TENSOR_CORES: the tensor-core kernel supports plain (not differential, D_*) 2 x 64 GRU networks only");
    const size_t tc_smem = cps_net_tc_smem(&h->mp, true) + sizeof(CostParams);
    if (S->d_tc && !(fl & CPS_FLAG_NET_FP32) && ((fl & CPS_FLAG_NET_TENSOR_CORES) || tc_smem <= 227 * 1024)) {
        if (tc_smem > 227 * 1024) return fail(h, CPS_ERR_UNSUPPORTED, "%s: horizon too large for the tensor-core kernel's shared memory", who);
        p->kernel = 2;
        p->rows = cps_net_tc_rows(h, (long long)E * K);
        p->smem = tc_smem;
    } else {
        int R = (K > 148 * 16) ? 32 : 16;
        if (net_smem_bytes(S->dev, R, true, &h->mp) > 227 * 1024) R = 16;
        p->kernel = 1;
        p->rows = R;
        p->smem = net_smem_bytes(S->dev, R, true, &h->mp) + sizeof(CostParams);
        if (p->smem > 227 * 1024)
            return fail(h, CPS_ERR_UNSUPPORTED, "%s: the network needs %zu bytes of shared memory per CTA here (limit 227 KB)", who, p->smem);
    }
    p->tiles = (K + p->rows - 1) / p->rows;
    return CPS_OK;
}

int cps_net_mppi_fleet(cps_handle *h, int E, const NetFleetPlan &p, const float *s_dev, float *u_nom_dev, float *u_prev_dev,
                       float *hid_dev, const float *tp_dev, const float *te_dev, const CostParams &cost_up, const CostParams &cost_dn,
                       const float *noise_dev, float *partials_dev, unsigned *tickets_dev, float *J_out_dev) {
    NetState *S = h->net;
    const int K = h->cfg.num_rollouts, T = h->cfg.horizon;
    NetArgs a;
    memset(&a, 0, sizeof(a));
    a.net = S->dev; a.weights = S->d_weights; a.tc = S->d_tc;
    a.B = K; a.T = T;
    a.cost_id = h->cfg.cost_id; a.cost = h->cost; a.mp = h->mp;
    a.noise = noise_dev; a.ns_i = K; a.ns_k = 1;
    a.J_out = J_out_dev; a.partials = partials_dev; a.nonfinite = h->d_nonfinite;
    a.tc_rows = p.rows;
    NetFleetMppiExt x;
    x.s = s_dev; x.u_nom = u_nom_dev; x.u_prev = u_prev_dev; x.h = hid_dev; x.tp = tp_dev; x.te = te_dev;
    x.cost_up = cost_up; x.cost_dn = cost_dn; x.tickets = tickets_dev;
    if (p.kernel == 2) return cps_net_tc_fleet_launch(h, a, x, E);
    net_fn fn = (p.rows == 32) ? pick_net2<32, true, true>(S->ht) : pick_net2<16, true, true>(S->ht);
    CUDA_TRY(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
    fn<<<dim3(p.tiles, E), p.rows * 8 + 32, p.smem, h->stream>>>(a, x);
    h->launches += 1;
    h->net_last_kernel = 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}
