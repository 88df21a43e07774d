// cps_net_tc.cu -- the GRU predictor on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//
// net_tc_kernel<MPPI>: one CTA advances 128 rollouts (one per TMEM lane) of a 2 x 64 GRU (narrower layers: zero-padded to 64
// units by cps_net_tc_build_image) through the horizon as a
// software pipeline of warp-specialised roles, so that the tensor pipe, the MUFU-bound gate epilogues and the per-rollout
// bookkeeping overlap instead of taking turns:
//   * warp 20 (converged, one elected lane executes): issues every tcgen05.mma.  Each layer is processed as two HALF-LAYER jobs of 32 hidden units
//     ([r | z | n] gate columns of those units = 96 weight rows): per step the jobs 1a, 1b, 2a, 2b.  A job accumulates
//     into one of THREE rotating 128-column tensor-memory regions {R, Z, NH, NI} (job j uses region j mod 3), which lets
//     the recurrent products W_hh h of the NEXT jobs be issued into the two idle regions while the epilogue of the
//     current job reads the third -- only the input products (W_ih1 x, W_ih2 h1) and the output layer stay on the
//     step's critical path;
//   * warps 0..15 (512 threads): gate epilogues.  Thread (rollout, quarter) reads its 8 units of the job's region with
//     tcgen05.ld, applies the GRU non-linearities and writes h(t) back as the next A operand (tensor memory, ".ts"
//     MMAs: no shared-memory round trip);
//   * warps 16..19 (128 threads, one per rollout): the output layer's result -> next network input (shared memory A
//     operand of the first layer), and off the critical path de-normalisation, angle augmentation, trajectory store,
//     stage / terminal cost, MPPI perturbation interpolation;
//   * hand-offs are mbarriers (tcgen05.commit towards the epilogue / row warps, per-warp arrivals towards the issuer).
//   * fp32 accuracy from fp16 tensor cores: every operand is split x = hi + lo (two fp16 values after a power-of-two
//     pre-scale that keeps lo out of the subnormal range: activations x 2^7, weight rows scaled to [64, 128)), and
//     each product runs as three MMAs  hi*hi + lo*hi + hi*lo  into the same accumulator (the dropped lo*lo term is
//     2^-22 relative).  The scales are undone, and the biases added, by one FMA in the epilogue;
//   * small batches (<= 32 rollouts per SM's worth: config 3, K = 2000) run with 8 live rollouts per lane quarter and put the
//     idle rows to work: row r + 8 of every 16-row group carries the lo parts of the rollout in row r ("stacked", see
//     gru_epilogue), so a product is two MMAs (W_hi, W_lo) instead of three and includes the lo * lo term;
//   * MPPI = true: block partials, last-block merge and the stored-hidden-state update as in net_kernel.
// Tensor memory (512 columns): 3 x 128 accumulator regions, h1 and h2 operands (hi + lo, 4 x 32); the output layer's 16
// columns alias the NI columns of a region that is idle at that moment.
// Reference: see cps_net.cu.  The tcgen05 building blocks were brought up with tools/tc/tc_test.cu.
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "cps_net.cuh"

namespace {
#include "cps_net_tc_common.cuh"
}  // namespace

// NARROW: both layers have at most 32 units (the reference's shipped GRU-6IN-32H1-32H2-5OUT): the second half-layer jobs
// (units 32..63) hold only padding -- their MMAs and epilogues are skipped, the hand-offs stay, so the pipeline's barrier
// protocol is the same -- and the products over a hidden state take 2 k-steps instead of 4.
//
// FLEET (MPPI only): grid (tiles, E); CTA (x, e = blockIdx.y) solves for experiment e with the per-experiment inputs of fx
// (cps_net.cuh NetFleetMppiExt), its cost parameters staged in shared memory behind the single solve's carve-up.
template <bool MPPI, bool NARROW = false, bool FLEET = false>
__global__ void __launch_bounds__(TC_NT, 1) net_tc_kernel(const __grid_constant__ NetArgs a, const __grid_constant__ NetFleetMppiExt fx) {
    constexpr int NKH = NARROW ? 2 : 4;
    constexpr bool JB = !NARROW;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint32_t s_tmem;
    // mbarriers: 0 weights landed; 1..3 region r complete (issuer -> epilogue); 4 output layer complete (issuer -> rows);
    // 5..8 epilogue of job 1a / 1b / 2a / 2b done (8 epilogue warps -> issuer); 9 next input written (4 row warps ->
    // issuer); 10 hidden-state update after the solve; 11 region of job 1a loaded into registers (8 epilogue warps -> issuer)
    __shared__ __align__(8) unsigned long long s_bars[12];
    __shared__ unsigned s_ticket;
    __shared__ float s_bmin[4];
#ifdef CPS_TC_TRACE
    __shared__ long long s_tr[48];
#endif
    const NetDev &N = a.net;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool is_epi = warp < TC_EW, is_row = warp >= TC_EW && warp < TC_EW + 4, is_mma = warp == TC_EW + 4;
    const int sub = (warp >> 2) & 3;           // epilogue warps: which 8 of a job's 32 units
    const int row = 32 * (warp & 3) + lane;    // rollout inside the tile (epilogue and row warps)
    const int T = a.T;
    const int e = FLEET ? (int)blockIdx.y : 0;   // FLEET: the CTA's experiment
    // Small batches are latency-bound by the step's dependence chain, not by throughput: with only the first 16 (or 8) tensor-
    // memory lanes of every lane quarter live (64 / 32 rollouts per CTA) the epilogues take half the time (12 % less again), because the
    // 16-lane access shapes spread those rollouts over all 32 threads of the epilogue warps -- and all four schedulers stay
    // in use, a warp's lane quarter being tied to its scheduler.  (The MMAs cost the same for any number of live rows:
    // M = 128 is the instruction's minimum.)
    const int rpq = a.tc_rows >> 2;            // live rollouts per lane quarter: 8 | 16 | 32
    const int row0 = blockIdx.x * a.tc_rows;
    const bool live = lane < rpq;              // per lane; dead lanes run along on clamped indices and store nothing
    // 32 live rollouts: the hi / lo parts of a rollout's operands are stacked in rows r and r + 8 (gru_epilogue<.., STACK>);
    // the epilogue warps' lanes r + 8 then work on the rollout of lane r
    const bool stk = rpq == 8;
    const int k = row0 + rpq * (warp & 3) + ((stk && is_epi) ? (lane & 7) : lane);
    const bool active = is_row && live && k < a.B;
    const int kc = min(k, a.B - 1);
    float *s_f = reinterpret_cast<float *>(smem + O_FLOATS);
    float *s_unom = s_f;                                   // MPPI: [T] shifted nominal inputs, [p] w0, [p] w1, scratch
    float *s_w0 = s_unom + (MPPI ? a.mp.T : 0);
    float *s_w1 = s_w0 + (MPPI ? a.mp.p : 0);
    float *s_red = s_w1 + (MPPI ? a.mp.p : 0);             // [4][n_red + 2] then [n_red + 2 + warps]
    float *s_rs = s_red + (MPPI ? 5 * (a.mp.n_red + 2) + 8 : 0);   // MAX_COST plugins: row-sum slots [32][128] (RowSumPlan)
    CostParams *s_cost = reinterpret_cast<CostParams *>(s_rs + 32 * TC_ROWS);   // FLEET: the experiment's cost parameters
    const float *cst1 = reinterpret_cast<const float *>(smem + O_CST1);
    const float *cst2 = reinterpret_cast<const float *>(smem + O_CST2);
    const float *csto = reinterpret_cast<const float *>(smem + O_CSTO);   // [16][2] output layer, then {c, cn} of the two layers
    const uint32_t sm0 = smem_u32(smem), bars = smem_u32(s_bars);
    const uint32_t wbar = bars, outb = bars + 32, xrdy = bars + 72, tailb = bars + 80, ldb = bars + 88;
    auto doneb = [&](int r) { return bars + 8u + 8u * (uint32_t)r; };
    auto epib = [&](int job) { return bars + 40u + 8u * (uint32_t)job; };

    // ---- weights: bulk asynchronous copy; tensor memory; MPPI tables ------------------------------------------------
    if (tid == 0) {
        bar_init(wbar, 1);
        for (int r = 0; r < 3; ++r) bar_init(doneb(r), 1);
        bar_init(outb, 1);
        for (int j = 0; j < 4; ++j) bar_init(epib(j), TC_EW / 2);   // a job is one group's: 8 warps
        bar_init(xrdy, 4);
        bar_init(tailb, 1);
        bar_init(ldb, TC_EW / 2);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(wbar), "r"(TC_IMAGE_BYTES) : "memory");
        for (uint32_t done = 0; done < TC_IMAGE_BYTES; done += 32768u) {
            const uint32_t chunk = min(TC_IMAGE_BYTES - done, 32768u);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(sm0 + done), "l"(a.tc + done), "r"(chunk), "r"(wbar) : "memory");
        }
    }
    __syncwarp();
    if (is_mma) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem)), "n"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (MPPI) {
        for (int t = tid; t < T; t += TC_NT) s_unom[t] = (FLEET ? fx.u_nom + (long long)e * T : a.u_nom)[min(t + 1, T - 1)];   // warm-start shift (:183)
        for (int j = tid; j < a.mp.p; j += TC_NT) {
            s_w0[j] = (float)(a.mp.p - j) / (float)a.mp.p;
            s_w1[j] = (float)j / (float)a.mp.p;
        }
        if (FLEET && tid == 0) fleet_cost_stage(fx, e, s_cost);
    }
    for (int i = tid; i < 2048; i += TC_NT) reinterpret_cast<uint32_t *>(smem + O_X_HI)[i] = 0u;   // x tiles: k = 7..15 stay 0
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;
    const uint32_t tl = tmem + ((uint32_t)(32 * (warp & 3)) << 16);   // this warp's lane quarter

    // ---- row bookkeeping (row warps) ------------------------------------------------------------------------------------
    float Jacc = 0.0f, corr = 0.0f, up = FLEET ? fx.u_prev[e] : a.u_prev, u_cur = 0.0f, du_cur = 0.0f, u_nxt = 0.0f, du_nxt = 0.0f;
    int seg = 0, jj = 0;
    float na = 0.0f, nb = 0.0f;
    const float *nz = nullptr, *qrow = nullptr;
    float *traj = (a.traj_out && active) ? a.traj_out + (long long)k * a.ts_k : nullptr;
    // default / quadratic_boundary: the T+1 cost entries are summed in the reference backend's order (cps_device.cuh)
    const bool rowsum = MPPI && (a.cost_id == CPS_COST_DEFAULT || a.cost_id == CPS_COST_QUADRATIC_BOUNDARY);
    const RowSumPlan rsp = row_sum_plan(T + 1);
    float *sl = s_rs + row;
    float rs_tail = 0.0f;
    if (is_row) {
        if (MPPI) {
            nz = (FLEET ? a.noise + (long long)e * a.mp.n_ind * a.B : a.noise) + (long long)kc * a.ns_k;
            na = nz[0] * a.mp.sigma;
            nb = (a.mp.n_ind > 1) ? nz[a.ns_i] * a.mp.sigma : 0.0f;
            if (rowsum) row_sum_init(rsp, sl, TC_ROWS);
        } else {
            qrow = a.Q + (long long)kc * a.qs_b;
        }
    }
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
    // network input x = [control, state features] -> shared-memory A operand of the first layer (K padded to 16; k >= 8 is
    // zero for good).  Followed by the generic -> async proxy fence the tensor core's read needs.
    auto write_x = [&](float ctrl, const float (&feat)[6], bool stacked) {
        float x[8];
        x[0] = fmaf(N.norm_a[0], ctrl, N.norm_b[0]);
#pragma unroll
        for (int i = 0; i < 6; ++i) x[1 + i] = (i < N.n_state_in) ? feat[i] : 0.0f;
        x[7] = 0.0f;
        uint32_t ph[4], pl[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            __half h0, l0, h1, l1;
            split_h(x[2 * q] * A_SCALE, h0, l0);
            split_h(x[2 * q + 1] * A_SCALE, h1, l1);
            ph[q] = pack_h2(h0, h1);
            pl[q] = pack_h2(l0, l1);
        }
        const uint32_t off = (uint32_t)(row >> 3) * 256u + (uint32_t)(row & 7) * 16u;
        if (!stacked) {
            *reinterpret_cast<uint4 *>(smem + O_X_HI + off) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
            *reinterpret_cast<uint4 *>(smem + O_X_LO + off) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
        } else if (live) {   // rows r and r + 8 of the hi tile (the next 8-row core matrix); lanes 8.. own no row
            *reinterpret_cast<uint4 *>(smem + O_X_HI + off) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
            *reinterpret_cast<uint4 *>(smem + O_X_HI + off + 256u) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    };
    // this thread's units of a layer, chunk ch = 0, 1: [32 ch + 8 sub, + 8) -- the units it handles in job (layer, ch)
    auto chunk_u0 = [&](int ch) { return 32 * ch + TC_EU * sub; };

    // ---- initial operands -------------------------------------------------------------------------------------------------
    float st[6], y[6], feat[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) { st[c] = 0.0f; y[c] = 0.0f; }
    if (is_epi) {
        float v[TC_EU];
#pragma unroll 1
        for (int l = 0; l < 2; ++l) {
#pragma unroll 1
            for (int ch = 0; ch < 2; ++ch) {
                const int u0 = chunk_u0(ch);
#pragma unroll
                for (int i = 0; i < TC_EU; ++i)   // layers narrower than 64 units: the padding units carry (and keep) zero
                    v[i] = (u0 + i < N.hsz[l]) ? (FLEET ? fx.h[(long long)e * N.htot + N.hoff[l] + u0 + i]
                                                        : a.h0[(long long)kc * a.hs_b + N.hoff[l] + u0 + i]) : 0.0f;
                if (stk) write_operand8_stacked(tl, (l ? C_AH2_HI : C_AH1_HI) + (u0 >> 1), v, lane);
                else write_operand8(tl, (l ? C_AH2_HI : C_AH1_HI) + (u0 >> 1), (l ? C_AH2_LO : C_AH1_LO) + (u0 >> 1), v);
            }
        }
    }
    if (is_row) {
#pragma unroll
        for (int c = 0; c < 6; ++c) st[c] = (FLEET ? fx.s + (long long)e * 8 : a.s0)[(long long)kc * a.ss_b + c];
        next_control(0);
#pragma unroll
        for (int i = 0; i < 6; ++i)
            feat[i] = (i < N.n_state_in) ? fmaf(N.norm_a[1 + i], (FLEET ? fx.s + (long long)e * 8 : a.s0)[(long long)kc * a.ss_b + N.in_idx[i]], N.norm_b[1 + i]) : 0.0f;
        write_x(u_nxt, feat, stk);
    }
    bar_wait(wbar, 0);   // weights have landed
    tc_sync();

    const uint32_t AX_HI = sm0 + O_X_HI, AX_LO = sm0 + O_X_LO;
    const float ec1 = csto[32], ecn1 = csto[33], ec2 = csto[34], ecn2 = csto[35];   // epilogue scale constants (see gru_epilogue16)
    auto region = [&](int j) { return (uint32_t)(128 * (j % 3)); };   // column base of job j's accumulator region

    // ---- the horizon ------------------------------------------------------------------------------------------------------
    if (is_mma) {
        // warp-uniform operands (the compiler keeps them in uniform registers): tensor-memory base via a broadcast
        const uint32_t tm = __shfl_sync(0xffffffffu, tmem, 0);
        const uint32_t ah1_hi = tm + C_AH1_HI, ah1_lo = tm + C_AH1_LO, ah2_hi = tm + C_AH2_HI, ah2_lo = tm + C_AH2_LO;
        // recurrent parts of the first two jobs (1a, 1b of step 0); job j accumulates in region j mod 3
        issue_H<NKH>(tm + 0, ah1_hi, ah1_lo, sm0 + O_WHH1_HI, sm0 + O_WHH1_LO, 0, stk);
        if (JB) issue_H<NKH>(tm + 128, ah1_hi, ah1_lo, sm0 + O_WHH1_HI, sm0 + O_WHH1_LO, 1, stk);
        int t3 = 0;   // t mod 3 = (4 t) mod 3: region index of job 1a of this step
#pragma unroll 1
        for (int t = 0; t < T; ++t) {
            const uint32_t par = (uint32_t)(t & 1);
            const bool more = t + 1 < T;
            const int i1 = (t3 == 2) ? 0 : t3 + 1, i2 = (i1 == 2) ? 0 : i1 + 1;
            const uint32_t q0 = tm + 128u * (uint32_t)t3, q1 = tm + 128u * (uint32_t)i1, q2 = tm + 128u * (uint32_t)i2;
            // jobs of this step: 1a -> q0, 1b -> q1, 2a -> q2, 2b -> q0; next step: 1a -> q1, 1b -> q2, 2a -> q0
            TC_TR(0);
            if (t > 0) { bar_wait(xrdy, (uint32_t)((t - 1) & 1)); tc_fence_after(); }   // x(t) is in shared memory
            TC_TR(1);
            issue_X1(q0, AX_HI, AX_LO, sm0 + O_WIH1_HI, sm0 + O_WIH1_LO, 0, stk);
            tc_commit(doneb(t3));
            if (JB) issue_X1(q1, AX_HI, AX_LO, sm0 + O_WIH1_HI, sm0 + O_WIH1_LO, 1, stk);
            tc_commit(doneb(i1));
            // (after the critical input products) recurrent part of job 2a; its region was read by job 2b of step t - 1
            issue_H<NKH>(q2, ah2_hi, ah2_lo, sm0 + O_WHH2_HI, sm0 + O_WHH2_LO, 0, stk);
            TC_TR(2);
            // job 1a's region is consumed as soon as its epilogue warps hold it in registers: the recurrent part
            // of job 2b goes there right away and runs under the gate arithmetic instead of between h1(t) and the second layer
            bar_wait(ldb, par);
            tc_fence_after();
            TC_TR(3);
            if (JB) issue_H<NKH>(q0, ah2_hi, ah2_lo, sm0 + O_WHH2_HI, sm0 + O_WHH2_LO, 1, stk);
            TC_TR(4);
            bar_wait(epib(0), par);
            bar_wait(epib(1), par); tc_fence_after();      // h1(t) complete
            TC_TR(5);
            issue_X2<NKH>(q2, ah1_hi, ah1_lo, sm0 + O_WIH2_HI, sm0 + O_WIH2_LO, 0, stk);
            tc_commit(doneb(i2));
            if (JB) issue_X2<NKH>(q0, ah1_hi, ah1_lo, sm0 + O_WIH2_HI, sm0 + O_WIH2_LO, 1, stk);
            tc_commit(doneb(t3));
            if (more) issue_H<NKH>(q1, ah1_hi, ah1_lo, sm0 + O_WHH1_HI, sm0 + O_WHH1_LO, 0, stk);
            TC_TR(6);
            bar_wait(epib(2), par); tc_fence_after();
            TC_TR(7);
            TC_TR(8);
            bar_wait(epib(3), par); tc_fence_after();      // h2(t) complete; the region of job 2b is idle
            TC_TR(9);
            issue_OUT<NKH>(q0 + C_NI, ah2_hi, ah2_lo, sm0 + O_WOUT_HI, sm0 + O_WOUT_LO, stk);
            tc_commit(outb);
            TC_TR(10);
            // recurrent part of job 1b of the next step, behind the output layer: the tensor pipe executes in order, and in
            // front of it these 12 MMAs would sit between h2(t) and x(t + 1); here they run under the row warps' feedback
            if (more && JB) issue_H<NKH>(q2, ah1_hi, ah1_lo, sm0 + O_WHH1_HI, sm0 + O_WHH1_LO, 1, stk);
            t3 = i1;
        }
    } else if (is_epi) {
        // Two groups of 8 warps (two per scheduler each): group g takes the half-layer jobs (layer 1, g) and (layer 2, g) of
        // every step, a warp 16 of the job's 32 units.  The two jobs of a layer become ready almost together, so the groups
        // run side by side and one group's tensor-memory latencies and hand-offs are filled with the other's MUFU work.
        const bool two = rpq > 16;   // both 16-lane halves of the quarter carry rollouts
        const int g = warp >> 3, hs = (warp >> 2) & 1;   // job group; which 16 of the job's 32 units
#pragma unroll 1
        for (int t = 0; t < T; ++t) {
#pragma unroll 1
            for (int l = 0; l < 2; ++l) {
                const int job = 2 * l + g, j = 4 * t + job;
                if (warp == 8 * g) TC_TR(16 + 4 * job);
                bar_wait(doneb(j % 3), (uint32_t)((j / 3) & 1));
                tc_fence_after();
                if (warp == 8 * g) TC_TR(16 + 4 * job + 1);
                if (!JB && g == 1) {
                    // units 32..63 are padding in both layers: nothing to compute, their operand columns stay zero
                } else if (two) {
#pragma unroll 1
                    for (int e = 0; e < 2; ++e) {   // both 16-lane halves of 8 units at a time
                        const int cu = 16 * hs + 8 * e;   // first unit inside the job
                        gru_epilogue<2, false>(tl, region(j), (uint32_t)cu, l ? cst2 : cst1, l ? ec2 : ec1, l ? ecn2 : ecn1,
                                               l ? C_AH2_HI : C_AH1_HI, l ? C_AH2_LO : C_AH1_LO, 32 * g + cu, lane,
                                               (job == 0 && e == 1) ? ldb : 0u);
                    }
                } else if (rpq > 8) {   // 16 rollouts x this warp's 16 units in one interleaved pass
                    gru_epilogue<2, true>(tl, region(j), (uint32_t)(16 * hs), l ? cst2 : cst1, l ? ec2 : ec1, l ? ecn2 : ecn1,
                                          l ? C_AH2_HI : C_AH1_HI, l ? C_AH2_LO : C_AH1_LO, 32 * g + 16 * hs, lane,
                                          job == 0 ? ldb : 0u);
                } else {   // 8 rollouts, hi / lo rows stacked: one rollout per thread and chunk, two-pass MMAs
                    gru_epilogue<2, true, true>(tl, region(j), (uint32_t)(16 * hs), l ? cst2 : cst1, l ? ec2 : ec1, l ? ecn2 : ecn1,
                                                l ? C_AH2_HI : C_AH1_HI, l ? C_AH2_LO : C_AH1_LO, 32 * g + 16 * hs, lane,
                                                job == 0 ? ldb : 0u);   // job 1a tells the issuer when its region is in registers
                }
                if (warp == 8 * g) TC_TR(16 + 4 * job + 2);
                warp_signal(epib(job), lane);
                if (warp == 8 * g) TC_TR(16 + 4 * job + 3);
            }
        }
    } else if (is_row) {
#pragma unroll 1
        for (int t = 0; t < T; ++t) {
            // behind the tensor cores: state s_t -> trajectory row, stage cost; the control of step t + 1
            if (warp == TC_EW) TC_TR(40);
            {
                u_cur = u_nxt; du_cur = du_nxt;
                if (t > 0) compose_state(N, y, st);
                if (traj) {
#pragma unroll
                    for (int c = 0; c < 6; ++c) traj[(long long)t * a.ts_t + c * a.ts_c] = st[c];
                }
                if (MPPI) {
                    const float stc = stage_cost_rt(a.cost_id, FLEET ? *s_cost : a.cost, cosf(st[IDX_ANGLE]), st[IDX_ANGLED], st[IDX_POS], u_cur, up);
                    if (rowsum) row_sum_push(rsp, sl, TC_ROWS, rs_tail, t, stc);
                    else Jacc += stc;
                    corr = fmaf(a.mp.cc_half_nu * du_cur, du_cur,
                                fmaf(a.mp.cc_R * u_cur, du_cur, fmaf(a.mp.cc_half_R * u_cur, u_cur, corr)));
                    if (a.u_run_out && active) a.u_run_out[(long long)k * T + t] = u_cur;
                    up = u_cur;
                }
                if (t + 1 < T) next_control(t + 1);
            }
            // linear output layer -> feedback as the next input (autoregression.py:94-98)
            if (warp == TC_EW) TC_TR(41);
            bar_wait(outb, (uint32_t)(t & 1));
            tc_fence_after();
            if (warp == TC_EW) TC_TR(42);
            {
                uint32_t o[8];
                ld8(tl + region(4 * t + 6) + C_NI, o);
                ld_wait();
                if (stk) {   // row r + 8 holds the product with the lo parts of h2
#pragma unroll
                    for (int i = 0; i < 6; ++i)
                        o[i] = __float_as_uint(__uint_as_float(o[i]) + __shfl_down_sync(0xffffffffu, __uint_as_float(o[i]), 8));
                }
#pragma unroll
                for (int i = 0; i < 6; ++i) y[i] = (i < N.n_out) ? fmaf(__uint_as_float(o[i]), csto[2 * i], csto[2 * i + 1]) : 0.0f;
                if (t + 1 < T) write_x(u_nxt, y, stk);
            }
            if (t + 1 < T) {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) bar_arrive(xrdy);
            }
            if (warp == TC_EW) TC_TR(43);
        }
    }
    tc_sync();
#ifdef CPS_TC_TRACE
    if (blockIdx.x == 0 && tid == 0) {
        const long long b = s_tr[0];
        printf("TRACE step %d (cycles after the issuer's step start)\n", TC_TRACE_STEP);
        printf(" issuer: x ready %lld | X1a X1b H2a issued %lld | e1a seen %lld | H2b issued %lld | e1b seen %lld | X2a X2b H1a' issued %lld | e2a seen %lld | H1b' issued %lld | e2b seen %lld | OUT issued %lld\n",
               s_tr[1] - b, s_tr[2] - b, s_tr[3] - b, s_tr[4] - b, s_tr[5] - b, s_tr[6] - b, s_tr[7] - b, s_tr[8] - b, s_tr[9] - b, s_tr[10] - b);
        for (int j = 0; j < 4; ++j)
            printf(" epilogue job %d: wait from %lld | region ready %lld | math done %lld | signalled %lld\n", j, s_tr[16 + 4 * j] - b,
                   s_tr[17 + 4 * j] - b, s_tr[18 + 4 * j] - b, s_tr[19 + 4 * j] - b);
        printf(" row: step start %lld | bookkeeping done %lld | out ready %lld | x written %lld\n", s_tr[40] - b, s_tr[41] - b, s_tr[42] - b, s_tr[43] - b);
    }
#endif

    // ---- last state, costs, hidden state out ---------------------------------------------------------------------------
    float J = 0.0f;
    if (is_row) {
        compose_state(N, y, st);
        if (traj) {
#pragma unroll
            for (int c = 0; c < 6; ++c) traj[(long long)T * a.ts_t + c * a.ts_c] = st[c];
        }
        if (MPPI) {
            if (a.cost_id == CPS_COST_DEFAULT || a.cost_id == CPS_COST_QUADRATIC_BOUNDARY) {
                const float term = terminal_cost<COST_DEFAULT>(FLEET ? *s_cost : a.cost, st[IDX_ANGLE], st[IDX_POS]);
                if (rowsum) {
                    row_sum_push(rsp, sl, TC_ROWS, rs_tail, T, term);
                    Jacc = row_sum_finish(rsp, sl, TC_ROWS, rs_tail);
                } else {
                    Jacc += term;
                }
            }
            J = __fdiv_rn(Jacc, a.mp.T1) + corr;   // mean over T+1 entries (true division, as torch.mean) + correction
            if (active) {
                if (a.J_out) (FLEET ? a.J_out + (long long)e * a.B : a.J_out)[k] = J;
                if (!isfinite(J)) atomicAdd(a.nonfinite, 1);
            }
        }
    }
    auto store_hidden = [&](float *dst, bool stacked) {  // this epilogue thread's 2 x 2 x 8 units of the current hidden state
        float v[TC_EU];
#pragma unroll 1
        for (int l = 0; l < 2; ++l) {
#pragma unroll 1
            for (int ch = 0; ch < 2; ++ch) {
                const int u0 = chunk_u0(ch);
                if (stacked) read_operand8_stacked(tl, (l ? C_AH2_HI : C_AH1_HI) + (u0 >> 1), v);
                else read_operand8(tl, (l ? C_AH2_HI : C_AH1_HI) + (u0 >> 1), (l ? C_AH2_LO : C_AH1_LO) + (u0 >> 1), v);
                if (dst) {
#pragma unroll
                    for (int i = 0; i < TC_EU; ++i)
                        if (u0 + i < N.hsz[l]) dst[N.hoff[l] + u0 + i] = v[i];
                }
            }
        }
    };
    if (a.h_final && is_epi) store_hidden((live && k < a.B) ? a.h_final + (long long)k * N.htot : nullptr, stk);

    bool last = false;
    if (MPPI) {
        // ---- block partial {min J, sum w, sum w*eps[.]} over the 128 rollouts (row warps) ------------------------------
        const MppiParams &mp = a.mp;
        const int rec = 2 + mp.n_red;
        const int rw = warp - TC_EW;
        if (is_row) {
            const float m = warp_min(active ? J : INFINITY);
            if (lane == 0) s_bmin[rw] = m;
        }
        __syncthreads();
        const float m = fminf(fminf(s_bmin[0], s_bmin[1]), fminf(s_bmin[2], s_bmin[3]));
        if (is_row) {
            const float wgt = active ? expf(-(J - m) * mp.inv_lambda) : 0.0f;
            const float S = warp_sum(wgt);
            if (lane == 0) s_red[rw * rec + 1] = S;
            for (int i = 0; i < mp.n_red; ++i) {
                const float e = active ? nz[(long long)i * a.ns_i] : 0.0f;
                const float v = warp_sum(wgt * e);
                if (lane == 0) s_red[rw * rec + 2 + i] = v;
            }
        }
        __syncthreads();
        float *part = (FLEET ? a.partials + (size_t)e * gridDim.x * rec : a.partials) + (size_t)blockIdx.x * rec;
        for (int c = tid; c < mp.n_red + 1; c += TC_NT)
            part[1 + c] = (s_red[1 + c] + s_red[rec + 1 + c]) + (s_red[2 * rec + 1 + c] + s_red[3 * rec + 1 + c]);
        if (tid == 0) part[0] = m;
        __threadfence();
        __syncthreads();
        if (tid == 0) s_ticket = atomicAdd(FLEET ? fx.tickets + e : a.ticket, 1u);
        __syncthreads();
        last = s_ticket == gridDim.x - 1;
        if (last) {
            __threadfence();
            // FLEET: the experiment's tiles, warm start and last control
            merge_and_finish(mp, FLEET ? a.partials + (size_t)e * gridDim.x * rec : a.partials, gridDim.x, s_red, s_unom,
                             FLEET ? fx.u_nom + (long long)e * T : a.u_nom, FLEET ? fx.u_prev + e : a.u_out, a.shard_out, false, &a.px);
            if (tid == 0) *(FLEET ? fx.tickets + e : a.ticket) = 0u;
        }
        if (last && !a.shard_out && (FLEET ? fx.h : a.h_ref)) {
            // ---- advance the stored hidden state by one step on (u, s) (optimizer_mppi.py:191,194-196): one more,
            //      unpipelined, network step with every rollout carrying the stored state --------------------------------
            __syncthreads();
            float *const h_ref = FLEET ? fx.h + (long long)e * N.htot : a.h_ref;
            const float u_sel = __ldcg(FLEET ? fx.u_prev + e : a.u_out);
            const bool upd = row < 32;   // the stored state is one row: the first lane quarter carries it
            if (is_epi && upd) {
                float v[TC_EU];
#pragma unroll 1
                for (int l = 0; l < 2; ++l) {
#pragma unroll 1
                    for (int ch = 0; ch < 2; ++ch) {
                        const int u0 = chunk_u0(ch);
#pragma unroll
                        for (int i = 0; i < TC_EU; ++i) v[i] = (u0 + i < N.hsz[l]) ? h_ref[N.hoff[l] + u0 + i] : 0.0f;
                        write_operand8(tl, (l ? C_AH2_HI : C_AH1_HI) + (u0 >> 1), (l ? C_AH2_LO : C_AH1_LO) + (u0 >> 1), v);
                    }
                }
            }
            if (is_row && upd) {
#pragma unroll
                for (int i = 0; i < 6; ++i)
                    feat[i] = (i < N.n_state_in) ? fmaf(N.norm_a[1 + i], (FLEET ? fx.s + (long long)e * 8 : a.s0)[N.in_idx[i]], N.norm_b[1 + i]) : 0.0f;
                write_x(u_sel, feat, false);
            }
            tc_sync();
            const uint32_t tmu = __shfl_sync(0xffffffffu, tmem, 0);   // warp-uniform for the issuer (see tc_mma)
            if (is_mma) {
                issue_H(tmu + 0, tmu + C_AH1_HI, tmu + C_AH1_LO, sm0 + O_WHH1_HI, sm0 + O_WHH1_LO, 0, false);
                issue_X1(tmu + 0, AX_HI, AX_LO, sm0 + O_WIH1_HI, sm0 + O_WIH1_LO, 0, false);
                issue_H(tmu + 128, tmu + C_AH1_HI, tmu + C_AH1_LO, sm0 + O_WHH1_HI, sm0 + O_WHH1_LO, 1, false);
                issue_X1(tmu + 128, AX_HI, AX_LO, sm0 + O_WIH1_HI, sm0 + O_WIH1_LO, 1, false);
                tc_commit(tailb);
            }
            bar_wait(tailb, 0);
            tc_fence_after();
            if (is_epi && upd) {
                gru_epilogue<1, true>(tl, 0, (uint32_t)(TC_EU * sub), cst1, ec1, ecn1, C_AH1_HI, C_AH1_LO, chunk_u0(0), lane);
                gru_epilogue<1, true>(tl, 128, (uint32_t)(TC_EU * sub), cst1, ec1, ecn1, C_AH1_HI, C_AH1_LO, chunk_u0(1), lane);
            }
            tc_sync();
            if (is_mma) {
                issue_H(tmu + 256, tmu + C_AH2_HI, tmu + C_AH2_LO, sm0 + O_WHH2_HI, sm0 + O_WHH2_LO, 0, false);
                issue_X2(tmu + 256, tmu + C_AH1_HI, tmu + C_AH1_LO, sm0 + O_WIH2_HI, sm0 + O_WIH2_LO, 0, false);
                issue_H(tmu + 0, tmu + C_AH2_HI, tmu + C_AH2_LO, sm0 + O_WHH2_HI, sm0 + O_WHH2_LO, 1, false);
                issue_X2(tmu + 0, tmu + C_AH1_HI, tmu + C_AH1_LO, sm0 + O_WIH2_HI, sm0 + O_WIH2_LO, 1, false);
                tc_commit(tailb);
            }
            bar_wait(tailb, 1);
            tc_fence_after();
            if (is_epi && upd) {
                gru_epilogue<1, true>(tl, 256, (uint32_t)(TC_EU * sub), cst2, ec2, ecn2, C_AH2_HI, C_AH2_LO, chunk_u0(0), lane);
                gru_epilogue<1, true>(tl, 0, (uint32_t)(TC_EU * sub), cst2, ec2, ecn2, C_AH2_HI, C_AH2_LO, chunk_u0(1), lane);
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                store_hidden(row == 0 ? h_ref : nullptr, false);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (is_mma) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(512));
}

// =====================================================================================================
// host side
// =====================================================================================================
bool cps_net_tc_eligible(const NetDev &N) {
    // layers of up to 64 units: narrower ones are padded with units whose weights and biases are zero (their gates give
    // h' = h / 2 from h = 0, and nothing reads them)
    return N.type == CPS_NET_GRU && N.n_layers == 2 && N.hsz[0] >= 1 && N.hsz[0] <= TC_H && N.hsz[1] >= 1 && N.hsz[1] <= TC_H && N.n_in <= 7 && N.n_out <= 6
           && !N.differential;
}

size_t cps_net_tc_smem(const MppiParams *mp, bool mppi) {
    size_t f = 0;
    if (mppi) f = (size_t)mp->T + 2 * (size_t)mp->p + 5 * ((size_t)mp->n_red + 2) + 8 + 32 * TC_ROWS;   // + row-sum slots
    return O_FLOATS + f * sizeof(float);
}

// Builds the kernel image from the torch-order weights: fp16 hi/lo parts of the row-scaled matrices in UMMA core-matrix
// order + the per-column epilogue constants {c = 1 / (128 s_n), b = bias}.
void cps_net_tc_build_image(const NetDev &N, const float *w, std::vector<unsigned char> &img) {
    img.assign(TC_IMAGE_BYTES, 0);
    const int H = TC_H, n_in = N.n_in, H1 = N.hsz[0], H2 = N.hsz[1];
    // torch-order weights of the H1 / H2-unit layers -> the same order for two 64-unit layers, zero in the padding units
    std::vector<float> wp((size_t)3 * H * n_in + 3 * H * H + 6 * H + 6 * H * H + 6 * H + (size_t)N.n_out * H + N.n_out, 0.0f);
    {
        const float *s_ih1 = w, *s_hh1 = s_ih1 + 3 * H1 * n_in, *s_bi1 = s_hh1 + 3 * H1 * H1, *s_bh1 = s_bi1 + 3 * H1;
        const float *s_ih2 = s_bh1 + 3 * H1, *s_hh2 = s_ih2 + 3 * H2 * H1, *s_bi2 = s_hh2 + 3 * H2 * H2, *s_bh2 = s_bi2 + 3 * H2;
        const float *s_out = s_bh2 + 3 * H2, *s_bo = s_out + N.n_out * H2;
        float *d_ih1 = wp.data(), *d_hh1 = d_ih1 + 3 * H * n_in, *d_bi1 = d_hh1 + 3 * H * H, *d_bh1 = d_bi1 + 3 * H;
        float *d_ih2 = d_bh1 + 3 * H, *d_hh2 = d_ih2 + 3 * H * H, *d_bi2 = d_hh2 + 3 * H * H, *d_bh2 = d_bi2 + 3 * H;
        float *d_out = d_bh2 + 3 * H, *d_bo = d_out + N.n_out * H;
        for (int g = 0; g < 3; ++g) {
            for (int u = 0; u < H1; ++u) {
                for (int kk = 0; kk < n_in; ++kk) d_ih1[(size_t)(g * H + u) * n_in + kk] = s_ih1[(size_t)(g * H1 + u) * n_in + kk];
                for (int kk = 0; kk < H1; ++kk) d_hh1[(size_t)(g * H + u) * H + kk] = s_hh1[(size_t)(g * H1 + u) * H1 + kk];
                d_bi1[g * H + u] = s_bi1[g * H1 + u];
                d_bh1[g * H + u] = s_bh1[g * H1 + u];
            }
            for (int u = 0; u < H2; ++u) {
                for (int kk = 0; kk < H1; ++kk) d_ih2[(size_t)(g * H + u) * H + kk] = s_ih2[(size_t)(g * H2 + u) * H1 + kk];
                for (int kk = 0; kk < H2; ++kk) d_hh2[(size_t)(g * H + u) * H + kk] = s_hh2[(size_t)(g * H2 + u) * H2 + kk];
                d_bi2[g * H + u] = s_bi2[g * H2 + u];
                d_bh2[g * H + u] = s_bh2[g * H2 + u];
            }
        }
        for (int o = 0; o < N.n_out; ++o) {
            for (int kk = 0; kk < H2; ++kk) d_out[(size_t)o * H + kk] = s_out[(size_t)o * H2 + kk];
            d_bo[o] = s_bo[o];
        }
    }
    w = wp.data();
    const float *w_ih1 = w, *w_hh1 = w_ih1 + 3 * H * n_in, *b_ih1 = w_hh1 + 3 * H * H, *b_hh1 = b_ih1 + 3 * H;
    const float *w_ih2 = b_hh1 + 3 * H, *w_hh2 = w_ih2 + 3 * H * H, *b_ih2 = w_hh2 + 3 * H * H, *b_hh2 = b_ih2 + 3 * H;
    const float *w_out = b_hh2 + 3 * H, *b_out = w_out + N.n_out * H;
    auto row_scale = [](const float *r1, int n1, const float *r2, int n2) {
        float m = 0.0f;
        for (int i = 0; i < n1; ++i) m = fmaxf(m, fabsf(r1[i]));
        for (int i = 0; i < n2; ++i) m = fmaxf(m, fabsf(r2[i]));
        if (!(m > 0.0f)) return 1.0f;
        int e;
        frexpf(m, &e);            // m = f * 2^e, f in [0.5, 1)
        return ldexpf(1.0f, 7 - e);  // s * m in [64, 128)
    };
    auto put = [&](uint32_t o_hi, uint32_t o_lo, int r, int kk, int K, float v) {
        const __half hi = __float2half_rn(v);
        const __half lo = __float2half_rn(v - __half2float(hi));
        memcpy(&img[o_hi + kmajor_off(r, kk, K)], &hi, 2);
        memcpy(&img[o_lo + kmajor_off(r, kk, K)], &lo, 2);
    };
    // one power-of-two scale per layer (the epilogue undoes it with one uniform constant): S max|w| in [64, 128).  Rows
    // with small weights lose nothing that matters: their lo parts become fp16 subnormals with an absolute resolution of
    // 2^-24 in scaled units, i.e. 2^-31 of the layer's largest weight.
    auto layer = [&](int li, const float *wih, int kin, int Kpad, const float *whh, const float *bih, const float *bhh, uint32_t oih_hi,
                     uint32_t oih_lo, uint32_t ohh_hi, uint32_t ohh_lo, uint32_t ocst) {
        float *cst = reinterpret_cast<float *>(&img[ocst]);
        const float s = row_scale(wih, 3 * H * kin, whh, 3 * H * H);
        const float c = 1.0f / (A_SCALE * s);
        const double L2E = 1.4426950408889634;
        float *cu = reinterpret_cast<float *>(&img[O_CSTO]) + 32 + 2 * li;
        cu[0] = c;
        cu[1] = (float)(-(double)c * L2E);
        for (int n = 0; n < 3 * H; ++n) {
            const int u = n % H, g = n / H;   // gate 0 = r, 1 = z, 2 = n
            const int nr = 96 * (u / 32) + 32 * g + (u % 32);               // input matrices: [r | z | n] per half-layer job
            const int nh = 96 * (u / 32) + 32 * ((g + 1) % 3) + (u % 32);   // recurrent matrices: [n | r | z]
            for (int kk = 0; kk < kin; ++kk) put(oih_hi, oih_lo, nr, kk, Kpad, wih[(size_t)n * kin + kk] * s);
            for (int kk = 0; kk < H; ++kk) put(ohh_hi, ohh_lo, nh, kk, H, whh[(size_t)n * H + kk] * s);
            // epilogue constants of the pair of units (u & ~1, u | 1): {brn x 2, bzn x 2, bni x 2, bnh x 2}
            float *k = cst + (u >> 1) * 8 + (u & 1);
            if (g == 0) k[0] = (float)(-L2E * ((double)bih[n] + (double)bhh[n]));
            else if (g == 1) k[2] = (float)(-L2E * ((double)bih[n] + (double)bhh[n]));
            else { k[4] = bih[n]; k[6] = bhh[n]; }
        }
    };
    layer(0, w_ih1, n_in, 16, w_hh1, b_ih1, b_hh1, O_WIH1_HI, O_WIH1_LO, O_WHH1_HI, O_WHH1_LO, O_CST1);
    layer(1, w_ih2, H, H, w_hh2, b_ih2, b_hh2, O_WIH2_HI, O_WIH2_LO, O_WHH2_HI, O_WHH2_LO, O_CST2);
    float *co = reinterpret_cast<float *>(&img[O_CSTO]);
    for (int o = 0; o < 16; ++o) { co[2 * o] = 0.0f; co[2 * o + 1] = 0.0f; }
    for (int o = 0; o < N.n_out; ++o) {
        const float s = row_scale(w_out + (size_t)o * H, H, nullptr, 0);
        for (int kk = 0; kk < H; ++kk) put(O_WOUT_HI, O_WOUT_LO, o, kk, H, w_out[(size_t)o * H + kk] * s);
        co[2 * o] = 1.0f / (A_SCALE * s);
        co[2 * o + 1] = b_out[o];
    }
}

int cps_net_tc_image_bytes() { return (int)TC_IMAGE_BYTES; }

// live rollouts per CTA for a launch of n_rows rollouts: 32 or 64 while that still gives every CTA its own SM (see the
// kernel's comment on rpq)
int cps_net_tc_rows(cps_handle *h, long long n_rows) {
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->cfg.device);
    int rows = (n_rows <= 32LL * sms) ? 32 : (n_rows <= 64LL * sms) ? 64 : TC_ROWS;
    if (const char *e = getenv("CPS_TC_ROWS")) {   // A/B switch (tools/bench_net.py)
        const int r = atoi(e);
        if (r == 32 || r == 64 || r == 128) rows = r;
    }
    return rows;
}

int cps_net_tc_launch(cps_handle *h, NetArgs &a, bool mppi, int n_rows) {
    const size_t smem = cps_net_tc_smem(&h->mp, mppi);
    const bool narrow = h->net->dev.hsz[0] <= 32 && h->net->dev.hsz[1] <= 32;
    void (*fn)(const NetArgs, const NetFleetMppiExt) = narrow ? (mppi ? net_tc_kernel<true, true> : net_tc_kernel<false, true>)
                                                              : (mppi ? net_tc_kernel<true, false> : net_tc_kernel<false, false>);
    CUDA_TRY(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    a.tc_rows = cps_net_tc_rows(h, n_rows);
    const int grid = (n_rows + a.tc_rows - 1) / a.tc_rows;
    fn<<<grid, TC_NT, smem, h->stream>>>(a, NetFleetMppiExt());
    h->launches += 1;
    h->net_last_kernel = 2;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

// The MPPI fleet (cps_net_mppi_fleet): a.tc_rows and the experiments' draws / partials are set by the caller
int cps_net_tc_fleet_launch(cps_handle *h, NetArgs &a, const NetFleetMppiExt &x, int E) {
    const size_t smem = cps_net_tc_smem(&h->mp, true) + sizeof(CostParams);
    const bool narrow = h->net->dev.hsz[0] <= 32 && h->net->dev.hsz[1] <= 32;
    void (*fn)(const NetArgs, const NetFleetMppiExt) = narrow ? net_tc_kernel<true, true, true> : net_tc_kernel<true, false, true>;
    CUDA_TRY(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const dim3 grid((a.B + a.tc_rows - 1) / a.tc_rows, E);
    fn<<<grid, TC_NT, smem, h->stream>>>(a, x);
    h->launches += 1;
    h->net_last_kernel = 2;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}
