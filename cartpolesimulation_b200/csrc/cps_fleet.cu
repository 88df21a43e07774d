// cps_fleet.cu -- E independent closed-loop experiments advanced together (BASELINE configs[4]: data_generator with
// 8192 MPPI-controlled cartpoles; SURVEY.md 8f row f1).
//
// One launch = one controller period of EVERY experiment:
//   grid (blocks_per_experiment, E).  All blocks of experiment e run its MPPI solve (mppi_solve_block, the same code
//   as mppi_kernel) on the experiment's own state, nominal inputs, last control and targets; the block that finishes
//   last merges the partials, obtains Q = u_nom[0], writes the experiment's record row and then integrates the PLANT
//   (CartPole.update_state, CartPole/__init__.py:283-324: Euler-Cromer at dt_simulation, edge bounce, cos/sin, fmod
//   wrap; second derivatives refreshed every tick) for one controller period in the reference's mixed
//   float32/float64 arithmetic, and stores the new state.  Nothing returns to the host between periods.
//
// Perturbations are either supplied ([E][n_ind][K] standard-normal draws per period -- the "identical injected noise"
// hook of the parity tests) or generated in the kernel: Philox4x32-10 keyed by the seed, counter = (rollout, draw group,
// period, GLOBAL experiment index) + Box-Muller, staged in shared memory so the integration loop keeps its registers.
// The streams depend only on the global experiment index, so results do not change with the sharding over GPUs.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>
#include <cstring>
#include <new>
#include <vector>

#include "cps_internal.cuh"
#include "cps_plant.cuh"

// Plant-side models between the plant and the controller (all OFF in the shipped configuration,
// cartpole_physical_parameters.yml:13-24): control disturbance (CartPole/noise_control_signal.py:5-26), measurement
// noise (CartPole/noise_adder.py:69-84), latency (CartPole/latency_adder.py:10-74).  Per plant tick the reference pushes
// the true state into a ring buffer, reads it back `latency` seconds late (linear interpolation between the two
// neighbouring ticks, all six components), adds the measurement noise and recomputes cos / sin; the controller is handed
// that observation, the plant keeps integrating the true state.
struct PlantModels {
    int on;                    // any of the three enabled: the solve reads `obs`, the plant stage maintains ring / obs
    int ctrl_mode;             // 0 OFF, 1 additive, 2 truncnorm
    float ctrl_mult, ctrl_add;
    int meas_on;
    float sig_a, sig_p, sig_aD, sig_pD;
    int lat_int;               // int(latency / dt_simulation)
    double lat_frac;           // latency / dt_simulation - lat_int
    int ring_len;              // lat_int + 2 slots of 6 floats per experiment
    float *obs;                // [E][8] the controller's view of the state for the next solve
    float *ring;               // [E][ring_len][6]
    long long pushed;          // states pushed per experiment before this launch
    const float *ctrl_draws;   // [E] standard normal (additive) / uniform (truncnorm) draw of this period, or null: Philox
    const float *meas_draws;   // [n_sim][E][4] standard normals of this period (angle, position, angleD, positionD), or null
};

struct FleetArgs {
    PlantModels pm;
    OdeParams ode;              // the controller's model (L, m_pole "for controller")
    CostParams cost_up, cost_dn;  // folded for target_equilibrium = +1 / -1 (quadratic_boundary_grad selects its set)
    MppiParams mp;
    PlantParams plant;
    int bpe;                    // blocks per experiment
    float *s;                   // [E][8] current state (6 used)
    float *u_nom;               // [E][T]
    float *u_prev;              // [E] last returned control
    const float *tp, *te;       // [E] targets of this period (null: 0 / +1)
    const float *noise;         // supplied draws [E][n_ind][K] of this period, or null (Philox)
    unsigned long long seed;
    unsigned period;            // controller period index (Philox counter)
    unsigned e_offset;          // global index of local experiment 0
    float *partials;            // [E][bpe][2 + n_red]
    unsigned *tickets;          // [E]
    int *nonfinite;
    float *record;              // [E][CPS_FLEET_RECORD] of this period, or null
    float *J_out;               // [E][K] or null
    double time;                // period * dt_control
    // relabel mode (cps_fleet_relabel): states come from a recording, the plant is not integrated
    const float *replay_s;      // [E][6] recorded states of this row, or null (closed loop)
    const float *L_row, *mp_row;  // [E] controller-model pole length / mass of this row, or null (handle's values)
    float *Q_out;               // [E] controls computed for this row
    const int *active;          // [E] or null: files with 0 sit this row out (controller state untouched, no output)
    FoldInputs fold;            // the device-side fold of (L, m_pole)
};

// cps_fleet_noise: materialise the draws the kernel generates, [E][n_ind][K]
__global__ void __launch_bounds__(256) fleet_noise_kernel(unsigned long long seed, unsigned period, unsigned e_offset, int E,
                                                          int K, int n_ind, float *out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x, e = blockIdx.y;
    if (k >= K || e >= E) return;
    philox_normals(seed, (unsigned)k, 0u, period, e_offset + (unsigned)e, n_ind, out + ((size_t)e * n_ind) * K + k, K);
}

// The controller's view after `pushed` ring pushes: delayed + interpolated state (latency_adder.py:67-71), measurement
// noise (noise_adder.py:69-84, draws n[0..3] = angle, position, angleD, positionD; null: none) and the cos / sin refresh of
// update_vertical_angle_offset with a zero offset (CartPole/__init__.py:348-358).  float64 like the reference's buffer.
__device__ __forceinline__ void plant_observe(const PlantModels &M, const float *ring, long long pushed, const float *n,
                                              float *obs) {
    const int RL = M.ring_len;
    const int i1 = (int)(((pushed - 1 - M.lat_int) % RL + RL) % RL), i2 = (int)(((pushed - 2 - M.lat_int) % RL + RL) % RL);
    double v[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) {
        const double s1 = (double)ring[i1 * 6 + c], s2 = (double)ring[i2 * 6 + c];
        v[c] = __dadd_rn(s1, __dmul_rn(M.lat_frac, __dsub_rn(s2, s1)));
    }
    if (M.meas_on && n) {
        v[IDX_ANGLE] = plant_wrap(__dadd_rn(v[IDX_ANGLE], (double)__fmul_rn(M.sig_a, n[0])));
        v[IDX_POS] = __dadd_rn(v[IDX_POS], (double)__fmul_rn(M.sig_p, n[1]));
        v[IDX_ANGLED] = __dadd_rn(v[IDX_ANGLED], (double)__fmul_rn(M.sig_aD, n[2]));
        v[IDX_POSD] = __dadd_rn(v[IDX_POSD], (double)__fmul_rn(M.sig_pD, n[3]));
    }
    v[IDX_ANGLE] = plant_wrap(v[IDX_ANGLE]);
    v[IDX_COS] = cos(v[IDX_ANGLE]);
    v[IDX_SIN] = sin(v[IDX_ANGLE]);
#pragma unroll
    for (int c = 0; c < 6; ++c) obs[c] = (float)v[c];
}

// Philox draws of the plant-side models: counter (0xFFFFFF00 + j, 0xFFFFFFFF, period, experiment) -- disjoint from the
// rollout draws, whose first word is a rollout index < K.  j = tick inside the period (measurement) or 0xFF (control).
__device__ __forceinline__ uint4 plant_philox(unsigned long long seed, unsigned period, unsigned e_global, unsigned j) {
    return philox4x32_10(make_uint4(0xFFFFFF00u + j, 0xFFFFFFFFu, period, e_global), make_uint2((unsigned)seed, (unsigned)(seed >> 32)));
}

// add_control_noise (CartPole/noise_control_signal.py:5-26): d = a standard normal (additive) or a uniform (truncnorm)
__device__ __forceinline__ float plant_control_noise(const PlantModels &M, float Q, float d) {
    if (M.ctrl_mode == 1) return __fadd_rn(__fadd_rn(Q, __fmul_rn(M.ctrl_mult, d)), M.ctrl_add);
    if (M.ctrl_mode == 2) {   // truncnorm.rvs((-1 - loc) / scale, (1 - loc) / scale, loc, scale): inverse-CDF of the draw
        const double scale = (double)M.ctrl_mult, loc = (double)Q + (double)M.ctrl_add;
        const double ca = normcdf((-1.0 - loc) / scale), cb = normcdf((1.0 - loc) / scale);
        const double z = normcdfinv(ca + (double)d * (cb - ca));
        return (float)fmin(fmax(loc + scale * z, -1.0), 1.0);
    }
    return Q;
}

// NSUB = 10 (packed solve only): the substeps of the predictors' operating point unrolled; 0: ode.n substeps in a loop.
template <int INTEG, int COST, bool PHILOX, bool PAIR, int NSUB = 0>
__global__ void __launch_bounds__(256, 4) fleet_kernel(const __grid_constant__ FleetArgs a) {
    extern __shared__ float smem[];
    __shared__ CostParams s_cost;
    const MppiParams &mp = a.mp;
    const int e = blockIdx.y, tid = threadIdx.x;
    if (a.active && a.active[e] == 0) return;   // whole experiment (all its blocks): warm start, last control and ticket stay
    const float tp = a.tp ? a.tp[e] : 0.0f, te = a.te ? a.te[e] : 1.0f;
    if (tid == 0) {
        s_cost = (te == 1.0f) ? a.cost_up : a.cost_dn;
        s_cost.target_position = tp;
        s_cost.target_equilibrium = te;
    }
    const int nwarps = blockDim.x >> 5;
    // [n_ind][rollouts of this block]; even offset: a pair's draws are read as one 8-byte word (layout: mppi_smem_floats)
    float *s_eps = smem + ((mp.T + 2 * mp.p + nwarps * (mp.n_red + 2) + mp.n_red + 4 + 1) & ~1);
    const int per_block = PAIR ? 2 * (int)blockDim.x : (int)blockDim.x;   // rollouts per block
    if (PHILOX) {
        if (PAIR) {
            const int k = 2 * (blockIdx.x * blockDim.x + tid);
            philox_normals(a.seed, (unsigned)min(k, mp.K - 2), 0u, a.period, a.e_offset + (unsigned)e, mp.n_ind, s_eps + 2 * tid, per_block);
            philox_normals(a.seed, (unsigned)min(k + 1, mp.K - 1), 0u, a.period, a.e_offset + (unsigned)e, mp.n_ind, s_eps + 2 * tid + 1,
                           per_block);
        } else {
            const int k = blockIdx.x * blockDim.x + tid;
            philox_normals(a.seed, (unsigned)min(k, mp.K - 1), 0u, a.period, a.e_offset + (unsigned)e, mp.n_ind, s_eps + tid, per_block);
        }
    }
    __syncthreads();

    SolveIO io;
    io.s = a.replay_s ? a.replay_s + (size_t)e * 6 : ((a.pm.on ? a.pm.obs : a.s) + (size_t)e * 8);
    if (PHILOX) {  // rollout k of the experiment sits at s_eps[i * per_block + (k - first rollout of this block)]
        io.noise = s_eps - (long long)blockIdx.x * per_block;
        io.ns_i = per_block; io.ns_k = 1;
    } else {
        io.noise = a.noise + (size_t)e * mp.n_ind * mp.K;
        io.ns_i = mp.K; io.ns_k = 1;
    }
    io.u_prev = a.u_prev[e];
    io.u_nom = a.u_nom + (size_t)e * mp.T;
    io.u_out = a.u_prev + e;   // the returned control becomes the next period's u_prev (optimizer_mppi.py:210)
    io.J_out = a.J_out ? a.J_out + (size_t)e * mp.K : nullptr;
    io.traj_out = nullptr; io.ts_k = io.ts_t = io.ts_c = 0; io.u_run_out = nullptr;
    io.partials = a.partials + (size_t)e * a.bpe * (mp.n_red + 2);
    io.ticket = a.tickets + e;
    io.nonfinite = a.nonfinite;
    io.shard_out = nullptr;
    io.px.world = 0;
    OdeParams ode = a.ode;
    if (a.L_row || a.mp_row)
        fold_ode_device<INTEG>(a.fold, a.L_row ? (double)a.L_row[e] : (double)a.fold.L_default,
                               a.mp_row ? (double)a.mp_row[e] : (double)a.fold.mp_default, ode);
    const bool last = PAIR ? mppi_solve_block2<INTEG, COST, NSUB, false>(ode, s_cost, mp, io, smem, blockIdx.x, a.bpe)
                           : mppi_solve_block<INTEG, COST, SC_ROTATE, CPS_NOISE_INDUCING, false, false, 0, false>(ode, s_cost, mp, io, smem,
                                                                                                       blockIdx.x, a.bpe);
    if (!last) return;
    __syncthreads();
    if (tid != 0) return;
    if (a.replay_s) {   // relabel: the control is the result; the next row brings its own state
        a.Q_out[e] = *io.u_out;
        return;
    }

    // ---- the plant: one controller period with Q held (CartPole/__init__.py:283-324, 475-527) -------------------------
    const PlantParams &P = a.plant;
    const PlantModels &M = a.pm;
    float s[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) s[c] = a.s[(size_t)e * 8 + c];   // the TRUE state (io.s is the controller's view when M.on)
    const float Qc = *io.u_out;   // written by this thread in merge_and_finish
    float Q = Qc;
    if (M.on && M.ctrl_mode) {
        float d;
        if (M.ctrl_draws) d = M.ctrl_draws[e];
        else {
            const uint4 r = plant_philox(a.seed, a.period, a.e_offset + (unsigned)e, 0xFFu);
            float n0, n1;
            box_muller(r.x, r.y, n0, n1);
            d = (M.ctrl_mode == 1) ? n0 : ((float)(r.z >> 8) + 0.5f) * 5.9604644775390625e-8f;
        }
        Q = plant_control_noise(M, Qc, d);
    }
    const float u = __fmul_rn(P.u_max, Q);
    double aDD, pDD;
    plant_ode(P, s[IDX_COS], s[IDX_SIN], s[IDX_ANGLED], s[IDX_POSD], u, aDD, pDD);
    if (a.record) plant_record(a.record + (size_t)e * CPS_FLEET_RECORD, a.time, s, aDD, pDD, Qc, Q, u, tp, te);
    float *ring = M.on ? M.ring + (size_t)e * M.ring_len * 6 : nullptr;
    plant_ticks(P, s, u, aDD, pDD, [&](int i) {
        if (M.on) {   // add_current_state_to_latency_buffer (latency_adder.py:36-47)
            float *slot = ring + (size_t)((M.pushed + i) % M.ring_len) * 6;
#pragma unroll
            for (int c = 0; c < 6; ++c) slot[c] = s[c];
        }
    });
    float *so = a.s + (size_t)e * 8;
#pragma unroll
    for (int c = 0; c < 6; ++c) so[c] = s[c];
    if (M.on) {   // what the controller will see at the start of the next period: the observation made on the last tick
        float n[4];
        const float *np_ = nullptr;
        if (M.meas_on) {
            if (M.meas_draws) {
#pragma unroll
                for (int q = 0; q < 4; ++q) n[q] = M.meas_draws[((size_t)(P.n_sim - 1) * gridDim.y + e) * 4 + q];
            } else {
                const uint4 r = plant_philox(a.seed, a.period, a.e_offset + (unsigned)e, (unsigned)(P.n_sim - 1));
                box_muller(r.x, r.y, n[0], n[1]);
                box_muller(r.z, r.w, n[2], n[3]);
            }
            np_ = n;
        }
        plant_observe(M, ring, M.pushed + P.n_sim, np_, M.obs + (size_t)e * 8);
    }
}

// Neural fleets (CPS_PREDICTOR_NEURAL): the solve is net_kernel / net_tc_kernel<.., FLEET> (cps_net.cu, cps_net_tc.cu),
// which leaves each experiment's u in u_prev[e]; this kernel is the plant period that follows, one thread per experiment:
// fleet_kernel's record row and plant with Q_applied = Q (plant-side models are not offered on neural fleets).  CEM
// fleets (cps_cem_fleet.cu) end their periods with it too.
__global__ void __launch_bounds__(128) fleet_net_plant_kernel(const __grid_constant__ NetPlantArgs a) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= a.E) return;
    const PlantParams &P = a.plant;
    float s[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) s[c] = a.s[(size_t)e * 8 + c];
    const float Q = a.u[e];
    const float u = __fmul_rn(P.u_max, Q);
    double aDD, pDD;
    plant_ode(P, s[IDX_COS], s[IDX_SIN], s[IDX_ANGLED], s[IDX_POSD], u, aDD, pDD);
    if (a.record)
        plant_record(a.record + (size_t)e * CPS_FLEET_RECORD, a.time, s, aDD, pDD, Q, Q, u, a.tp ? a.tp[e] : 0.0f,
                     a.te ? a.te[e] : 1.0f);
    plant_ticks(P, s, u, aDD, pDD, [](int) {});
    float *so = a.s + (size_t)e * 8;
#pragma unroll
    for (int c = 0; c < 6; ++c) so[c] = s[c];
}

int fleet_plant_launch(cps_handle *h, const NetPlantArgs &a) {
    fleet_net_plant_kernel<<<(a.E + 127) / 128, 128, 0, h->stream>>>(a);
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

// (Re)start of the observation chain: ring = the reference's initial buffer (zeros, cos = 1, latency_adder.py:26-28), nothing
// pushed yet; the first solve sees the TRUE state, as the controller call of set_cartpole_state_at_t0 does
// (CartPole/__init__.py:869-880: self.s, no noise, no latency).
__global__ void fleet_observe_reset_kernel(PlantModels M, const float *s, int E) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    float *ring = M.ring + (size_t)e * M.ring_len * 6;
    for (int j = 0; j < M.ring_len; ++j)
        for (int c = 0; c < 6; ++c) ring[j * 6 + c] = (c == IDX_COS) ? 1.0f : 0.0f;
    for (int c = 0; c < 8; ++c) M.obs[(size_t)e * 8 + c] = s[(size_t)e * 8 + c];
}

// ---- host side ---------------------------------------------------------------------------------------------------------
struct FleetState {
    cps_fleet_config cfg;
    int E, bpe, block, pair;   // pair: two rollouts per thread (packed FP32), K even
    size_t smem;
    int rs_off;                // MppiParams::rs_off for this geometry
    float *d_s, *d_unom, *d_uprev, *d_partials;
    unsigned *d_tickets;
    long long period;
    CostParams cost_up, cost_dn;
    PlantModels pm;            // plant-side models (cps_fleet_set_plant_models); pm.pushed counts the ring pushes
    // neural fleets (CPS_PREDICTOR_NEURAL): the controller runs net_kernel / net_tc_kernel<.., FLEET>
    int neural;
    int htot;                  // hidden-state floats per experiment of the network the fleet was created for
    float *d_h;                // [E][htot] each experiment's hidden state
    float *d_noise;            // Philox: [E][n_ind][K] the period's draws (fleet_noise_kernel), read like supplied ones
    size_t part_cap;           // floats allocated at d_partials
};

void cps_fleet_free(cps_handle *h) {
    FleetState *F = h->fleet;
    if (!F) return;
    cudaFree(F->d_s); cudaFree(F->d_unom); cudaFree(F->d_uprev); cudaFree(F->d_partials); cudaFree(F->d_tickets);
    cudaFree(F->pm.obs); cudaFree(F->pm.ring);
    cudaFree(F->d_h); cudaFree(F->d_noise);
    delete F;
    h->fleet = nullptr;
}

typedef void (*fleet_fn)(const FleetArgs);
template <int INTEG, bool PHILOX, bool PAIR, int NSUB>
static fleet_fn pick_fleet2(int cost) {
    switch (cost) {
    case CPS_COST_DEFAULT: return fleet_kernel<INTEG, COST_DEFAULT, PHILOX, PAIR, NSUB>;
    case CPS_COST_QUADRATIC_BOUNDARY: return fleet_kernel<INTEG, COST_QB, PHILOX, PAIR, NSUB>;
    case CPS_COST_QB_GRAD_MINIMAL: return fleet_kernel<INTEG, COST_GRADMIN, PHILOX, PAIR, NSUB>;
    case CPS_COST_QB_GRAD: return fleet_kernel<INTEG, COST_GRAD, PHILOX, PAIR, NSUB>;
    default: return nullptr;
    }
}
template <int INTEG>
static fleet_fn pick_fleet1(int cost, bool philox, bool pair, bool n10) {
    if (pair && n10) return philox ? pick_fleet2<INTEG, true, true, 10>(cost) : pick_fleet2<INTEG, false, true, 10>(cost);
    if (pair) return philox ? pick_fleet2<INTEG, true, true, 0>(cost) : pick_fleet2<INTEG, false, true, 0>(cost);
    return philox ? pick_fleet2<INTEG, true, false, 0>(cost) : pick_fleet2<INTEG, false, false, 0>(cost);
}
static fleet_fn pick_fleet(int integ, int cost, bool philox, bool pair, bool n10) {
    return integ == CPS_EULER_V0 ? pick_fleet1<0>(cost, philox, pair, n10) : pick_fleet1<1>(cost, philox, pair, n10);
}

extern "C" int cps_fleet_create(cps_handle *h, const cps_fleet_config *cfg) {
    if (!h) return CPS_ERR_INVALID;
    if (!cfg || cfg->struct_size != (int)sizeof(cps_fleet_config))
        return fail(h, CPS_ERR_INVALID, "cps_fleet_create: cps_fleet_config size mismatch");
    if (cfg->n_experiments < 1 || cfg->sim_substeps < 1 || !(cfg->dt_simulation > 0.0))
        return fail(h, CPS_ERR_INVALID, "cps_fleet_create: need n_experiments >= 1, sim_substeps >= 1, dt_simulation > 0");
    if (cfg->noise_source != CPS_FLEET_NOISE_SUPPLIED && cfg->noise_source != CPS_FLEET_NOISE_PHILOX)
        return fail(h, CPS_ERR_INVALID, "cps_fleet_create: unknown noise source %d", cfg->noise_source);
    if (h->cfg.cost_id == CPS_COST_NONE) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_fleet_create: the handle has no cost function");
    if (h->cfg.noise_mode != CPS_NOISE_INDUCING)
        return fail(h, CPS_ERR_UNSUPPORTED, "cps_fleet_create: fleets use inducing-point noise (CPS_NOISE_INDUCING)");
    if (cfg->n_experiments > 65535) return fail(h, CPS_ERR_INVALID, "cps_fleet_create: at most 65535 experiments per handle");
    const bool neural = h->cfg.integrator == CPS_PREDICTOR_NEURAL;
    NetFleetPlan p;
    int rc;
    if (neural && (rc = cps_net_mppi_fleet_plan(h, cfg->n_experiments, "cps_fleet_create", &p)) != CPS_OK) return rc;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    cps_fleet_free(h);
    FleetState *F = new (std::nothrow) FleetState();
    if (!F) return fail(h, CPS_ERR_INVALID, "cps_fleet_create: out of host memory");
    memset(F, 0, sizeof(*F));
    F->cfg = *cfg;
    F->E = cfg->n_experiments;
    const int K = h->cfg.num_rollouts, T = h->cfg.horizon;
    if (neural) {
        // the controller predicts with the loaded network: per experiment a hidden state, partials and tickets for the
        // network kernel's tiling, a draw workspace for Philox
        F->neural = 1;
        F->htot = cps_net_state_size(h);
        F->bpe = p.tiles;
    } else {
        // large fleets are throughput work: two rollouts per thread in packed FP32 (mppi_solve_block2) from 65536 rollouts
        // per launch on, as for a single solve (tools/ab_fleet_pairs.py: 14 % faster at E = 256 and 1024, 30 % slower at E <= 16)
        F->pair = (K % 2 == 0 && K >= 64 && (long long)cfg->n_experiments * K >= CPS_MPPI_PAIR_MIN_ROLLOUTS &&
                   !(h->cfg.flags & CPS_FLAG_NO_PAIRS)) ? 1 : 0;
        const int threads = F->pair ? K / 2 : K;   // threads per experiment
        F->block = threads >= 256 ? 256 : ((threads + 31) / 32) * 32;
        F->bpe = (threads + F->block - 1) / F->block;
        MppiParams mp_geo = h->mp;
        const size_t draws = (cfg->noise_source == CPS_FLEET_NOISE_PHILOX) ? (size_t)h->n_ind * F->block * (F->pair ? 2 : 1) : 0;
        F->smem = sizeof(float) * mppi_smem_floats(mp_geo, h->cfg.cost_id, F->block, F->pair ? 2 : 1, draws);
        F->rs_off = mp_geo.rs_off;
        if (F->smem > 200 * 1024) { delete F; return fail(h, CPS_ERR_UNSUPPORTED, "cps_fleet_create: horizon too large for shared memory"); }
    }
    h->fleet = F;
    const size_t E = F->E, hn = F->htot > 0 ? F->htot : 1;
    F->part_cap = E * F->bpe * (h->n_red + 2);
    CUDA_TRY(h, cudaMalloc(&F->d_s, sizeof(float) * E * 8));
    CUDA_TRY(h, cudaMalloc(&F->d_unom, sizeof(float) * E * T));
    CUDA_TRY(h, cudaMalloc(&F->d_uprev, sizeof(float) * E));
    CUDA_TRY(h, cudaMalloc(&F->d_partials, sizeof(float) * F->part_cap));
    CUDA_TRY(h, cudaMalloc(&F->d_tickets, sizeof(unsigned) * E));
    CUDA_TRY(h, cudaMemset(F->d_s, 0, sizeof(float) * E * 8));
    CUDA_TRY(h, cudaMemset(F->d_unom, 0, sizeof(float) * E * T));
    CUDA_TRY(h, cudaMemset(F->d_uprev, 0, sizeof(float) * E));
    CUDA_TRY(h, cudaMemset(F->d_tickets, 0, sizeof(unsigned) * E));
    if (neural) {
        CUDA_TRY(h, cudaMalloc(&F->d_h, sizeof(float) * E * hn));
        CUDA_TRY(h, cudaMemset(F->d_h, 0, sizeof(float) * E * hn));
        if (cfg->noise_source == CPS_FLEET_NOISE_PHILOX) CUDA_TRY(h, cudaMalloc(&F->d_noise, sizeof(float) * E * h->n_ind * K));
    }
    CUDA_TRY(h, cudaDeviceSynchronize());
    return CPS_OK;
}

int fleet_states_to_device(cps_handle *h, const float *s_host, float *s_dev, int E, const char *who) {
    float *tmp = new (std::nothrow) float[(size_t)E * 8];
    if (!tmp) return fail(h, CPS_ERR_INVALID, "%s: out of host memory", who);
    for (int e = 0; e < E; ++e) {
        for (int c = 0; c < 6; ++c) tmp[(size_t)e * 8 + c] = s_host[(size_t)e * 6 + c];
        tmp[(size_t)e * 8 + 6] = tmp[(size_t)e * 8 + 7] = 0.0f;
    }
    cudaError_t er = cudaMemcpyAsync(s_dev, tmp, sizeof(float) * (size_t)E * 8, cudaMemcpyHostToDevice, h->stream);
    if (er == cudaSuccess) er = cudaStreamSynchronize(h->stream);
    delete[] tmp;
    CUDA_TRY(h, er);
    return CPS_OK;
}

int fleet_states_to_host(cps_handle *h, const float *s_dev, float *s_host, int E, const char *who) {
    float *tmp = new (std::nothrow) float[(size_t)E * 8];
    if (!tmp) return fail(h, CPS_ERR_INVALID, "%s: out of host memory", who);
    cudaError_t er = cudaMemcpyAsync(tmp, s_dev, sizeof(float) * (size_t)E * 8, cudaMemcpyDeviceToHost, h->stream);
    if (er == cudaSuccess) er = cudaStreamSynchronize(h->stream);
    if (er == cudaSuccess)
        for (int e = 0; e < E; ++e)
            for (int c = 0; c < 6; ++c) s_host[(size_t)e * 6 + c] = tmp[(size_t)e * 8 + c];
    delete[] tmp;
    CUDA_TRY(h, er);
    return CPS_OK;
}

extern "C" int cps_fleet_set_states(cps_handle *h, const float *s_host, long long period) {
    if (!h) return CPS_ERR_INVALID;
    FleetState *F = h->fleet;
    if (!F) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_fleet_set_states: no fleet (cps_fleet_create)");
    if (!s_host || period < 0) return fail(h, CPS_ERR_INVALID, "cps_fleet_set_states: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaMemsetAsync(F->d_unom, 0, sizeof(float) * (size_t)F->E * h->cfg.horizon, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(F->d_uprev, 0, sizeof(float) * (size_t)F->E, h->stream));
    int rc = fleet_states_to_device(h, s_host, F->d_s, F->E, "cps_fleet_set_states");
    if (rc != CPS_OK) return rc;
    F->period = period;
    if (F->neural && F->htot > 0) {   // every experiment starts from the handle's stored state (what a fresh predictor holds)
        std::vector<float> h0((size_t)F->htot), all((size_t)F->E * F->htot);
        if (F->htot != cps_net_state_size(h))
            return fail(h, CPS_ERR_INVALID, "cps_fleet_set_states: the loaded network's hidden state differs from the fleet's; "
                        "recreate the fleet (cps_fleet_create)");
        if ((rc = cps_net_get_state(h, h0.data())) != CPS_OK) return rc;
        for (int e = 0; e < F->E; ++e) memcpy(&all[(size_t)e * F->htot], h0.data(), sizeof(float) * F->htot);
        CUDA_TRY(h, cudaMemcpyAsync(F->d_h, all.data(), sizeof(float) * all.size(), cudaMemcpyHostToDevice, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    }
    if (F->pm.on) {   // ring = the reference's initial buffer; the first solve sees the true state
        F->pm.pushed = 0;
        fleet_observe_reset_kernel<<<(F->E + 127) / 128, 128, 0, h->stream>>>(F->pm, F->d_s, F->E);
        h->launches += 1;
        CUDA_TRY(h, cudaGetLastError());
    }
    return CPS_OK;
}

extern "C" int cps_fleet_set_plant_models(cps_handle *h, const cps_fleet_plant_models *m) {
    if (!h) return CPS_ERR_INVALID;
    FleetState *F = h->fleet;
    if (!F) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_fleet_set_plant_models: no fleet (cps_fleet_create)");
    if (F->neural) return fail(h, CPS_ERR_UNSUPPORTED, "cps_fleet_set_plant_models: plant-side models are not offered on fleets "
                               "with the neural predictor");
    if (!m || m->struct_size != (int)sizeof(cps_fleet_plant_models))
        return fail(h, CPS_ERR_INVALID, "cps_fleet_set_plant_models: cps_fleet_plant_models size mismatch");
    if (m->control_noise_mode < 0 || m->control_noise_mode > 2) return fail(h, CPS_ERR_INVALID, "cps_fleet_set_plant_models: control_noise_mode must be 0 (OFF), 1 (additive) or 2 (truncnorm)");
    if (m->control_noise_mode == 2 && !(m->control_noise_mult > 0.0f)) return fail(h, CPS_ERR_INVALID, "cps_fleet_set_plant_models: truncnorm needs a positive scale");
    const double lat_len = m->latency / F->cfg.dt_simulation;
    if (!(m->latency >= 0.0) || lat_len > 200.0)   // MAX_LATENCY_LEN (latency_adder.py:8,74-75)
        return fail(h, CPS_ERR_INVALID, "cps_fleet_set_plant_models: latency must lie in [0, 200 plant ticks]");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    PlantModels &M = F->pm;
    cudaFree(M.obs); cudaFree(M.ring);
    memset(&M, 0, sizeof(M));
    M.ctrl_mode = m->control_noise_mode; M.ctrl_mult = m->control_noise_mult; M.ctrl_add = m->control_noise_add;
    M.meas_on = m->measurement_noise ? 1 : 0;
    M.sig_a = m->sigma_angle; M.sig_p = m->sigma_position; M.sig_aD = m->sigma_angleD; M.sig_pD = m->sigma_positionD;
    M.lat_int = (int)lat_len; M.lat_frac = lat_len - (double)M.lat_int;
    M.ring_len = M.lat_int + 2;
    M.on = (M.ctrl_mode || M.meas_on || m->latency > 0.0) ? 1 : 0;
    if (!M.on) return CPS_OK;
    CUDA_TRY(h, cudaMalloc(&M.obs, sizeof(float) * (size_t)F->E * 8));
    CUDA_TRY(h, cudaMalloc(&M.ring, sizeof(float) * (size_t)F->E * M.ring_len * 6));
    M.pushed = 0;
    fleet_observe_reset_kernel<<<(F->E + 127) / 128, 128, 0, h->stream>>>(M, F->d_s, F->E);
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

extern "C" int cps_fleet_get_observed(cps_handle *h, float *obs_host) {
    if (!h) return CPS_ERR_INVALID;
    FleetState *F = h->fleet;
    if (!F || !F->pm.on) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_fleet_get_observed: no plant-side models (cps_fleet_set_plant_models)");
    if (!obs_host) return fail(h, CPS_ERR_INVALID, "cps_fleet_get_observed: null pointer");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    return fleet_states_to_host(h, F->pm.obs, obs_host, F->E, "cps_fleet_get_observed");
}

extern "C" int cps_fleet_reset(cps_handle *h, long long period) {
    if (!h) return CPS_ERR_INVALID;
    FleetState *F = h->fleet;
    if (!F) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_fleet_reset: no fleet (cps_fleet_create)");
    if (period < 0) return fail(h, CPS_ERR_INVALID, "cps_fleet_reset: period < 0");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaMemsetAsync(F->d_unom, 0, sizeof(float) * (size_t)F->E * h->cfg.horizon, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(F->d_uprev, 0, sizeof(float) * (size_t)F->E, h->stream));
    F->period = period;
    return CPS_OK;
}

extern "C" int cps_fleet_get_states(cps_handle *h, float *s_host, float *u_nom_host, float *u_prev_host) {
    if (!h) return CPS_ERR_INVALID;
    FleetState *F = h->fleet;
    if (!F) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_fleet_get_states: no fleet (cps_fleet_create)");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc;
    if (s_host && (rc = fleet_states_to_host(h, F->d_s, s_host, F->E, "cps_fleet_get_states")) != CPS_OK) return rc;
    if (u_nom_host)
        CUDA_TRY(h, cudaMemcpyAsync(u_nom_host, F->d_unom, sizeof(float) * (size_t)F->E * h->cfg.horizon, cudaMemcpyDeviceToHost, h->stream));
    if (u_prev_host)
        CUDA_TRY(h, cudaMemcpyAsync(u_prev_host, F->d_uprev, sizeof(float) * (size_t)F->E, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}

// [E][htot] hidden states of a neural fleet, host <-> device; synchronises
static int fleet_net_states_io(cps_handle *h, float *host, bool get, const char *who) {
    if (!h) return CPS_ERR_INVALID;
    FleetState *F = h->fleet;
    if (!F || !F->neural) return fail(h, CPS_ERR_NOT_CONFIGURED, "%s: no fleet with the neural predictor (cps_fleet_create)", who);
    if (!host) return fail(h, CPS_ERR_INVALID, "%s: null pointer", who);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t bytes = sizeof(float) * (size_t)F->E * F->htot;
    if (bytes) {
        CUDA_TRY(h, get ? cudaMemcpyAsync(host, F->d_h, bytes, cudaMemcpyDeviceToHost, h->stream)
                        : cudaMemcpyAsync(F->d_h, host, bytes, cudaMemcpyHostToDevice, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    }
    return CPS_OK;
}
extern "C" int cps_fleet_get_net_states(cps_handle *h, float *out_host) {
    return fleet_net_states_io(h, out_host, true, "cps_fleet_get_net_states");
}
extern "C" int cps_fleet_set_net_states(cps_handle *h, const float *in_host) {
    return fleet_net_states_io(h, const_cast<float *>(in_host), false, "cps_fleet_set_net_states");
}

extern "C" long long cps_fleet_period(const cps_handle *h) { return (h && h->fleet) ? h->fleet->period : -1; }

// CostParams for a given target equilibrium: fold_cost() depends on it for quadratic_boundary_grad (weight set, w[9]).
int cps_fold_cost_for(cps_handle *h, float target_equilibrium, CostParams *out);

// The period's draws: supplied by the caller or generated (Philox), as the fleet was created
static int fleet_check_noise(cps_handle *h, const FleetState *F, const float *noise_dev, const char *who) {
    const bool philox = F->cfg.noise_source == CPS_FLEET_NOISE_PHILOX;
    if (!philox && !noise_dev) return fail(h, CPS_ERR_INVALID, "%s: this fleet expects supplied noise", who);
    if (philox && noise_dev) return fail(h, CPS_ERR_INVALID, "%s: this fleet generates its noise (Philox); pass NULL", who);
    return CPS_OK;
}

// Shared by cps_fleet_step (closed loop: replay_dev == nullptr) and cps_fleet_relabel (states from a recording).
static int fleet_launch(cps_handle *h, const char *who, int n_periods, const float *tp_dev, const float *te_dev,
                        const float *noise_dev, float *record_dev, float *J_out_dev, const float *replay_dev,
                        const float *L_dev, const float *mp_dev, float *Q_out_dev, const int *active_dev = nullptr,
                        const float *ctrl_draws_dev = nullptr, const float *meas_draws_dev = nullptr) {
    FleetState *F = h->fleet;
    if (!F) return fail(h, CPS_ERR_NOT_CONFIGURED, "%s: no fleet (cps_fleet_create)", who);
    if (n_periods < 0) return fail(h, CPS_ERR_INVALID, "%s: negative number of periods / rows", who);
    int rc;
    if ((rc = fleet_check_noise(h, F, noise_dev, who)) != CPS_OK) return rc;
    const bool philox = F->cfg.noise_source == CPS_FLEET_NOISE_PHILOX;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    FleetArgs a;
    a.ode = h->ode; a.mp = h->mp;
    a.mp.rs_off = F->rs_off;
    a.pm = F->pm;
    if (replay_dev) a.pm.on = 0;   // relabelling feeds recorded states: no plant, no observation chain
    if (a.pm.on && !philox && ((a.pm.ctrl_mode && !ctrl_draws_dev) || (a.pm.meas_on && !meas_draws_dev)))
        return fail(h, CPS_ERR_INVALID, "%s: a fleet with supplied noise needs the plant-side draws as well (cps_fleet_step_noisy)", who);
    if ((rc = cps_fold_cost_for(h, 1.0f, &a.cost_up)) != CPS_OK) return rc;
    if ((rc = cps_fold_cost_for(h, -1.0f, &a.cost_dn)) != CPS_OK) return rc;
    a.plant = plant_params(h, F->cfg.dt_simulation, F->cfg.sim_substeps);
    a.bpe = F->bpe;
    a.s = F->d_s; a.u_nom = F->d_unom; a.u_prev = F->d_uprev;
    a.seed = F->cfg.seed; a.e_offset = (unsigned)F->cfg.experiment_offset;
    a.partials = F->d_partials; a.tickets = F->d_tickets; a.nonfinite = h->d_nonfinite;
    a.fold = fold_inputs(h);
    if (F->pair && noise_dev && ((uintptr_t)noise_dev % 8) != 0)
        return fail(h, CPS_ERR_INVALID, "%s: supplied noise must be 8-byte aligned", who);
    fleet_fn fn = pick_fleet(h->cfg.integrator, h->cfg.cost_id, philox, F->pair != 0, h->ode.n == 10);
    if (!fn) return fail(h, CPS_ERR_NOT_CONFIGURED, "%s: no kernel for this configuration", who);
    if (F->smem > 48 * 1024) CUDA_TRY(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)F->smem));
    const size_t E = F->E, K = h->cfg.num_rollouts;
    const double dt_control = F->cfg.dt_simulation * F->cfg.sim_substeps;
    const dim3 grid(F->bpe, F->E);
    for (int j = 0; j < n_periods; ++j) {
        a.tp = tp_dev ? tp_dev + (size_t)j * E : nullptr;
        a.te = te_dev ? te_dev + (size_t)j * E : nullptr;
        a.noise = noise_dev ? noise_dev + (size_t)j * E * h->n_ind * K : nullptr;
        a.record = record_dev ? record_dev + (size_t)j * E * CPS_FLEET_RECORD : nullptr;
        a.J_out = J_out_dev ? J_out_dev + (size_t)j * E * K : nullptr;
        a.replay_s = replay_dev ? replay_dev + (size_t)j * E * 6 : nullptr;
        a.L_row = L_dev ? L_dev + (size_t)j * E : nullptr;
        a.mp_row = mp_dev ? mp_dev + (size_t)j * E : nullptr;
        a.Q_out = Q_out_dev ? Q_out_dev + (size_t)j * E : nullptr;
        a.active = active_dev ? active_dev + (size_t)j * E : nullptr;
        if (a.pm.on) {
            a.pm.pushed = F->pm.pushed;
            a.pm.ctrl_draws = ctrl_draws_dev ? ctrl_draws_dev + (size_t)j * E : nullptr;
            a.pm.meas_draws = meas_draws_dev ? meas_draws_dev + (size_t)j * F->cfg.sim_substeps * E * 4 : nullptr;
            F->pm.pushed += F->cfg.sim_substeps;
        }
        a.period = (unsigned)F->period;
        a.time = (double)F->period * dt_control;
        fn<<<grid, F->block, F->smem, h->stream>>>(a);
        F->period += 1;
        h->launches += 1;
    }
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

// cps_fleet_step on a neural fleet: per period [Philox draws ->] the network solve of all experiments -> the plant
static int fleet_step_neural(cps_handle *h, int n_periods, const float *tp_dev, const float *te_dev, const float *noise_dev,
                             float *record_dev, float *J_out_dev) {
    const char *who = "cps_fleet_step";
    FleetState *F = h->fleet;
    if (n_periods < 0) return fail(h, CPS_ERR_INVALID, "%s: negative number of periods", who);
    int rc;
    if ((rc = fleet_check_noise(h, F, noise_dev, who)) != CPS_OK) return rc;
    const bool philox = F->cfg.noise_source == CPS_FLEET_NOISE_PHILOX;
    NetFleetPlan p;
    if ((rc = cps_net_mppi_fleet_plan(h, F->E, who, &p)) != CPS_OK) return rc;
    if (cps_net_state_size(h) != F->htot)
        return fail(h, CPS_ERR_INVALID, "%s: the loaded network has %d hidden-state floats, the fleet was created for %d; "
                    "recreate the fleet (cps_fleet_create)", who, cps_net_state_size(h), F->htot);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t E = F->E, K = h->cfg.num_rollouts, need = E * p.tiles * (h->n_red + 2);
    if (need > F->part_cap) {   // a different tiling than at create (CPS_TC_ROWS)
        cudaFree(F->d_partials);
        F->d_partials = nullptr;
        F->part_cap = 0;
        CUDA_TRY(h, cudaMalloc(&F->d_partials, sizeof(float) * need));
        F->part_cap = need;
    }
    F->bpe = p.tiles;
    CostParams cost_up, cost_dn;
    if ((rc = cps_fold_cost_for(h, 1.0f, &cost_up)) != CPS_OK) return rc;
    if ((rc = cps_fold_cost_for(h, -1.0f, &cost_dn)) != CPS_OK) return rc;
    NetPlantArgs pa;
    pa.plant = plant_params(h, F->cfg.dt_simulation, F->cfg.sim_substeps);
    pa.s = F->d_s; pa.u = F->d_uprev; pa.E = F->E;
    const double dt_control = F->cfg.dt_simulation * F->cfg.sim_substeps;
    for (int j = 0; j < n_periods; ++j) {
        const float *tp = tp_dev ? tp_dev + (size_t)j * E : nullptr, *te = te_dev ? te_dev + (size_t)j * E : nullptr;
        const float *noise = noise_dev ? noise_dev + (size_t)j * E * h->n_ind * K : F->d_noise;
        if (philox) {   // the draws cps_fleet_noise returns for this period
            fleet_noise_kernel<<<dim3((unsigned)(K + 255) / 256, F->E), 256, 0, h->stream>>>(
                F->cfg.seed, (unsigned)F->period, (unsigned)F->cfg.experiment_offset, F->E, (int)K, h->n_ind, F->d_noise);
            h->launches += 1;
        }
        if ((rc = cps_net_mppi_fleet(h, F->E, p, F->d_s, F->d_unom, F->d_uprev, F->d_h, tp, te, cost_up, cost_dn, noise,
                                     F->d_partials, F->d_tickets, J_out_dev ? J_out_dev + (size_t)j * E * K : nullptr)) != CPS_OK)
            return rc;
        pa.tp = tp; pa.te = te;
        pa.record = record_dev ? record_dev + (size_t)j * E * CPS_FLEET_RECORD : nullptr;
        pa.time = (double)F->period * dt_control;
        if ((rc = fleet_plant_launch(h, pa)) != CPS_OK) return rc;
        F->period += 1;
    }
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

extern "C" int cps_fleet_step(cps_handle *h, int n_periods, const float *tp_dev, const float *te_dev, const float *noise_dev,
                              float *record_dev, float *J_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    if (h->fleet && h->fleet->neural) return fleet_step_neural(h, n_periods, tp_dev, te_dev, noise_dev, record_dev, J_out_dev);
    return fleet_launch(h, "cps_fleet_step", n_periods, tp_dev, te_dev, noise_dev, record_dev, J_out_dev, nullptr, nullptr, nullptr, nullptr);
}

static int fleet_reject_neural(cps_handle *h, const char *who) {
    return fail(h, CPS_ERR_UNSUPPORTED, "%s: not offered on fleets with the neural predictor (no plant-side models, no "
                "relabelling with a network)", who);
}

extern "C" int cps_fleet_step_noisy(cps_handle *h, int n_periods, const float *tp_dev, const float *te_dev, const float *noise_dev,
                                    float *record_dev, float *J_out_dev, const float *ctrl_draws_dev, const float *meas_draws_dev) {
    if (!h) return CPS_ERR_INVALID;
    if (h->fleet && h->fleet->neural) return fleet_reject_neural(h, "cps_fleet_step_noisy");
    if (!h->fleet || !h->fleet->pm.on)
        return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_fleet_step_noisy: no plant-side models (cps_fleet_set_plant_models)");
    return fleet_launch(h, "cps_fleet_step_noisy", n_periods, tp_dev, te_dev, noise_dev, record_dev, J_out_dev, nullptr, nullptr, nullptr,
                        nullptr, nullptr, ctrl_draws_dev, meas_draws_dev);
}

extern "C" int cps_fleet_relabel(cps_handle *h, int n_rows, const float *states_dev, const float *tp_dev, const float *te_dev,
                                 const float *L_dev, const float *m_pole_dev, const float *noise_dev, float *Q_out_dev,
                                 float *J_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    if (h->fleet && h->fleet->neural) return fleet_reject_neural(h, "cps_fleet_relabel");
    if (!states_dev || !Q_out_dev) return fail(h, CPS_ERR_INVALID, "cps_fleet_relabel: null pointer");
    return fleet_launch(h, "cps_fleet_relabel", n_rows, tp_dev, te_dev, noise_dev, nullptr, J_out_dev, states_dev, L_dev, m_pole_dev, Q_out_dev);
}

extern "C" int cps_fleet_relabel_masked(cps_handle *h, int n_rows, const float *states_dev, const float *tp_dev, const float *te_dev,
                                        const float *L_dev, const float *m_pole_dev, const float *noise_dev, float *Q_out_dev,
                                        float *J_out_dev, const int *active_dev) {
    if (!h) return CPS_ERR_INVALID;
    if (h->fleet && h->fleet->neural) return fleet_reject_neural(h, "cps_fleet_relabel_masked");
    if (!states_dev || !Q_out_dev) return fail(h, CPS_ERR_INVALID, "cps_fleet_relabel_masked: null pointer");
    return fleet_launch(h, "cps_fleet_relabel_masked", n_rows, tp_dev, te_dev, noise_dev, nullptr, J_out_dev, states_dev, L_dev,
                        m_pole_dev, Q_out_dev, active_dev);
}

extern "C" int cps_fleet_noise(cps_handle *h, long long period, float *out_dev) {
    if (!h) return CPS_ERR_INVALID;
    FleetState *F = h->fleet;
    if (!F) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_fleet_noise: no fleet (cps_fleet_create)");
    if (!out_dev || period < 0) return fail(h, CPS_ERR_INVALID, "cps_fleet_noise: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const int K = h->cfg.num_rollouts;
    const dim3 grid((K + 255) / 256, F->E);
    fleet_noise_kernel<<<grid, 256, 0, h->stream>>>(F->cfg.seed, (unsigned)period, (unsigned)F->cfg.experiment_offset, F->E, K,
                                                    h->n_ind, out_dev);
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}
