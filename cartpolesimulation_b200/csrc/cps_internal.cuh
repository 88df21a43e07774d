// cps_internal.cuh -- declarations shared by the translation units of libcps_b200.so (not part of the ABI).
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>

#include "../../include/cps.h"
#include "cps_device.cuh"

using namespace cps;

// =====================================================================================================
// kernel argument blocks (passed by value: they live in the constant bank)
// =====================================================================================================
struct MppiArgs {
    OdeParams ode;
    CostParams cost;
    MppiParams mp;
    SolveIO io;
    float s_inline[6];   // cps_mppi_step_host: the state travels in the parameter block (no host-to-device copy)
    int use_inline;
};

typedef void (*mppi_fn)(const MppiArgs);
static inline int sc_mode(unsigned flags) {
    if (flags & CPS_FLAG_SUBSTEP_SINCOS) return (flags & CPS_FLAG_FAST_SINCOS) ? SC_MUFU : SC_ACCURATE;
    return SC_ROTATE;
}

struct RolloutArgs {
    OdeParams ode;
    const float *s0;
    long long ss_b;          // 6 if batched, 0 if one shared state
    const float *Q;
    long long qs_b, qs_t;
    int B, T;
    float *traj_out;
    long long ts_k, ts_t, ts_c;
    float *final_out;        // [B][6] or null
};

struct CostArgs {
    CostParams cost;
    const float *traj;       // [K][rows][6], rows = T+1 (or T for get_stage_cost on states[:, :-1])
    const float *Q;          // [K][T]
    float u_prev;
    int K, T, rows;
    float inv_T1;
    float *J;                // [K] or null
    float *stage;            // [K][T] or null
    int unshifted;
};

struct FinalizeArgs {
    MppiParams mp;
    const float *partials;   // [n_parts][2 + n_red]
    int n_parts;
    float *u_nom;
    float *u_out;
    float *shard_out;
};


struct NetState;    // cps_net.cu
struct FleetState;  // cps_fleet.cu
struct RpgdFleetState;  // cps_rpgd_fleet.cu
struct CemFleetState;   // cps_cem_fleet.cu
struct ForwardFleetState;   // cps_forward_fleets.cu
struct LegacyFleetState;    // cps_legacy.cu
struct PlanState;  // cps_plan.cu
struct GmmState;    // cps_gmm.cu
struct GradState;   // cps_grad.cu

struct cps_handle {
    cps_config cfg;
    int n_ind, n_red;
    float phys[CPS_PH_COUNT];
    float cost_in[24];
    int cost_in_n;
    float mppi_in[7];  // cc_weight, R, LBD, NU, sigma, lo, hi
    float target_position, target_equilibrium, L_var, m_pole_var;
    OdeParams ode;
    CostParams cost;
    MppiParams mp;
    cudaStream_t stream;
    // scratch owned by the handle
    float *d_partials;
    unsigned *d_ticket;
    int *d_nonfinite;
    float *d_s, *d_unom, *d_u;
    float *d_uprev;   // legacy front-end: previous nominal sequence [T]
    float *d_ldu;     // legacy front-end: staging of delta_u for cps_legacy_step_host [K][T]
    float *d_lknots;  // legacy front-end: knot draws of the interpolated sampler [K][n_knots]
    size_t n_lknots;  // bytes allocated at d_lknots
    float *h_pin;  // pinned: [0..6) s, [8] u
    float *h_pin_dev;        // device view of h_pin (mapped): the solve writes u straight into host memory
    const float *inline_s;   // set by solve_host around the launch of a solve that reads its state inline
    int grid, block;
    size_t smem;
    int shard;
    float *shard_out;
    // growable buffers of cps_rollout_host
    float *d_rs0, *d_rQ, *d_rtraj, *d_rfinal;
    size_t cap_rs0, cap_rQ, cap_rtraj, cap_rfinal;
    // cps_rollout_host pipeline: copy-in / copy-out streams and per-chunk events (created on first use)
    cudaStream_t st_in, st_out;
    cudaEvent_t ev_start, ev_in[16], ev_k[16];
    int pipe_ready;
    long long launches;
    int net_last_kernel;       // 0 none, 1 net_kernel (FP32), 2 net_tc_kernel
    int rollout_last_kernel;   // 0 none, 1 rollout_kernel, 2 rollout_pair_kernel
    PeerExchange px;           // cps_mppi_set_peers (world <= 1: off); px.epoch = solves exchanged so far
    int *d_px_timeouts;
    std::string err;
    NetState *net;      // neural predictor (cps_net_load), owned
    FleetState *fleet;  // closed-loop experiments (cps_fleet_create), owned
    PlanState *plan;    // forward-only planners (cps_plan_*, cps_cem_*), owned
    GmmState *gmm;      // CEM with a Gaussian-mixture sampling distribution (cps_cem_gmm_*), owned
    GradState *grad;    // adjoint workspace and Adam moments (cps_plan_cost_grad, cps_rpgd_*), owned
    RpgdFleetState *rfleet;  // closed-loop experiments under RPGD (cps_rpgd_fleet_create), owned
    CemFleetState *cfleet;   // closed-loop experiments under CEM (cps_cem_fleet_create), owned
    ForwardFleetState *gfleet;   // ... under CEM-GMM (cps_cem_gmm_fleet_create), owned
    ForwardFleetState *rafleet;  // ... under random action (cps_random_action_fleet_create), owned
    LegacyFleetState *lfleet;    // ... under the legacy controller_mppi_cartpole (cps_legacy_fleet_create), owned
};

extern thread_local std::string g_create_err;

// Dynamic shared memory (in floats) of mppi_solve_block / mppi_solve_block2 for a block of `block` threads carrying
// `per_thread` rollouts each: [T] shifted nominal inputs, 2 [p] tent weights, reduction scratch, `extra` floats the
// caller appends (fleet: Philox draws) and, for the MAX_COST plugins, the row-sum slots (cps_device.cuh RowSumPlan).
// Sets mp.rs_off.
static inline size_t mppi_smem_floats(MppiParams &mp, int cost_id, int block, int per_thread, size_t extra = 0) {
    size_t fl = (size_t)mp.T + 2 * (size_t)mp.p + (size_t)(block / 32) * (mp.n_red + 2) + (size_t)mp.n_red + 4;
    fl = ((fl + 1) & ~(size_t)1) + ((extra + 1) & ~(size_t)1);
    mp.rs_off = (int)fl;
    if (cost_id == CPS_COST_DEFAULT || cost_id == CPS_COST_QUADRATIC_BOUNDARY)
        fl += (size_t)row_sum_slots(mp.T + 1) * block * per_thread;
    return fl;
}

// cps_fleet.cu
void cps_fleet_free(cps_handle *h);
// cps_rpgd_fleet.cu
void cps_rpgd_fleet_free(cps_handle *h);
// cps_cem_fleet.cu
void cps_cem_fleet_free(cps_handle *h);
// cps_forward_fleets.cu
void cps_forward_fleets_free(cps_handle *h);
// cps_legacy.cu
void cps_legacy_fleet_free(cps_handle *h);
// cps_plan.cu
void cps_plan_free(cps_handle *h);
// the refusals every forward-only planner shares: no cost plugin, substep sin/cos or fast division; with the neural
// predictor those of cps_plan_cost on a network (cps_net_plan_check) and K above the single-block selection
int cps_plan_check(cps_handle *h, const char *who);
// CEM fleets: the refusals of cps_cem_fleet_create that concern the planner (those of cps_cem_configure, K above the
// single-block selection, shared memory of plan_fleet_kernel), and one outer iteration of E experiments: plan_fleet_kernel,
// then cem_update_fleet_kernel when best_k x T > 2048 (h->launches counts them)
struct CemFleetIteration {
    int E, best_k, last_iter;
    float sd_init, sd_min;
    const float *s;              // [E][8] states
    float *u;                    // [E] u_prev of the costs; <- u = elite_Q[0, 0] after the last iteration
    const float *tp, *te;        // [E] targets of this period (null: 0 / +1)
    CostParams cost_up, cost_dn; // folded for target_equilibrium = +1 / -1
    const float *mu, *sd;        // [E][T] the distribution the plans are drawn from
    float *mu_out, *sd_out;      // [E][T] <- the updated one (clipped and shifted after the last iteration)
    const float *eps;            // [E][T][K] supplied draws, or null: Philox, counter (plan, w1 + group, period, e_offset + e)
    unsigned long long seed;
    unsigned w1, period, e_offset;
    float *J;                    // [E][K] <- the costs
    float *Q_out;                // [E][T][K] <- the plans, or null
    int *elite;                  // [E][K] scratch of the deferred statistics
    unsigned *tickets;           // [E], zero between launches
    float *P;                    // neural predictor: [E][K][T] scratch, the sampled plans net_grad_kernel reads
    CostParams *costs;           // neural predictor: [E] scratch, the folded cost parameters of this period
};
int cps_cem_fleet_check(cps_handle *h, int best_k, float initial_stdev, float stdev_min, int philox, const char *who);
int cps_cem_fleet_iteration(cps_handle *h, const CemFleetIteration &c);
// CEM-GMM and random-action fleets (cps_forward_fleets.cu): the refusals of their creates that concern the planner (gmm:
// those of cps_cem_gmm_configure; both: K above the single-block selection, shared memory of the rollout kernel), and the
// rollouts of one iteration of E experiments, one launch of plan_forward_fleet_kernel, grid (ceil(K / 256), E).  gmm: the
// plans Q = clip(loc[c][t] + scale[c][t] eps_c) from each experiment's mixture, costs into J, no selection; random action:
// the plans as given (or lo + (hi - lo) u from Philox), costs, and in the last block of each experiment u = Q[argmin J, 0].
struct ForwardFleetRollouts {
    int gmm, E;
    const float *s;              // [E][8] states
    float *u;                    // [E] u_prev of the costs; random action: <- u
    const float *tp, *te;        // [E] targets of this period (null: 0 / +1)
    CostParams cost_up, cost_dn; // folded for target_equilibrium = +1 / -1
    const float *dist;           // gmm: [E][4T + 1] loc[2][T], scale[2][T], p1 the plans are drawn from
    const float *Q;              // supplied: random action plans [E][T][K]; gmm normals [E][2][T][K]; null: Philox
    const float *u01;            // gmm, supplied: uniforms [E][T][K]
    unsigned long long seed;     // Philox: counter (plan, w1 + draw word, period, e_offset + e), cps_plant.cuh
    unsigned w1, period, e_offset;
    float *J;                    // [E][K] <- the costs
    float *Q_out;                // [E][T][K] <- the plans, or null
    unsigned *tickets;           // [E], zero between launches (random action)
    float *P;                    // neural predictor: [E][K][T] scratch, the sampled plans net_grad_kernel reads
    CostParams *costs;           // neural predictor: [E] scratch, the folded cost parameters of this period
};
int cps_forward_fleet_check(cps_handle *h, int gmm, int best_k, float initial_stdev, float stdev_min, const char *who);
int cps_forward_fleet_rollouts(cps_handle *h, const ForwardFleetRollouts &c);
// cps_gmm.cu
void cps_gmm_free(cps_handle *h);
// CEM-GMM fleets: the selection and update of one iteration for E experiments, gmm_update_fleet_kernel, grid E, per
// experiment the arithmetic of gmm_update_kernel in the same order
struct GmmFleetUpdate {
    int E, K, T, best_k, last_iter;
    float lo, hi, sd_min;
    const float *J;              // [E][K] the costs
    const float *dist;           // [E][4T + 1] the mixture the plans were drawn from
    float *dist_out;             // [E][4T + 1] <- the update (shifted after the last iteration)
    const float *eps, *u01;      // supplied draws of this iteration [E][2][T][K], [E][T][K], or null: Philox
    unsigned long long seed;
    unsigned w1, period, e_offset;
    int *elite;                  // [E][2K] scratch: elite indices, cluster flags
    float *rows;                 // [E][best_k][T] scratch: the elites' plans
    float *u;                    // [E] <- u = elite_Q[0, 0] after the last iteration
};
int cps_gmm_fleet_update(cps_handle *h, const GmmFleetUpdate &a);
// cps_grad.cu
#define CPS_GRAD_REC 20   /* floats per (control step, plan) record: M[3][4], r[4], cost partials (3), control term */
void cps_grad_free(cps_handle *h);
// the RPGD fleet's gradient (G != nullptr; ck [T][4][n_plans], jac [T][CPS_GRAD_REC][n_plans]) or costs (G == nullptr) of
// n_plans = E * kpe plans [n_plans][T] from the fleet's states [E][8], per-experiment cost parameters and u_prev [E];
// odes_dev [E] per-experiment model constants (relabelling with per-row L / m_pole) or nullptr (the handle's)
int cps_grad_fleet(cps_handle *h, int n_plans, int kpe, const float *s_dev, const float *Q_dev, const CostParams *costs_dev,
                   const float *u_prev_dev, float *ck, float *jac, float *J, float *G, const OdeParams *odes_dev = nullptr);
int cps_grad_fleet_update(cps_handle *h, int n_plans, float *Q_dev, const float *G_dev, float *m_dev, float *v_dev, float lr_t,
                          float beta_1, float beta_2, float epsilon, float gradmax_clip);
// cps_lib.cu: cost parameters folded for a given target equilibrium
int cps_fold_cost_for(cps_handle *h, float target_equilibrium, CostParams *out);
// cps_net.cu
void cps_net_free(cps_handle *h);
// cps_net_grad.cu: cps_plan_cost / cps_plan_cost_grad with CPS_PREDICTOR_NEURAL
int cps_net_plan_cost(cps_handle *h, const float *s_dev, const float *Q_dev, int q_layout, int K, int T, float u_prev,
                      float *J_out_dev, float *traj_out_dev, int traj_layout);
int cps_net_plan_cost_grad(cps_handle *h, const float *s_dev, const float *Q_dev, int q_layout, float u_prev, float *J_out_dev,
                           float *G_out_dev);
// the refusals of cps_plan_cost with CPS_PREDICTOR_NEURAL (no network, D_* network, plugin, tensor-core flag, shared memory)
int cps_net_plan_check(cps_handle *h, const char *who);
// the RPGD fleet with CPS_PREDICTOR_NEURAL: cps_net_grad_fleet_prepare runs the network checks of cps_plan_cost_grad and
// sizes the workspace for E experiments; cps_net_grad_fleet is net_grad_kernel over E experiments x K plans [E][K][T] from
// the fleet's states [E][8], per-experiment cost parameters and u_prev [E]: the gradient (G != nullptr, J and G [E][K][T])
// or the costs only (G == nullptr), per plan bit-identical to cps_plan_cost_grad / cps_plan_cost
int cps_net_grad_fleet_prepare(cps_handle *h, int E, const char *who);
int cps_net_grad_fleet(cps_handle *h, int E, const float *s_dev, const float *Q_dev, const CostParams *costs_dev,
                       const float *u_prev_dev, float *J_dev, float *G_dev, const char *who);   // who: for the messages
int cps_net_mppi_step(cps_handle *h, const float *s_dev, const float *noise_dev, int noise_layout, float u_prev,
                      float *u_nom_dev, float *u_out_dev, float *J_out_dev, float *traj_out_dev, int traj_layout,
                      float *u_run_out_dev);
// the MPPI fleet with CPS_PREDICTOR_NEURAL: cps_net_mppi_fleet_plan runs the network checks of cps_mppi_step and picks the
// kernel (kernel 1 net_kernel, 2 net_tc_kernel), its rollouts per CTA, CTAs per experiment and shared memory;
// cps_net_mppi_fleet is one launch of that kernel over E experiments x K rollouts, per experiment the arithmetic of
// cps_mppi_step: states [E][8], warm starts [E][T], u_prev [E] (<- u), hidden states [E][htot] (advanced on (u, s)),
// draws [E][n_ind][K], partials [E][tiles][2 + n_red], tickets [E], J_out [E][K] or null
struct NetFleetPlan { int kernel, rows, tiles; size_t smem; };
int cps_net_mppi_fleet_plan(cps_handle *h, int E, const char *who, NetFleetPlan *p);
int cps_net_mppi_fleet(cps_handle *h, int E, const NetFleetPlan &p, const float *s_dev, float *u_nom_dev, float *u_prev_dev,
                       float *hid_dev, const float *tp_dev, const float *te_dev, const CostParams &cost_up, const CostParams &cost_dn,
                       const float *noise_dev, float *partials_dev, unsigned *tickets_dev, float *J_out_dev);

static inline int fail(cps_handle *h, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (h) h->err = buf;
    else g_create_err = buf;
    return code;
}

#define CUDA_TRY(h, expr)                                                                          \
    do {                                                                                           \
        cudaError_t e_ = (expr);                                                                   \
        if (e_ != cudaSuccess) return fail(h, CPS_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e_)); \
    } while (0)

// ---- host form of a solve (the *_host entry points) --------------------------------------------------------------------
// The argument blocks of MppiArgs / PlanArgs carry the state of a host-form solve when h->inline_s is set.
template <class Args>
static inline void fill_inline_state(const cps_handle *h, Args &a) {
    a.use_inline = h->inline_s ? 1 : 0;
    for (int c = 0; c < 6; ++c) a.s_inline[c] = h->inline_s ? h->inline_s[c] : 0.0f;
}

// The u-return half: u_dev is h->d_u (copied back) or the mapped h_pin_dev + 8 (already in host memory); synchronises.
static inline int return_u_host(cps_handle *h, const float *u_dev, float *u_out_host) {
    if (u_dev == h->d_u) CUDA_TRY(h, cudaMemcpyAsync(h->h_pin + 8, h->d_u, sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    *u_out_host = h->h_pin[8];
    return CPS_OK;
}

// One host-form solve, after cudaSetDevice: the state goes in, launch(s_dev, u_dev) enqueues the solve, u comes back.
// direct (the kernel reads the state from its parameter block): the state rides inline and, with mapped memory, u is
// written straight into host memory -- one stream operation.  Otherwise the state is copied through h_pin to d_s and u back
// from d_u.
template <class Launch>
static inline int solve_host(cps_handle *h, const float *s_host, float *u_out_host, bool direct, Launch launch) {
    float *u_dev = direct && h->h_pin_dev ? h->h_pin_dev + 8 : h->d_u;
    if (!direct) {
        memcpy(h->h_pin, s_host, sizeof(float) * 6);
        CUDA_TRY(h, cudaMemcpyAsync(h->d_s, h->h_pin, sizeof(float) * 6, cudaMemcpyHostToDevice, h->stream));
    }
    h->inline_s = direct ? s_host : nullptr;
    const int rc = launch((const float *)h->d_s, u_dev);
    h->inline_s = nullptr;
    if (rc != CPS_OK) return rc;
    return return_u_host(h, u_dev, u_out_host);
}

