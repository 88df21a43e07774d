// cps_forward_fleets.cu -- E independent closed-loop experiments under optimizer_cem_gmm_tf or optimizer_random_action_tf
// (Control_Toolkit/Optimizers/optimizer_cem_gmm_tf.py:14-140, optimizer_random_action_tf.py:12-86; `cem-gmm-tf` and
// `random-action-tf` in Control_Toolkit_ASF/config_controllers.yml), advanced together.
//
// One controller period of EVERY experiment, no host round trip (launches independent of E):
//   CEM-GMM, per outer iteration
//     plan_forward_fleet_kernel   (cps_plan.cu), grid (ceil(K / 256), E): each experiment's K plans sampled from its own
//                                 mixture (component c = 0 iff u01 < p1, Q = clip(loc[c] + scale[c] eps_c)) and their
//                                 costs from its state, u_prev and targets;
//     gmm_update_fleet_kernel     (cps_gmm.cu), grid E: the best_k elites, the two clusters around the two cheapest, the
//                                 per-cluster mean / stdev and p1 (gmm_update_kernel's arithmetic); after the last
//                                 iteration the shift and u = elite_Q[0, 0], which becomes the experiment's u_prev;
//   random action
//     plan_forward_fleet_kernel   each experiment's K uniform plans in [lo, hi), their costs, and in the last block of the
//                                 experiment (its own ticket) u = Q[argmin J, 0];
//   fleet_net_plant_kernel        (cps_fleet.cu) the plant period with Q = u and the record row, one thread per experiment.
// Launches per period: 2 x cem_outer_it + 1 (CEM-GMM), 2 (random action).
// With the neural predictor the rollouts are plan_sample_kernel (the plans into [E][K][T], the period's cost parameters
// into [E]) and net_grad_kernel<.., FLEET> (cps_net_grad.cu), and random action takes its argmin in plan_select_kernel,
// one block per experiment: 3 x cem_outer_it + 1 (CEM-GMM), 4 (random action) launches per period.  Every rollout starts
// from the network's stored hidden state; the fleets keep none per experiment.  The mixtures live in [2][E][4T + 1] ping-pong
// buffers (an iteration reads one half and writes the other).  No [E][T][K] plan or draw buffer is materialised on a
// Philox fleet: the update rebuilds the elites' plans, best_k x T per experiment, from the mixture and the regenerated draws.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include "cps_internal.cuh"
#include "cps_plant.cuh"

struct ForwardFleetState {
    FleetCore core;
    int gmm;                          // 1: CEM-GMM, 0: random action
    int K, T;
    int outer_its, best_k;            // CEM-GMM
    float sd_init, sd_min;
    float *d_dist;                    // CEM-GMM: [2][E][4T + 1] ping-pong mixtures loc[2][T], scale[2][T], p1; `cur` is live
    int cur;
    float *d_J;                       // [E][K] costs when the caller does not ask for them
    int *d_elite;                     // CEM-GMM: [E][2K] elite indices and cluster flags
    float *d_rows;                    // CEM-GMM: [E][best_k][T] the elites' plans
    unsigned *d_tickets;              // random action: [E]
    float *d_P;                       // neural predictor: [E][K][T] the sampled plans
    CostParams *d_costs;              // neural predictor: [E] the period's folded cost parameters
};

static void forward_fleet_free(ForwardFleetState *&F) {
    if (!F) return;
    fleet_core_free(F->core);
    cudaFree(F->d_dist); cudaFree(F->d_J); cudaFree(F->d_elite); cudaFree(F->d_rows); cudaFree(F->d_tickets);
    cudaFree(F->d_P); cudaFree(F->d_costs);
    delete F;
    F = nullptr;
}

void cps_forward_fleets_free(cps_handle *h) {
    forward_fleet_free(h->gfleet);
    forward_fleet_free(h->rafleet);
}

// What both creates share once the config struct is checked: the planner's refusals, the header, E <= 65535 (gridDim.y
// of the rollouts), the state and the buffers.
static int forward_fleet_create(cps_handle *h, ForwardFleetState *&slot, int gmm, int n_experiments, int sim_substeps,
                                int source, double dt_simulation, unsigned long long seed, long long experiment_offset,
                                int outer_its, int best_k, float initial_stdev, float stdev_min, const char *who) {
    int rc;
    if ((rc = cps_forward_fleet_check(h, gmm, best_k, initial_stdev, stdev_min, who)) != CPS_OK) return rc;
    FleetCore core;
    if ((rc = fleet_core_init(h, core, n_experiments, sim_substeps, source, dt_simulation, seed, experiment_offset, who)) != CPS_OK)
        return rc;
    if (core.E > 65535) return fail(h, CPS_ERR_INVALID, "%s: at most 65535 experiments per handle", who);
    const int K = h->cfg.num_rollouts, T = h->cfg.horizon;
    if (gmm) {   // the Philox streams of the iterations stay below GMM_DRAWS + 2^28 (cps_plant.cuh)
        const long long max_its = std::min(65535LL, (long long)(1 << 28) / (3 * ((T + 3) / 4)));
        if (outer_its < 1 || outer_its > max_its)
            return fail(h, CPS_ERR_INVALID, "%s: outer_its must lie in [1, %lld]", who, max_its);
    }
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    forward_fleet_free(slot);
    ForwardFleetState *F = new (std::nothrow) ForwardFleetState();
    if (!F) return fail(h, CPS_ERR_INVALID, "%s: out of host memory", who);
    memset(F, 0, sizeof(*F));
    F->core = core;
    F->gmm = gmm;
    F->K = K; F->T = T;
    F->outer_its = outer_its; F->best_k = best_k; F->sd_init = initial_stdev; F->sd_min = stdev_min;
    slot = F;
    const size_t E = core.E;
    if ((rc = fleet_core_alloc(h, F->core)) != CPS_OK) return rc;
    CUDA_TRY(h, cudaMalloc(&F->d_J, sizeof(float) * E * K));
    if (gmm) {
        CUDA_TRY(h, cudaMalloc(&F->d_dist, sizeof(float) * 2 * E * (4 * T + 1)));
        CUDA_TRY(h, cudaMalloc(&F->d_elite, sizeof(int) * E * 2 * K));
        CUDA_TRY(h, cudaMalloc(&F->d_rows, sizeof(float) * E * best_k * T));
    } else {
        CUDA_TRY(h, cudaMalloc(&F->d_tickets, sizeof(unsigned) * E));
        CUDA_TRY(h, cudaMemset(F->d_tickets, 0, sizeof(unsigned) * E));
    }
    if (h->cfg.integrator == CPS_PREDICTOR_NEURAL) {
        CUDA_TRY(h, cudaMalloc(&F->d_P, sizeof(float) * E * K * T));
        CUDA_TRY(h, cudaMalloc(&F->d_costs, sizeof(CostParams) * E));
    }
    return CPS_OK;
}

static int forward_fleet_set_states(cps_handle *h, ForwardFleetState *F, const float *s_host, long long period, const char *who) {
    int rc;
    if ((rc = fleet_core_set_states(h, F->core, s_host, period, who)) != CPS_OK) return rc;
    if (F->gmm) {   // optimizer_reset of every experiment (cem_gmm_tf.py:133-139), as cps_cem_gmm_reset
        const int T = F->T;
        const float mid = (h->mppi_in[5] + h->mppi_in[6]) * 0.5f;
        std::vector<float> d((size_t)F->core.E * (4 * T + 1));
        for (int e = 0; e < F->core.E; ++e) {
            float *de = &d[(size_t)e * (4 * T + 1)];
            for (int t = 0; t < 2 * T; ++t) { de[t] = mid; de[2 * T + t] = F->sd_init; }
            de[4 * T] = 0.5f;
        }
        F->cur = 0;
        CUDA_TRY(h, cudaMemcpyAsync(F->d_dist, d.data(), sizeof(float) * d.size(), cudaMemcpyHostToDevice, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));   // the host vector above is free to go
    }
    F->core.ready = 1;
    return CPS_OK;
}

// n_periods controller periods; draws: CEM-GMM normals (a) and uniforms (b), random action plans (a)
static int forward_fleet_step(cps_handle *h, ForwardFleetState *F, int n_periods, const float *tp_dev, const float *te_dev,
                              const float *a_dev, const float *b_dev, float *record_dev, float *J_out_dev, float *Q_out_dev,
                              const char *who) {
    FleetCore &fc = F->core;
    if (!fc.ready) return fail(h, CPS_ERR_NOT_CONFIGURED, "%s: no states yet (set_states first)", who);
    if (n_periods < 0) return fail(h, CPS_ERR_INVALID, "%s: negative number of periods", who);
    int rc;
    if ((rc = fleet_core_check_draws(h, fc, a_dev, true, who)) != CPS_OK) return rc;
    if (F->gmm && (a_dev == nullptr) != (b_dev == nullptr))
        return fail(h, CPS_ERR_INVALID, "%s: pass both the normals and the uniforms, or neither", who);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t E = fc.E, K = F->K, T = F->T, D = 4 * T + 1;
    const unsigned G4 = (unsigned)((T + 3) / 4);
    ForwardFleetRollouts r;
    memset(&r, 0, sizeof(r));
    if ((rc = fleet_fold_costs(h, &r.cost_up, &r.cost_dn)) != CPS_OK) return rc;
    r.gmm = F->gmm; r.E = fc.E;
    r.s = fc.d_s; r.u = fc.d_uprev;
    r.seed = fc.seed; r.e_offset = fc.e_offset;
    r.tickets = F->d_tickets;
    r.P = F->d_P; r.costs = F->d_costs;
    GmmFleetUpdate g;
    memset(&g, 0, sizeof(g));
    g.E = fc.E; g.K = F->K; g.T = F->T; g.best_k = F->best_k;
    g.lo = h->mppi_in[5]; g.hi = h->mppi_in[6]; g.sd_min = F->sd_min;
    g.seed = fc.seed; g.e_offset = fc.e_offset;
    g.elite = F->d_elite; g.rows = F->d_rows; g.u = fc.d_uprev;
    NetPlantArgs pa;
    memset(&pa, 0, sizeof(pa));
    pa.plant = plant_params(h, fc.dt_sim, fc.n_sim);
    pa.s = fc.d_s; pa.u = fc.d_uprev; pa.E = fc.E;
    const float *da = a_dev, *db = b_dev;   // supplied draws of all periods, back to back
    for (int j = 0; j < n_periods; ++j) {
        const FleetRow row = fleet_core_row(fc, j, tp_dev, te_dev, record_dev);
        r.tp = row.tp; r.te = row.te; r.period = row.period;
        float *J_j = J_out_dev ? J_out_dev + (size_t)j * E * K : nullptr;
        float *Q_j = Q_out_dev ? Q_out_dev + (size_t)j * E * T * K : nullptr;
        if (F->gmm) {
            g.period = row.period;
            for (int i = 0; i < F->outer_its; ++i) {
                const int last = (i == F->outer_its - 1) ? 1 : 0;
                r.dist = F->d_dist + (size_t)F->cur * E * D;
                r.Q = da ? da + (size_t)i * E * 2 * T * K : nullptr;
                r.u01 = db ? db + (size_t)i * E * T * K : nullptr;
                r.w1 = g.w1 = GMM_DRAWS + (unsigned)i * 3 * G4;
                // J / Q of the last iteration (cem_gmm_tf.py:104-105) go to the caller's arrays when given
                r.J = (last && J_j) ? J_j : F->d_J;
                r.Q_out = last ? Q_j : nullptr;
                if ((rc = cps_forward_fleet_rollouts(h, r)) != CPS_OK) return rc;
                g.last_iter = last;
                g.J = r.J; g.dist = r.dist; g.dist_out = F->d_dist + (size_t)(1 - F->cur) * E * D;
                g.eps = r.Q; g.u01 = r.u01;
                if ((rc = cps_gmm_fleet_update(h, g)) != CPS_OK) return rc;
                F->cur = 1 - F->cur;
            }
            if (da) { da += (size_t)F->outer_its * E * 2 * T * K; db += (size_t)F->outer_its * E * T * K; }
        } else {
            r.Q = da ? da + (size_t)j * E * T * K : nullptr;
            r.w1 = RA_DRAWS;
            r.J = J_j ? J_j : F->d_J;
            r.Q_out = Q_j;
            if ((rc = cps_forward_fleet_rollouts(h, r)) != CPS_OK) return rc;
        }
        pa.tp = row.tp; pa.te = row.te; pa.record = row.record; pa.time = row.time;
        if ((rc = fleet_plant_launch(h, pa)) != CPS_OK) return rc;
        fc.period += 1;
    }
    return CPS_OK;
}

// ---- CEM-GMM ------------------------------------------------------------------------------------------------------------
static ForwardFleetState *gmm_fleet(cps_handle *h, const char *who) {
    ForwardFleetState *F = h->gfleet;
    if (!F) fail(h, CPS_ERR_NOT_CONFIGURED, "%s: no CEM-GMM fleet (cps_cem_gmm_fleet_create)", who);
    return F;
}
static ForwardFleetState *gmm_fleet_ready(cps_handle *h, const char *who) {
    ForwardFleetState *F = h->gfleet;
    if (!F || !F->core.ready)
        fail(h, CPS_ERR_NOT_CONFIGURED, "%s: no CEM-GMM fleet with states (cps_cem_gmm_fleet_create, cps_cem_gmm_fleet_set_states)", who);
    return F && F->core.ready ? F : nullptr;
}

extern "C" int cps_cem_gmm_fleet_create(cps_handle *h, const cps_cem_gmm_fleet_config *cfg) {
    if (!h) return CPS_ERR_INVALID;
    const char *who = "cps_cem_gmm_fleet_create";
    if (!cfg || cfg->struct_size != (int)sizeof(cps_cem_gmm_fleet_config))
        return fail(h, CPS_ERR_INVALID, "%s: cps_cem_gmm_fleet_config size mismatch", who);
    return forward_fleet_create(h, h->gfleet, 1, cfg->n_experiments, cfg->sim_substeps, cfg->draw_source, cfg->dt_simulation,
                                cfg->seed, cfg->experiment_offset, cfg->outer_its, cfg->best_k, cfg->initial_stdev,
                                cfg->stdev_min, who);
}

extern "C" int cps_cem_gmm_fleet_set_states(cps_handle *h, const float *s_host, long long period) {
    if (!h) return CPS_ERR_INVALID;
    ForwardFleetState *F = gmm_fleet(h, "cps_cem_gmm_fleet_set_states");
    return F ? forward_fleet_set_states(h, F, s_host, period, "cps_cem_gmm_fleet_set_states") : CPS_ERR_NOT_CONFIGURED;
}

extern "C" int cps_cem_gmm_fleet_get_states(cps_handle *h, float *s_host, float *u_prev_host) {
    if (!h) return CPS_ERR_INVALID;
    ForwardFleetState *F = gmm_fleet_ready(h, "cps_cem_gmm_fleet_get_states");
    return F ? fleet_core_get_states(h, F->core, s_host, u_prev_host, "cps_cem_gmm_fleet_get_states") : CPS_ERR_NOT_CONFIGURED;
}

extern "C" int cps_cem_gmm_fleet_get_distribution(cps_handle *h, float *loc_host, float *scale_host, float *p1_host) {
    if (!h) return CPS_ERR_INVALID;
    ForwardFleetState *F = gmm_fleet_ready(h, "cps_cem_gmm_fleet_get_distribution");
    if (!F) return CPS_ERR_NOT_CONFIGURED;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t E = F->core.E, T = F->T, D = 4 * T + 1;
    std::vector<float> d(E * D);
    CUDA_TRY(h, cudaMemcpyAsync(d.data(), F->d_dist + (size_t)F->cur * E * D, sizeof(float) * d.size(), cudaMemcpyDeviceToHost,
                                h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    for (size_t e = 0; e < E; ++e) {
        if (loc_host) memcpy(loc_host + e * 2 * T, &d[e * D], sizeof(float) * 2 * T);
        if (scale_host) memcpy(scale_host + e * 2 * T, &d[e * D + 2 * T], sizeof(float) * 2 * T);
        if (p1_host) p1_host[e] = d[e * D + 4 * T];
    }
    return CPS_OK;
}

extern "C" int cps_cem_gmm_fleet_step(cps_handle *h, int n_periods, const float *tp_dev, const float *te_dev,
                                      const float *eps_dev, const float *u01_dev, float *record_dev, float *J_out_dev,
                                      float *Q_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    const char *who = "cps_cem_gmm_fleet_step";
    ForwardFleetState *F = gmm_fleet(h, who);
    if (!F) return CPS_ERR_NOT_CONFIGURED;
    return forward_fleet_step(h, F, n_periods, tp_dev, te_dev, eps_dev, u01_dev, record_dev, J_out_dev, Q_out_dev, who);
}

// eps_out [n_it][E][2][T][K], u01_out [n_it][E][T][K]: what the rollouts of `period` draw (either may be null)
extern "C" int cps_cem_gmm_fleet_draws(cps_handle *h, long long period, float *eps_out_dev, float *u01_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    ForwardFleetState *F = gmm_fleet_ready(h, "cps_cem_gmm_fleet_draws");
    if (!F) return CPS_ERR_NOT_CONFIGURED;
    if (period < 0) return fail(h, CPS_ERR_INVALID, "cps_cem_gmm_fleet_draws: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const FleetCore &c = F->core;
    const int K = F->K, T = F->T;
    const unsigned G4 = (unsigned)((T + 3) / 4);
    const long long ETK = (long long)c.E * T * K;
    int rc;
    for (int it = 0; eps_out_dev && it < F->outer_its; ++it) {   // layer = component
        const FleetDrawsArgs d = {c.seed, GMM_DRAWS + (unsigned)it * 3 * G4, G4, (unsigned)period, c.e_offset, c.E, K, T,
                                  (long long)T * K, 2LL * T * K, 1, K, eps_out_dev + (size_t)it * 2 * ETK};
        if ((rc = fleet_draws_launch(h, d, 2)) != CPS_OK) return rc;
    }
    if (u01_out_dev) {   // layer = iteration
        const FleetDrawsArgs d = {c.seed, GMM_DRAWS + 2 * G4, 3 * G4, (unsigned)period, c.e_offset, c.E, K, T, ETK,
                                  (long long)T * K, 1, K, u01_out_dev};
        if ((rc = fleet_uniforms_launch(h, d, F->outer_its, 0.0f, 1.0f)) != CPS_OK) return rc;
    }
    return CPS_OK;
}

extern "C" long long cps_cem_gmm_fleet_period(const cps_handle *h) { return (h && h->gfleet) ? h->gfleet->core.period : -1; }

// ---- random action ------------------------------------------------------------------------------------------------------
static ForwardFleetState *ra_fleet(cps_handle *h, const char *who, bool ready) {
    ForwardFleetState *F = h->rafleet;
    if (!F || (ready && !F->core.ready)) {
        fail(h, CPS_ERR_NOT_CONFIGURED, "%s: no random-action fleet%s", who,
             ready ? " with states (cps_random_action_fleet_create, cps_random_action_fleet_set_states)"
                   : " (cps_random_action_fleet_create)");
        return nullptr;
    }
    return F;
}

extern "C" int cps_random_action_fleet_create(cps_handle *h, const cps_random_action_fleet_config *cfg) {
    if (!h) return CPS_ERR_INVALID;
    const char *who = "cps_random_action_fleet_create";
    if (!cfg || cfg->struct_size != (int)sizeof(cps_random_action_fleet_config))
        return fail(h, CPS_ERR_INVALID, "%s: cps_random_action_fleet_config size mismatch", who);
    return forward_fleet_create(h, h->rafleet, 0, cfg->n_experiments, cfg->sim_substeps, cfg->draw_source, cfg->dt_simulation,
                                cfg->seed, cfg->experiment_offset, 1, 0, 0.0f, 0.0f, who);
}

extern "C" int cps_random_action_fleet_set_states(cps_handle *h, const float *s_host, long long period) {
    if (!h) return CPS_ERR_INVALID;
    ForwardFleetState *F = ra_fleet(h, "cps_random_action_fleet_set_states", false);
    return F ? forward_fleet_set_states(h, F, s_host, period, "cps_random_action_fleet_set_states") : CPS_ERR_NOT_CONFIGURED;
}

extern "C" int cps_random_action_fleet_get_states(cps_handle *h, float *s_host, float *u_prev_host) {
    if (!h) return CPS_ERR_INVALID;
    ForwardFleetState *F = ra_fleet(h, "cps_random_action_fleet_get_states", true);
    return F ? fleet_core_get_states(h, F->core, s_host, u_prev_host, "cps_random_action_fleet_get_states")
             : CPS_ERR_NOT_CONFIGURED;
}

extern "C" int cps_random_action_fleet_step(cps_handle *h, int n_periods, const float *tp_dev, const float *te_dev,
                                            const float *plans_dev, float *record_dev, float *J_out_dev, float *Q_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    const char *who = "cps_random_action_fleet_step";
    ForwardFleetState *F = ra_fleet(h, who, false);
    if (!F) return CPS_ERR_NOT_CONFIGURED;
    return forward_fleet_step(h, F, n_periods, tp_dev, te_dev, plans_dev, nullptr, record_dev, J_out_dev, Q_out_dev, who);
}

// out_dev [E][T][K]: the plans a Philox fleet evaluates in `period`
extern "C" int cps_random_action_fleet_draws(cps_handle *h, long long period, float *out_dev) {
    if (!h) return CPS_ERR_INVALID;
    ForwardFleetState *F = ra_fleet(h, "cps_random_action_fleet_draws", true);
    if (!F) return CPS_ERR_NOT_CONFIGURED;
    if (!out_dev || period < 0) return fail(h, CPS_ERR_INVALID, "cps_random_action_fleet_draws: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const FleetCore &c = F->core;
    const float lo = h->mppi_in[5], hi = h->mppi_in[6];
    const FleetDrawsArgs d = {c.seed, RA_DRAWS, 0u, (unsigned)period, c.e_offset, c.E, F->K, F->T, 0LL,
                              (long long)F->T * F->K, 1, F->K, out_dev};
    return fleet_uniforms_launch(h, d, 1, lo, hi - lo);
}

extern "C" long long cps_random_action_fleet_period(const cps_handle *h) {
    return (h && h->rafleet) ? h->rafleet->core.period : -1;
}
