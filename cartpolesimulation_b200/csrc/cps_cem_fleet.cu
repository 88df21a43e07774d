// cps_cem_fleet.cu -- E independent closed-loop experiments under optimizer_cem_tf (Control_Toolkit/Optimizers/
// optimizer_cem_tf.py:12-117; `cem-tf` in Control_Toolkit_ASF/config_controllers.yml), advanced together.
//
// One controller period of EVERY experiment, no host round trip (launches independent of E):
//   per outer iteration        plan_fleet_kernel (cps_plan.cu), grid (ceil(K / 256), E): each experiment's K plans
//                              Q = clip(mu_e + eps * sd_e) from its own distribution (:66-68), their costs from its state,
//                              u_prev and targets (predict_and_cost, :57-61), and in the last block of the experiment (its
//                              own ticket) the cem_best_k cheapest plans and their mean / population stdev per step (:63-83);
//                              above 2048 elite entries (best_k x T) the statistics follow in cem_update_fleet_kernel,
//                              grid (T, E); after the last iteration the stdev clip, the shift of both vectors and
//                              u = elite_Q[0, 0] (:96-99), which becomes the experiment's u_prev;
//   fleet_net_plant_kernel     (cps_fleet.cu) the plant period with Q = u and the record row, one thread per experiment.
// With the neural predictor an outer iteration is plan_sample_kernel (the plans into [E][K][T], the period's cost
// parameters into [E]), net_grad_kernel<.., FLEET> (cps_net_grad.cu) for the costs, plan_select_kernel with one block per
// experiment, and cem_update_fleet_kernel as above: n_it x (3, or 4 with deferred statistics) + 1 launches per period.
// Every rollout starts from the network's stored hidden state; the fleet keeps none per experiment.
// Per experiment every iteration is the arithmetic of one cps_cem_step iteration; the solve counter is shared (lockstep):
// first_iter_count iterations on the first period after cps_cem_fleet_set_states, outer_its after that.  The
// distribution lives in [2][E][T] ping-pong buffers (an iteration reads one half and writes the other).
// Launches per period: n_it x (1, or 2 with deferred statistics) + 1.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include "cps_internal.cuh"
#include "cps_plant.cuh"

struct CemFleetState {
    FleetCore core;
    cps_cem_fleet_config cfg;
    int K, T;
    float *d_mu, *d_sd;               // [2][E][T] ping-pong distribution; `cur` is the live half
    int cur;
    float *d_J;                       // [E][K] costs when the caller does not ask for them
    int *d_elite;                     // [E][K] elite lists of the deferred statistics (best_k x T > 2048), else null
    unsigned *d_tickets;              // [E]
    float *d_P;                       // neural predictor: [E][K][T] the sampled plans
    CostParams *d_costs;              // neural predictor: [E] the period's folded cost parameters
    long long first_period, solves;
};

void cps_cem_fleet_free(cps_handle *h) {
    CemFleetState *F = h->cfleet;
    if (!F) return;
    fleet_core_free(F->core);
    cudaFree(F->d_mu); cudaFree(F->d_sd); cudaFree(F->d_J); cudaFree(F->d_elite); cudaFree(F->d_tickets);
    cudaFree(F->d_P); cudaFree(F->d_costs);
    delete F;
    h->cfleet = nullptr;
}

static int iterations(const CemFleetState *F, long long period) {
    return period == F->first_period ? F->cfg.first_iter_count : F->cfg.outer_its;
}

extern "C" int cps_cem_fleet_create(cps_handle *h, const cps_cem_fleet_config *cfg) {
    if (!h) return CPS_ERR_INVALID;
    const char *who = "cps_cem_fleet_create";
    if (!cfg || cfg->struct_size != (int)sizeof(cps_cem_fleet_config))
        return fail(h, CPS_ERR_INVALID, "%s: cps_cem_fleet_config size mismatch", who);
    int rc;
    if ((rc = cps_cem_fleet_check(h, cfg->best_k, cfg->initial_stdev, cfg->stdev_min,
                                  cfg->draw_source == CPS_FLEET_NOISE_PHILOX, who)) != CPS_OK)
        return rc;
    FleetCore core;
    if ((rc = fleet_core_init(h, core, cfg->n_experiments, cfg->sim_substeps, cfg->draw_source, cfg->dt_simulation, cfg->seed,
                              cfg->experiment_offset, who)) != CPS_OK)
        return rc;
    if (core.E > 65535) return fail(h, CPS_ERR_INVALID, "%s: at most 65535 experiments per handle", who);
    const int K = h->cfg.num_rollouts, T = h->cfg.horizon;
    // the Philox streams of the iterations stay below CEM_DRAWS + 2^28 (cps_plant.cuh); a draws launch has one grid layer
    // per iteration
    const long long max_its = std::min(65535LL, (long long)(1 << 28) / ((T + 3) / 4));
    if (cfg->outer_its < 1 || cfg->first_iter_count < 1 || cfg->outer_its > max_its || cfg->first_iter_count > max_its)
        return fail(h, CPS_ERR_INVALID, "%s: outer_its and first_iter_count must lie in [1, %lld]", who, max_its);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    cps_cem_fleet_free(h);
    CemFleetState *F = new (std::nothrow) CemFleetState();
    if (!F) return fail(h, CPS_ERR_INVALID, "%s: out of host memory", who);
    memset(F, 0, sizeof(*F));
    F->core = core;
    F->cfg = *cfg;
    F->K = K; F->T = T;
    h->cfleet = F;
    const size_t E = core.E;
    if ((rc = fleet_core_alloc(h, F->core)) != CPS_OK) return rc;
    CUDA_TRY(h, cudaMalloc(&F->d_mu, sizeof(float) * 2 * E * T));
    CUDA_TRY(h, cudaMalloc(&F->d_sd, sizeof(float) * 2 * E * T));
    CUDA_TRY(h, cudaMalloc(&F->d_J, sizeof(float) * E * K));
    if ((long long)cfg->best_k * T > 2048) CUDA_TRY(h, cudaMalloc(&F->d_elite, sizeof(int) * E * K));
    CUDA_TRY(h, cudaMalloc(&F->d_tickets, sizeof(unsigned) * E));
    CUDA_TRY(h, cudaMemset(F->d_tickets, 0, sizeof(unsigned) * E));
    if (h->cfg.integrator == CPS_PREDICTOR_NEURAL) {
        CUDA_TRY(h, cudaMalloc(&F->d_P, sizeof(float) * E * K * T));
        CUDA_TRY(h, cudaMalloc(&F->d_costs, sizeof(CostParams) * E));
    }
    return CPS_OK;
}

extern "C" int cps_cem_fleet_set_states(cps_handle *h, const float *s_host, long long period) {
    if (!h) return CPS_ERR_INVALID;
    const char *who = "cps_cem_fleet_set_states";
    CemFleetState *F = h->cfleet;
    if (!F) return fail(h, CPS_ERR_NOT_CONFIGURED, "%s: no CEM fleet (cps_cem_fleet_create)", who);
    int rc;
    if ((rc = fleet_core_set_states(h, F->core, s_host, period, who)) != CPS_OK) return rc;
    // optimizer_reset of every experiment (cem_tf.py:112-116), as cps_cem_reset
    const float mid = (h->mppi_in[5] + h->mppi_in[6]) * 0.5f;
    const size_t n = (size_t)F->core.E * F->T;
    std::vector<float> mu(n, mid), sd(n, F->cfg.initial_stdev);
    F->cur = 0;
    CUDA_TRY(h, cudaMemcpyAsync(F->d_mu, mu.data(), sizeof(float) * n, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(F->d_sd, sd.data(), sizeof(float) * n, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));   // the host vectors above are free to go
    F->first_period = period;
    F->solves = 0;
    F->core.ready = 1;
    return CPS_OK;
}

extern "C" int cps_cem_fleet_step(cps_handle *h, int n_periods, const float *tp_dev, const float *te_dev, const float *draws_dev,
                                  float *record_dev, float *J_out_dev, float *Q_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    const char *who = "cps_cem_fleet_step";
    CemFleetState *F = h->cfleet;
    if (!F) return fail(h, CPS_ERR_NOT_CONFIGURED, "%s: no CEM fleet (cps_cem_fleet_create)", who);
    FleetCore &fc = F->core;
    if (!fc.ready) return fail(h, CPS_ERR_NOT_CONFIGURED, "%s: no states yet (cps_cem_fleet_set_states)", who);
    if (n_periods < 0) return fail(h, CPS_ERR_INVALID, "%s: negative number of periods", who);
    int rc;
    if ((rc = fleet_core_check_draws(h, fc, draws_dev, true, who)) != CPS_OK) return rc;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const cps_cem_fleet_config &c = F->cfg;
    CemFleetIteration it;
    memset(&it, 0, sizeof(it));
    if ((rc = fleet_fold_costs(h, &it.cost_up, &it.cost_dn)) != CPS_OK) return rc;
    const size_t E = fc.E, K = F->K, T = F->T;
    it.E = fc.E; it.best_k = c.best_k; it.sd_init = c.initial_stdev; it.sd_min = c.stdev_min;
    it.s = fc.d_s; it.u = fc.d_uprev;
    it.seed = fc.seed; it.e_offset = fc.e_offset;
    it.elite = F->d_elite; it.tickets = F->d_tickets;
    it.P = F->d_P; it.costs = F->d_costs;
    NetPlantArgs pa;
    memset(&pa, 0, sizeof(pa));
    pa.plant = plant_params(h, fc.dt_sim, fc.n_sim);
    pa.s = fc.d_s; pa.u = fc.d_uprev; pa.E = fc.E;
    const float *eps = draws_dev;   // supplied draws of all periods, back to back
    for (int j = 0; j < n_periods; ++j) {
        const FleetRow row = fleet_core_row(fc, j, tp_dev, te_dev, record_dev);
        it.tp = row.tp; it.te = row.te;
        it.period = row.period;
        const int n_it = iterations(F, fc.period);
        for (int i = 0; i < n_it; ++i) {
            it.last_iter = (i == n_it - 1) ? 1 : 0;
            it.mu = F->d_mu + (size_t)F->cur * E * T; it.sd = F->d_sd + (size_t)F->cur * E * T;
            it.mu_out = F->d_mu + (size_t)(1 - F->cur) * E * T; it.sd_out = F->d_sd + (size_t)(1 - F->cur) * E * T;
            it.eps = eps ? eps + (size_t)i * E * T * K : nullptr;
            it.w1 = CEM_DRAWS + (unsigned)(i * ((T + 3) / 4));
            // J / Q of the last iteration (cem_tf.py:93) go to the caller's arrays when given
            it.J = (it.last_iter && J_out_dev) ? J_out_dev + (size_t)j * E * K : F->d_J;
            it.Q_out = (it.last_iter && Q_out_dev) ? Q_out_dev + (size_t)j * E * T * K : nullptr;
            if ((rc = cps_cem_fleet_iteration(h, it)) != CPS_OK) return rc;
            F->cur = 1 - F->cur;
        }
        if (eps) eps += (size_t)n_it * E * T * K;
        pa.tp = row.tp; pa.te = row.te; pa.record = row.record; pa.time = row.time;
        if ((rc = fleet_plant_launch(h, pa)) != CPS_OK) return rc;
        F->solves += 1;
        fc.period += 1;
    }
    return CPS_OK;
}

extern "C" int cps_cem_fleet_get_states(cps_handle *h, float *s_host, float *u_prev_host) {
    if (!h) return CPS_ERR_INVALID;
    CemFleetState *F = h->cfleet;
    if (!F || !F->core.ready) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_cem_fleet_get_states: no CEM fleet with states "
                                          "(cps_cem_fleet_create, cps_cem_fleet_set_states)");
    return fleet_core_get_states(h, F->core, s_host, u_prev_host, "cps_cem_fleet_get_states");
}

extern "C" int cps_cem_fleet_get_distribution(cps_handle *h, float *mean_host, float *stdev_host) {
    if (!h) return CPS_ERR_INVALID;
    CemFleetState *F = h->cfleet;
    if (!F || !F->core.ready) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_cem_fleet_get_distribution: no CEM fleet with states "
                                          "(cps_cem_fleet_create, cps_cem_fleet_set_states)");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t n = (size_t)F->core.E * F->T;
    if (mean_host) CUDA_TRY(h, cudaMemcpyAsync(mean_host, F->d_mu + F->cur * n, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
    if (stdev_host) CUDA_TRY(h, cudaMemcpyAsync(stdev_host, F->d_sd + F->cur * n, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}

extern "C" long long cps_cem_fleet_period(const cps_handle *h) { return (h && h->cfleet) ? h->cfleet->core.period : -1; }

// [n_it][E][T][K]: plan k's draws of experiment e in iteration it (the draws plan_fleet_kernel generates)
extern "C" int cps_cem_fleet_draws(cps_handle *h, long long period, float *out_dev) {
    if (!h) return CPS_ERR_INVALID;
    CemFleetState *F = h->cfleet;
    if (!F || !F->core.ready) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_cem_fleet_draws: no CEM fleet with states "
                                          "(cps_cem_fleet_create, cps_cem_fleet_set_states)");
    if (!out_dev || period < 0) return fail(h, CPS_ERR_INVALID, "cps_cem_fleet_draws: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const FleetCore &c = F->core;
    const FleetDrawsArgs d = {c.seed, CEM_DRAWS, (unsigned)((F->T + 3) / 4), (unsigned)period, c.e_offset, c.E, F->K, F->T,
                              (long long)c.E * F->T * F->K, (long long)F->T * F->K, 1, F->K, out_dev};
    return fleet_draws_launch(h, d, iterations(F, period));
}
