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

namespace {

// cps_cem_fleet_draws: out [n_it][E][T][K], the draws plan_fleet_kernel generates for plan k of experiment e in iteration it
__global__ void __launch_bounds__(256) cem_fleet_draws_kernel(unsigned long long seed, unsigned period, unsigned e_offset, int E,
                                                              int K, int T, float *out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x, e = blockIdx.y, it = blockIdx.z;
    if (k >= K) return;
    philox_normals(seed, (unsigned)k, CEM_DRAWS + (unsigned)(it * ((T + 3) / 4)), period, e_offset + (unsigned)e, T,
                   out + ((size_t)it * E + e) * T * K + k, K);
}

}  // namespace

struct CemFleetState {
    cps_cem_fleet_config cfg;
    int E, K, T;
    float *d_s, *d_uprev;             // [E][8], [E]
    float *d_mu, *d_sd;               // [2][E][T] ping-pong distribution; `cur` is the live half
    int cur;
    float *d_J;                       // [E][K] costs when the caller does not ask for them
    int *d_elite;                     // [E][K] elite lists of the deferred statistics (best_k x T > 2048), else null
    unsigned *d_tickets;              // [E]
    int ready;                        // cps_cem_fleet_set_states has run
    long long period, first_period, solves;
};

void cps_cem_fleet_free(cps_handle *h) {
    CemFleetState *F = h->cfleet;
    if (!F) return;
    cudaFree(F->d_s); cudaFree(F->d_uprev); cudaFree(F->d_mu); cudaFree(F->d_sd); cudaFree(F->d_J); cudaFree(F->d_elite);
    cudaFree(F->d_tickets);
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
    const bool philox = cfg->draw_source == CPS_FLEET_NOISE_PHILOX;
    int rc;
    if ((rc = cps_cem_fleet_check(h, cfg->best_k, cfg->initial_stdev, cfg->stdev_min, philox, who)) != CPS_OK) return rc;
    if (cfg->n_experiments < 1 || cfg->n_experiments > 65535 || cfg->sim_substeps < 1 || !(cfg->dt_simulation > 0.0))
        return fail(h, CPS_ERR_INVALID, "%s: need 1 <= n_experiments <= 65535, sim_substeps >= 1, dt_simulation > 0", who);
    if (cfg->draw_source != CPS_FLEET_NOISE_SUPPLIED && !philox)
        return fail(h, CPS_ERR_INVALID, "%s: unknown draw source %d", who, cfg->draw_source);
    const int K = h->cfg.num_rollouts, T = h->cfg.horizon;
    // the Philox streams of the iterations stay below CEM_DRAWS + 2^28 (cps_plant.cuh); a draws launch has one grid layer
    // per iteration
    const long long max_its = std::min(65535LL, (long long)(1 << 28) / ((T + 3) / 4));
    if (cfg->outer_its < 1 || cfg->first_iter_count < 1 || cfg->outer_its > max_its || cfg->first_iter_count > max_its)
        return fail(h, CPS_ERR_INVALID, "%s: outer_its and first_iter_count must lie in [1, %lld]", who, max_its);
    const double dt = (double)h->cfg.dt;
    if (std::fabs(cfg->sim_substeps * cfg->dt_simulation - dt) > 1e-6 * dt)
        return fail(h, CPS_ERR_INVALID, "%s: dt (control) must be sim_substeps x dt_simulation", who);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    cps_cem_fleet_free(h);
    CemFleetState *F = new (std::nothrow) CemFleetState();
    if (!F) return fail(h, CPS_ERR_INVALID, "%s: out of host memory", who);
    memset(F, 0, sizeof(*F));
    F->cfg = *cfg;
    F->E = cfg->n_experiments; F->K = K; F->T = T;
    h->cfleet = F;
    const size_t E = F->E;
    CUDA_TRY(h, cudaMalloc(&F->d_s, sizeof(float) * E * 8));
    CUDA_TRY(h, cudaMalloc(&F->d_uprev, sizeof(float) * E));
    CUDA_TRY(h, cudaMalloc(&F->d_mu, sizeof(float) * 2 * E * T));
    CUDA_TRY(h, cudaMalloc(&F->d_sd, sizeof(float) * 2 * E * T));
    CUDA_TRY(h, cudaMalloc(&F->d_J, sizeof(float) * E * K));
    if ((long long)cfg->best_k * T > 2048) CUDA_TRY(h, cudaMalloc(&F->d_elite, sizeof(int) * E * K));
    CUDA_TRY(h, cudaMalloc(&F->d_tickets, sizeof(unsigned) * E));
    CUDA_TRY(h, cudaMemset(F->d_tickets, 0, sizeof(unsigned) * E));
    return CPS_OK;
}

extern "C" int cps_cem_fleet_set_states(cps_handle *h, const float *s_host, long long period) {
    if (!h) return CPS_ERR_INVALID;
    CemFleetState *F = h->cfleet;
    if (!F) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_cem_fleet_set_states: no CEM fleet (cps_cem_fleet_create)");
    if (!s_host || period < 0) return fail(h, CPS_ERR_INVALID, "cps_cem_fleet_set_states: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    // optimizer_reset of every experiment (cem_tf.py:112-116), as cps_cem_reset
    const float mid = (h->mppi_in[5] + h->mppi_in[6]) * 0.5f;
    const size_t n = (size_t)F->E * F->T;
    std::vector<float> mu(n, mid), sd(n, F->cfg.initial_stdev);
    F->cur = 0;
    CUDA_TRY(h, cudaMemcpyAsync(F->d_mu, mu.data(), sizeof(float) * n, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(F->d_sd, sd.data(), sizeof(float) * n, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(F->d_uprev, 0, sizeof(float) * (size_t)F->E, h->stream));
    int rc;   // synchronises: the host vectors above are free to go
    if ((rc = fleet_states_to_device(h, s_host, F->d_s, F->E, "cps_cem_fleet_set_states")) != CPS_OK) return rc;
    F->period = F->first_period = period;
    F->solves = 0;
    F->ready = 1;
    return CPS_OK;
}

extern "C" int cps_cem_fleet_step(cps_handle *h, int n_periods, const float *tp_dev, const float *te_dev, const float *draws_dev,
                                  float *record_dev, float *J_out_dev, float *Q_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    const char *who = "cps_cem_fleet_step";
    CemFleetState *F = h->cfleet;
    if (!F) return fail(h, CPS_ERR_NOT_CONFIGURED, "%s: no CEM fleet (cps_cem_fleet_create)", who);
    if (!F->ready) return fail(h, CPS_ERR_NOT_CONFIGURED, "%s: no states yet (cps_cem_fleet_set_states)", who);
    if (n_periods < 0) return fail(h, CPS_ERR_INVALID, "%s: negative number of periods", who);
    const cps_cem_fleet_config &c = F->cfg;
    const bool philox = c.draw_source == CPS_FLEET_NOISE_PHILOX;
    if (!philox && !draws_dev) return fail(h, CPS_ERR_INVALID, "%s: this fleet expects supplied draws", who);
    if (philox && draws_dev) return fail(h, CPS_ERR_INVALID, "%s: this fleet generates its draws (Philox); pass NULL", who);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc;
    CemFleetIteration it;
    memset(&it, 0, sizeof(it));
    if ((rc = cps_fold_cost_for(h, 1.0f, &it.cost_up)) != CPS_OK) return rc;
    if ((rc = cps_fold_cost_for(h, -1.0f, &it.cost_dn)) != CPS_OK) return rc;
    const size_t E = F->E, K = F->K, T = F->T;
    it.E = F->E; it.best_k = c.best_k; it.sd_init = c.initial_stdev; it.sd_min = c.stdev_min;
    it.s = F->d_s; it.u = F->d_uprev;
    it.seed = c.seed; it.e_offset = (unsigned)c.experiment_offset;
    it.elite = F->d_elite; it.tickets = F->d_tickets;
    NetPlantArgs pa;
    memset(&pa, 0, sizeof(pa));
    pa.plant = plant_params(h, c.dt_simulation, c.sim_substeps);
    pa.s = F->d_s; pa.u = F->d_uprev; pa.E = F->E;
    const double dt_control = c.dt_simulation * c.sim_substeps;
    const float *eps = draws_dev;   // supplied draws of all periods, back to back
    for (int j = 0; j < n_periods; ++j) {
        it.tp = tp_dev ? tp_dev + (size_t)j * E : nullptr;
        it.te = te_dev ? te_dev + (size_t)j * E : nullptr;
        it.period = (unsigned)F->period;
        const int n_it = iterations(F, F->period);
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
        pa.tp = it.tp; pa.te = it.te;
        pa.record = record_dev ? record_dev + (size_t)j * E * CPS_FLEET_RECORD : nullptr;
        pa.time = (double)F->period * dt_control;
        if ((rc = fleet_plant_launch(h, pa)) != CPS_OK) return rc;
        F->solves += 1;
        F->period += 1;
    }
    return CPS_OK;
}

extern "C" int cps_cem_fleet_get_states(cps_handle *h, float *s_host, float *u_prev_host) {
    if (!h) return CPS_ERR_INVALID;
    CemFleetState *F = h->cfleet;
    if (!F || !F->ready) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_cem_fleet_get_states: no CEM fleet with states "
                                    "(cps_cem_fleet_create, cps_cem_fleet_set_states)");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc;
    if (s_host && (rc = fleet_states_to_host(h, F->d_s, s_host, F->E, "cps_cem_fleet_get_states")) != CPS_OK) return rc;
    if (u_prev_host)
        CUDA_TRY(h, cudaMemcpyAsync(u_prev_host, F->d_uprev, sizeof(float) * (size_t)F->E, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}

extern "C" int cps_cem_fleet_get_distribution(cps_handle *h, float *mean_host, float *stdev_host) {
    if (!h) return CPS_ERR_INVALID;
    CemFleetState *F = h->cfleet;
    if (!F || !F->ready) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_cem_fleet_get_distribution: no CEM fleet with states "
                                    "(cps_cem_fleet_create, cps_cem_fleet_set_states)");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t n = (size_t)F->E * F->T;
    if (mean_host) CUDA_TRY(h, cudaMemcpyAsync(mean_host, F->d_mu + F->cur * n, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
    if (stdev_host) CUDA_TRY(h, cudaMemcpyAsync(stdev_host, F->d_sd + F->cur * n, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}

extern "C" long long cps_cem_fleet_period(const cps_handle *h) { return (h && h->cfleet) ? h->cfleet->period : -1; }

extern "C" int cps_cem_fleet_draws(cps_handle *h, long long period, float *out_dev) {
    if (!h) return CPS_ERR_INVALID;
    CemFleetState *F = h->cfleet;
    if (!F || !F->ready) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_cem_fleet_draws: no CEM fleet with states "
                                    "(cps_cem_fleet_create, cps_cem_fleet_set_states)");
    if (!out_dev || period < 0) return fail(h, CPS_ERR_INVALID, "cps_cem_fleet_draws: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const dim3 grid((unsigned)(F->K + 255) / 256, (unsigned)F->E, (unsigned)iterations(F, period));
    cem_fleet_draws_kernel<<<grid, 256, 0, h->stream>>>(F->cfg.seed, (unsigned)period, (unsigned)F->cfg.experiment_offset, F->E,
                                                        F->K, F->T, out_dev);
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}
