// cps_rpgd_fleet.cu -- E independent closed-loop experiments under RPGD, the reference's shipped default optimizer
// (Control_Toolkit_ASF/config_controllers.yml:2; Control_Toolkit/Optimizers/optimizer_rpgd_tf.py), advanced together.
//
// One controller period of EVERY experiment, no host round trip (launches independent of E):
//   rpgd_fleet_cost_kernel     the cost parameters of each experiment's targets, folded once into an [E] array;
//   per Adam step              predictor "ODE": the three ODE adjoint kernels of cps_grad.cu over all E x K plans (plan k
//                              belongs to experiment k / K and takes its state, u_prev and cost parameters; per plan the
//                              arithmetic of cps_plan_cost_grad); neural predictor: net_grad_kernel<.., FLEET> of
//                              cps_net_grad.cu, one launch over E experiments x K plans with the single-experiment tiling
//                              (the same per-plan arithmetic, the stored hidden state read and never written); then
//                              rpgd_update_kernel over all E x K plans;
//   costs                      the adjoint's forward over all plans without checkpoints / records (J of cps_plan_cost bit
//                              for bit);
//   rpgd_fleet_finish_kernel   one block per experiment: stable ranks of its K costs, u = the cheapest plan's first
//                              input, the shifted / permuted plans, moments and ages into the other half of a ping-pong
//                              pair (fresh plans built in the kernel from the draws), then the plant period in the
//                              reference's mixed float32 / float64 arithmetic (cps_plant.cuh, as cps_fleet.cu) and the
//                              record row.
// The solve counter and Adam's iteration count are shared (lockstep), so lr_t is one host-computed scalar per Adam step.
// Launches per period: 3 + 4 x (Adam steps) with predictor "ODE", 3 + 2 x (Adam steps) with the neural predictor.
//
// Offline relabelling (cps_rpgd_fleet_relabel) is the same period with the plant replaced by a recording: per row,
// rpgd_relabel_row_kernel takes the place of rpgd_fleet_cost_kernel -- it also copies the row's recorded states into the
// fleet's states and, with per-row L / m_pole on predictor "ODE", folds each experiment's model constants (the _ode
// adjoint kernels of cps_grad.cu read them) -- and rpgd_relabel_finish_kernel does the bookkeeping of
// rpgd_fleet_finish_kernel, then writes u to u_prev and Q_out instead of integrating.  Same launches per row as per period.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>
#include <cstring>
#include <new>

#include "cps_internal.cuh"
#include "cps_plant.cuh"

namespace {

__global__ void __launch_bounds__(128) rpgd_fleet_cost_kernel(const CostParams up, const CostParams dn, const float *tp,
                                                               const float *te, CostParams *out, int E) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    out[e] = fold_cost_e(up, dn, tp, te, e);
}

struct RpgdRowArgs {
    CostParams up, dn;
    const float *tp, *te;            // [E] targets of this row (null: 0 / +1)
    const float *states;             // [E][6] recorded states of this row
    const float *L_row, *mp_row;     // [E] the controller model's pole length / mass of this row, or null
    CostParams *costs;               // [E] <- folded cost parameters
    float *s;                        // [E][8] <- the recorded states
    OdeParams *odes;                 // [E] <- per-experiment model constants, or null (neural, or no per-row L / m_pole)
    OdeParams ode;                   // the handle's fold (the constants that do not depend on L / m_pole)
    FoldInputs fold;
    int E;
};

// Relabelling, per row: what rpgd_fleet_cost_kernel does, the row's recorded states into the fleet's, and the model
// constants of each experiment's L / m_pole.  One thread per experiment.
__global__ void __launch_bounds__(128) rpgd_relabel_row_kernel(const __grid_constant__ RpgdRowArgs a) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= a.E) return;
    a.costs[e] = fold_cost_e(a.up, a.dn, a.tp, a.te, e);
#pragma unroll
    for (int c = 0; c < 6; ++c) a.s[(size_t)e * 8 + c] = a.states[(size_t)e * 6 + c];
    if (a.odes) {
        OdeParams o = a.ode;
        fold_ode_device<CPS_EULER_CROMER>(a.fold, a.L_row ? (double)a.L_row[e] : (double)a.fold.L_default,
                                          a.mp_row ? (double)a.mp_row[e] : (double)a.fold.mp_default, o);
        a.odes[e] = o;
    }
}

// Input t of a fresh plan from its raw draws d[i * ds], i < n_ind (optimizer_rpgd_b200.sample_actions): the draws scaled,
// shifted and clipped at the inducing points, then Interpolator's tent weights (the last inducing point enters its own
// step with weight 1 / p; Control_Toolkit/others/Interpolator.py:54-78), summed as oracle/cps_oracle.c does.
__device__ __forceinline__ float fresh_input(const float *d, long long ds, int t, int p, int n_ind, float stdev, float mean,
                                             float lo, float hi) {
    const int last = (n_ind - 1) * p;
    float acc = 0.0f;
    if (t < last) {
        const int i = t / p, j = t % p;
        const float z0 = fminf(fmaxf(__fadd_rn(__fmul_rn(d[i * ds], stdev), mean), lo), hi);
        acc = __fadd_rn(acc, __fmul_rn(z0, __fdiv_rn((float)(p - j), (float)p)));
        if (j) {
            const float z1 = fminf(fmaxf(__fadd_rn(__fmul_rn(d[(i + 1) * ds], stdev), mean), lo), hi);
            acc = __fadd_rn(acc, __fmul_rn(z1, __fdiv_rn((float)j, (float)p)));
        }
    } else if (t == last) {
        const float z = fminf(fmaxf(__fadd_rn(__fmul_rn(d[(n_ind - 1) * ds], stdev), mean), lo), hi);
        acc = __fadd_rn(acc, __fmul_rn(z, __fdiv_rn(1.0f, (float)p)));
    }
    return acc;
}

// The order of torch.sort(J, stable=True) (optimizer_rpgd_tf.py:186): numbers ascending, every NaN after them, ties and NaNs
// among themselves by index.  A strict total order whatever the costs hold, so the ranks counted with it are always a
// permutation of 0..K-1 (a NaN cost -- a NaN state or target -- must not leave ranks unassigned).
__device__ __forceinline__ bool sorts_before(float Jj, int j, float Ji, int i) {
    const bool nj = isnan(Jj), ni = isnan(Ji);
    if (nj != ni) return ni;   // a number before a NaN
    if (nj || Jj == Ji) return j < i;
    return Jj < Ji;
}

struct SampleParams {
    int p, n_ind;
    float stdev, mean, lo, hi;
};

// cps_rpgd_fleet_draws: rows [E][rows][n_ind]
__global__ void __launch_bounds__(128) rpgd_fleet_draws_kernel(unsigned long long seed, unsigned tag, unsigned period,
                                                                unsigned e_offset, int rows, int n_ind, float *out) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x, e = blockIdx.y;
    if (r >= rows) return;
    philox_normals(seed, (unsigned)r, tag, period, e_offset + (unsigned)e, n_ind, out + ((size_t)e * rows + r) * n_ind, 1);
}

// optimizer_reset of every experiment (:379-408): plans from the draws [E * K][n_ind], zero moments and ages
__global__ void __launch_bounds__(256) rpgd_fleet_reset_kernel(const float *draws, float *Q, float *m, float *v, int *ages,
                                                                long long n, int T, const SampleParams sp) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long row = i / T;
        const int t = (int)(i % T);
        Q[i] = fresh_input(draws + row * sp.n_ind, 1, t, sp.p, sp.n_ind, sp.stdev, sp.mean, sp.lo, sp.hi);
        m[i] = 0.0f;
        v[i] = 0.0f;
        if (t == 0) ages[row] = 0;
    }
}

struct RpgdFinishArgs {
    const float *J;                  // [E][K] costs of the improved plans
    const float *Q, *m, *v;          // [E][K][T] plans after the Adam steps and their moments
    const int *ages;                 // [E][K]
    float *Q2, *m2, *v2;             // the other half of the ping-pong pair
    int *ages2;
    const float *draws;              // supplied resampling draws [E][K - keep][n_ind] of this period, or null (Philox)
    int resample, philox;
    unsigned long long seed;
    unsigned period, e_offset;
    int K, T, keep, shift;
    SampleParams sp;
    float *u_prev;                   // [E] <- u
    float *s;                        // [E][8] plant states
    PlantParams plant;
    const float *tp, *te;            // [E] targets of this period (null: 0 / +1), for the record
    float *record;                   // [E][CPS_FLEET_RECORD] or null
    float *J_out;                    // [E][K] or null
    float *Q_opt;                    // [E][K][T] or null
    double time;
    float *Q_out;                    // relabelling: [E] <- u (no plant, no record)
};

// get_action + the bookkeeping of step() (:182-224, :297-356), then the plant: one block per experiment.  The plant stage
// reads nothing the bookkeeping writes; REPLAY (offline relabelling: the next state comes from a recording) replaces only
// that stage, by writing u to Q_out.
template <bool REPLAY>
__device__ __forceinline__ void rpgd_finish(const RpgdFinishArgs &a) {
    extern __shared__ float smem[];
    const int e = blockIdx.x, tid = threadIdx.x, nt = blockDim.x, K = a.K, T = a.T;
    float *s_J = smem;
    int *s_src = reinterpret_cast<int *>(smem + K);   // s_src[rank] = plan
    float *s_d = smem + 2 * K;                        // Philox resampling draws [K - keep][n_ind]
    const size_t base = (size_t)e * K * T;
    const int nf = a.resample ? K - a.keep : 0;       // fresh plans
    for (int i = tid; i < K; i += nt) s_J[i] = a.J[(size_t)e * K + i];
    if (a.philox)
        for (int r = tid; r < nf; r += nt)
            philox_normals(a.seed, (unsigned)r, RPGD_DRAWS_RESAMPLE, a.period, a.e_offset + (unsigned)e, a.sp.n_ind,
                           s_d + r * a.sp.n_ind, 1);
    __syncthreads();
    for (int i = tid; i < K; i += nt) {   // plans in front of plan i in torch.sort(J, stable=True)'s order
        const float Ji = s_J[i];
        int rank = 0;
        for (int j = 0; j < K; ++j) rank += sorts_before(s_J[j], j, Ji, i) ? 1 : 0;
        s_src[rank] = i;
        if (a.J_out) a.J_out[(size_t)e * K + i] = Ji;
    }
    __syncthreads();
    const float *Q = a.Q + base, *m = a.m + base, *v = a.v + base;
    const int *ages = a.ages + (size_t)e * K;
    for (int idx = tid; idx < K * T; idx += nt) {
        const int r = idx / T, t = idx - r * T;
        float q, mm = 0.0f, vv = 0.0f;
        int age;
        if (r < nf) {   // rows 0..K-keep-1 of a resampling solve: fresh plans, zero moments and age
            const float *d = a.philox ? s_d + r * a.sp.n_ind : a.draws + ((size_t)e * nf + r) * a.sp.n_ind;
            q = fresh_input(d, 1, t, a.sp.p, a.sp.n_ind, a.sp.stdev, a.sp.mean, a.sp.lo, a.sp.hi);
            age = 1;
        } else {        // kept plans in cost order (resampling) or every plan in place, shifted
            const int i = a.resample ? s_src[r - nf] : r;
            q = Q[(size_t)i * T + min(t + a.shift, T - 1)];
            if (t + 1 < T) { mm = m[(size_t)i * T + t + 1]; vv = v[(size_t)i * T + t + 1]; }
            age = ages[i] + 1;
        }
        a.Q2[base + idx] = q;
        a.m2[base + idx] = mm;
        a.v2[base + idx] = vv;
        if (t == 0) a.ages2[(size_t)e * K + r] = age;
        if (a.Q_opt) a.Q_opt[base + idx] = Q[idx];
    }
    if (tid != 0) return;

    // ---- the plant: one controller period with Q held (CartPole/__init__.py:283-324), as fleet_kernel without plant-side models
    const float Qc = Q[(size_t)s_src[0] * T];   // u_nom[0] of the cheapest improved plan
    a.u_prev[e] = Qc;                           // the returned control enters the next solve's cost
    if (REPLAY) {
        a.Q_out[e] = Qc;
        return;
    }
    const PlantParams &P = a.plant;
    float s[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) s[c] = a.s[(size_t)e * 8 + c];
    const float u = __fmul_rn(P.u_max, Qc);
    double aDD, pDD;
    plant_ode(P, s[IDX_COS], s[IDX_SIN], s[IDX_ANGLED], s[IDX_POSD], u, aDD, pDD);
    if (a.record)
        plant_record(a.record + (size_t)e * CPS_FLEET_RECORD, a.time, s, aDD, pDD, Qc, Qc, u, a.tp ? a.tp[e] : 0.0f,
                     a.te ? a.te[e] : 1.0f);
    plant_ticks(P, s, u, aDD, pDD, [](int) {});
    float *so = a.s + (size_t)e * 8;
#pragma unroll
    for (int c = 0; c < 6; ++c) so[c] = s[c];
}
__global__ void __launch_bounds__(128) rpgd_fleet_finish_kernel(const __grid_constant__ RpgdFinishArgs a) {
    rpgd_finish<false>(a);
}
__global__ void __launch_bounds__(128) rpgd_relabel_finish_kernel(const __grid_constant__ RpgdFinishArgs a) {
    rpgd_finish<true>(a);
}

}  // namespace

// ---- host side ---------------------------------------------------------------------------------------------------------
struct RpgdFleetState {
    cps_rpgd_fleet_config cfg;
    int E, K, T, nf;                  // nf = K - opt_keep_k fresh plans per resampling solve
    float *d_s, *d_uprev;             // [E][8], [E]
    float *d_Q[2], *d_m[2], *d_v[2];  // ping-pong plans and Adam moments [E][K][T]
    int *d_ages[2];                   // [E][K]
    int cur;                          // which half holds the current plans
    float *d_ck, *d_jac, *d_J, *d_G;  // adjoint workspace: [T][4][EK], [T][CPS_GRAD_REC][EK] (ODE only; the neural adjoint
                                      // keeps its records in the network's workspace), [EK], [EK][T]
    CostParams *d_costs;              // [E] this period's folded cost parameters
    OdeParams *d_odes;                // [E] relabelling: each experiment's model constants for its row's L / m_pole (ODE only)
    float *d_draws;                   // Philox reset draws [E][K][n_ind]
    size_t finish_smem;
    int ready;                        // cps_rpgd_fleet_set_states has run
    long long period, solves, adam_iterations;
};

void cps_rpgd_fleet_free(cps_handle *h) {
    RpgdFleetState *F = h->rfleet;
    if (!F) return;
    cudaFree(F->d_s); cudaFree(F->d_uprev);
    for (int i = 0; i < 2; ++i) { cudaFree(F->d_Q[i]); cudaFree(F->d_m[i]); cudaFree(F->d_v[i]); cudaFree(F->d_ages[i]); }
    cudaFree(F->d_ck); cudaFree(F->d_jac); cudaFree(F->d_J); cudaFree(F->d_G); cudaFree(F->d_costs); cudaFree(F->d_draws);
    cudaFree(F->d_odes);
    delete F;
    h->rfleet = nullptr;
}

static SampleParams sample_params(const cps_handle *h, const RpgdFleetState *F) {
    SampleParams sp;
    sp.p = h->cfg.interp_period; sp.n_ind = h->n_ind;
    sp.stdev = F->cfg.sample_stdev; sp.mean = F->cfg.sample_mean;
    sp.lo = h->mppi_in[5]; sp.hi = h->mppi_in[6];
    return sp;
}

extern "C" int cps_rpgd_fleet_create(cps_handle *h, const cps_rpgd_fleet_config *cfg) {
    if (!h) return CPS_ERR_INVALID;
    if (!cfg || cfg->struct_size != (int)sizeof(cps_rpgd_fleet_config))
        return fail(h, CPS_ERR_INVALID, "cps_rpgd_fleet_create: cps_rpgd_fleet_config size mismatch");
    const bool neural = h->cfg.integrator == CPS_PREDICTOR_NEURAL;
    if (h->cfg.integrator != CPS_EULER_CROMER && !neural)
        return fail(h, CPS_ERR_UNSUPPORTED, "cps_rpgd_fleet_create: the adjoint of an RPGD fleet is built for predictor \"ODE\" "
                    "(Euler-Cromer) and the neural predictor");
    if (h->cfg.cost_id != CPS_COST_QB_GRAD_MINIMAL && h->cfg.cost_id != CPS_COST_QB_GRAD)
        return fail(h, CPS_ERR_UNSUPPORTED, "cps_rpgd_fleet_create: the adjoint is built for the quadratic_boundary_grad_minimal and "
                    "quadratic_boundary_grad plugins");
    if (!neural && h->cfg.substeps > 32)
        return fail(h, CPS_ERR_UNSUPPORTED, "cps_rpgd_fleet_create: at most 32 substeps per control step");
    const int K = h->cfg.num_rollouts, T = h->cfg.horizon;
    if (K > 4096) return fail(h, CPS_ERR_UNSUPPORTED, "cps_rpgd_fleet_create: at most 4096 plans (ranks by counting)");
    if (cfg->n_experiments < 1 || cfg->sim_substeps < 1 || !(cfg->dt_simulation > 0.0))
        return fail(h, CPS_ERR_INVALID, "cps_rpgd_fleet_create: need n_experiments >= 1, sim_substeps >= 1, dt_simulation > 0");
    if ((long long)cfg->n_experiments * K > (1LL << 30))
        return fail(h, CPS_ERR_INVALID, "cps_rpgd_fleet_create: at most 2^30 plans (n_experiments x K) per handle");
    if (cfg->draw_source != CPS_FLEET_NOISE_SUPPLIED && cfg->draw_source != CPS_FLEET_NOISE_PHILOX)
        return fail(h, CPS_ERR_INVALID, "cps_rpgd_fleet_create: unknown draw source %d", cfg->draw_source);
    if (cfg->opt_keep_k < 1 || cfg->opt_keep_k > K)
        return fail(h, CPS_ERR_INVALID, "cps_rpgd_fleet_create: opt_keep_k must lie in [1, K]");
    if (cfg->shift_previous < 0) return fail(h, CPS_ERR_INVALID, "cps_rpgd_fleet_create: shift_previous < 0");
    if (cfg->outer_its < 0 || cfg->first_iter_count < 0 || cfg->resamp_per < 1)
        return fail(h, CPS_ERR_INVALID, "cps_rpgd_fleet_create: need outer_its >= 0, first_iter_count >= 0, resamp_per >= 1");
    const double dt = (double)h->cfg.dt;
    if (std::fabs(cfg->sim_substeps * cfg->dt_simulation - dt) > 1e-6 * dt)
        return fail(h, CPS_ERR_INVALID, "cps_rpgd_fleet_create: dt (control) must be sim_substeps x dt_simulation");
    const int nf = K - cfg->opt_keep_k;
    const size_t smem = sizeof(float) * (2 * (size_t)K + (cfg->draw_source == CPS_FLEET_NOISE_PHILOX ? (size_t)nf * h->n_ind : 0));
    if (smem > 227 * 1024)
        return fail(h, CPS_ERR_UNSUPPORTED, "cps_rpgd_fleet_create: (K - opt_keep_k) x n_ind too large for the finish kernel's "
                    "shared memory");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc;   // neural: the network checks of cps_plan_cost_grad, and the workspace sized now rather than mid-run
    if (neural && (rc = cps_net_grad_fleet_prepare(h, cfg->n_experiments, "cps_rpgd_fleet_create")) != CPS_OK) return rc;
    cps_rpgd_fleet_free(h);
    RpgdFleetState *F = new (std::nothrow) RpgdFleetState();
    if (!F) return fail(h, CPS_ERR_INVALID, "cps_rpgd_fleet_create: out of host memory");
    memset(F, 0, sizeof(*F));
    F->cfg = *cfg;
    F->E = cfg->n_experiments; F->K = K; F->T = T; F->nf = nf;
    F->finish_smem = smem;
    h->rfleet = F;
    const size_t E = F->E, EK = E * K, n = EK * T;
    CUDA_TRY(h, cudaMalloc(&F->d_s, sizeof(float) * E * 8));
    CUDA_TRY(h, cudaMalloc(&F->d_uprev, sizeof(float) * E));
    for (int i = 0; i < 2; ++i) {
        CUDA_TRY(h, cudaMalloc(&F->d_Q[i], sizeof(float) * n));
        CUDA_TRY(h, cudaMalloc(&F->d_m[i], sizeof(float) * n));
        CUDA_TRY(h, cudaMalloc(&F->d_v[i], sizeof(float) * n));
        CUDA_TRY(h, cudaMalloc(&F->d_ages[i], sizeof(int) * EK));
    }
    if (!neural) {
        CUDA_TRY(h, cudaMalloc(&F->d_ck, sizeof(float) * 4 * n));
        CUDA_TRY(h, cudaMalloc(&F->d_jac, sizeof(float) * CPS_GRAD_REC * n));
        CUDA_TRY(h, cudaMalloc(&F->d_odes, sizeof(OdeParams) * E));
    }
    CUDA_TRY(h, cudaMalloc(&F->d_J, sizeof(float) * EK));
    CUDA_TRY(h, cudaMalloc(&F->d_G, sizeof(float) * n));
    CUDA_TRY(h, cudaMalloc(&F->d_costs, sizeof(CostParams) * E));
    if (cfg->draw_source == CPS_FLEET_NOISE_PHILOX) CUDA_TRY(h, cudaMalloc(&F->d_draws, sizeof(float) * EK * h->n_ind));
    if (smem > 48 * 1024) {
        CUDA_TRY(h, cudaFuncSetAttribute((const void *)rpgd_fleet_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(h, cudaFuncSetAttribute((const void *)rpgd_relabel_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    return CPS_OK;
}

static int draws_launch(cps_handle *h, RpgdFleetState *F, long long period, float *out_dev) {
    const bool reset = period < 0;
    const int rows = reset ? F->K : F->nf;
    if (rows == 0) return CPS_OK;
    const dim3 grid((rows + 127) / 128, F->E);
    rpgd_fleet_draws_kernel<<<grid, 128, 0, h->stream>>>(F->cfg.seed, reset ? RPGD_DRAWS_RESET : RPGD_DRAWS_RESAMPLE,
                                                          reset ? 0u : (unsigned)period, (unsigned)F->cfg.experiment_offset,
                                                          rows, h->n_ind, out_dev);
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

extern "C" int cps_rpgd_fleet_set_states(cps_handle *h, const float *s_host, const float *init_draws_dev, long long period) {
    if (!h) return CPS_ERR_INVALID;
    RpgdFleetState *F = h->rfleet;
    if (!F) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_rpgd_fleet_set_states: no RPGD fleet (cps_rpgd_fleet_create)");
    const bool philox = F->cfg.draw_source == CPS_FLEET_NOISE_PHILOX;
    if (!s_host || period < 0) return fail(h, CPS_ERR_INVALID, "cps_rpgd_fleet_set_states: bad argument");
    if (!philox && !init_draws_dev) return fail(h, CPS_ERR_INVALID, "cps_rpgd_fleet_set_states: this fleet expects supplied draws");
    if (philox && init_draws_dev)
        return fail(h, CPS_ERR_INVALID, "cps_rpgd_fleet_set_states: this fleet generates its draws (Philox); pass NULL");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaMemsetAsync(F->d_uprev, 0, sizeof(float) * (size_t)F->E, h->stream));
    int rc;
    if ((rc = fleet_states_to_device(h, s_host, F->d_s, F->E, "cps_rpgd_fleet_set_states")) != CPS_OK) return rc;
    if (philox && (rc = draws_launch(h, F, -1, F->d_draws)) != CPS_OK) return rc;
    F->cur = 0;
    const long long n = (long long)F->E * F->K * F->T;
    const int grid = (int)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096);
    rpgd_fleet_reset_kernel<<<grid, 256, 0, h->stream>>>(philox ? F->d_draws : init_draws_dev, F->d_Q[0], F->d_m[0], F->d_v[0],
                                                          F->d_ages[0], n, F->T, sample_params(h, F));
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    F->period = period;
    F->solves = 0;
    F->adam_iterations = 0;
    F->ready = 1;
    return CPS_OK;
}

int cps_fold_cost_for(cps_handle *h, float target_equilibrium, CostParams *out);

// Shared by cps_rpgd_fleet_step (closed loop: replay_dev == nullptr) and cps_rpgd_fleet_relabel (states from a recording).
static int rpgd_fleet_launch(cps_handle *h, const char *who, int n_periods, const float *tp_dev, const float *te_dev,
                             const float *draws_dev, float *record_dev, float *J_out_dev, float *Q_opt_out_dev,
                             const float *replay_dev, const float *L_dev, const float *mp_dev, float *Q_out_dev) {
    RpgdFleetState *F = h->rfleet;
    if (!F) return fail(h, CPS_ERR_NOT_CONFIGURED, "%s: no RPGD fleet (cps_rpgd_fleet_create)", who);
    if (!F->ready) return fail(h, CPS_ERR_NOT_CONFIGURED, "%s: no states yet (cps_rpgd_fleet_set_states)", who);
    if (n_periods < 0) return fail(h, CPS_ERR_INVALID, "%s: negative number of periods / rows", who);
    const bool philox = F->cfg.draw_source == CPS_FLEET_NOISE_PHILOX;
    if (!philox && !draws_dev && F->nf > 0) return fail(h, CPS_ERR_INVALID, "%s: this fleet expects supplied draws", who);
    if (philox && draws_dev) return fail(h, CPS_ERR_INVALID, "%s: this fleet generates its draws (Philox); pass NULL", who);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const bool neural = h->cfg.integrator == CPS_PREDICTOR_NEURAL;
    int rc;   // neural: the network may have been reloaded since create (another size): check it, grow the workspace
    if (neural && (rc = cps_net_grad_fleet_prepare(h, F->E, who)) != CPS_OK) return rc;
    CostParams up, dn;
    if ((rc = cps_fold_cost_for(h, 1.0f, &up)) != CPS_OK) return rc;
    if ((rc = cps_fold_cost_for(h, -1.0f, &dn)) != CPS_OK) return rc;
    const cps_rpgd_fleet_config &c = F->cfg;
    const size_t E = F->E, K = F->K, T = F->T;
    const int EK = (int)(E * K);
    RpgdFinishArgs a;
    memset(&a, 0, sizeof(a));
    a.philox = philox ? 1 : 0;
    a.seed = c.seed; a.e_offset = (unsigned)c.experiment_offset;
    a.K = (int)K; a.T = (int)T; a.keep = c.opt_keep_k; a.shift = c.shift_previous;
    a.sp = sample_params(h, F);
    a.u_prev = F->d_uprev; a.s = F->d_s;
    a.plant = plant_params(h, c.dt_simulation, c.sim_substeps);
    const double dt_control = c.dt_simulation * c.sim_substeps;
    // relabelling: the network reads neither L nor m_pole, so only predictor "ODE" folds per-row model constants
    const OdeParams *odes = (replay_dev && !neural && (L_dev || mp_dev)) ? F->d_odes : nullptr;
    RpgdRowArgs ra;
    memset(&ra, 0, sizeof(ra));
    ra.up = up; ra.dn = dn;
    ra.costs = F->d_costs; ra.s = F->d_s; ra.odes = const_cast<OdeParams *>(odes);
    ra.ode = h->ode;
    ra.fold = fold_inputs(h);
    ra.E = (int)E;
    for (int j = 0; j < n_periods; ++j) {
        const float *tp = tp_dev ? tp_dev + (size_t)j * E : nullptr, *te = te_dev ? te_dev + (size_t)j * E : nullptr;
        if (replay_dev) {
            ra.tp = tp; ra.te = te;
            ra.states = replay_dev + (size_t)j * E * 6;
            ra.L_row = L_dev ? L_dev + (size_t)j * E : nullptr;
            ra.mp_row = mp_dev ? mp_dev + (size_t)j * E : nullptr;
            rpgd_relabel_row_kernel<<<(unsigned)((E + 127) / 128), 128, 0, h->stream>>>(ra);
        } else {
            rpgd_fleet_cost_kernel<<<(unsigned)((E + 127) / 128), 128, 0, h->stream>>>(up, dn, tp, te, F->d_costs, (int)E);
        }
        h->launches += 1;
        float *Q = F->d_Q[F->cur], *m = F->d_m[F->cur], *v = F->d_v[F->cur];
        const int its = F->solves == 0 ? c.first_iter_count : c.outer_its;
        for (int it = 0; it < its; ++it) {   // grad_step (:166-180)
            rc = neural ? cps_net_grad_fleet(h, (int)E, F->d_s, Q, F->d_costs, F->d_uprev, F->d_J, F->d_G)
                        : cps_grad_fleet(h, EK, (int)K, F->d_s, Q, F->d_costs, F->d_uprev, F->d_ck, F->d_jac, F->d_J, F->d_G,
                                         odes);
            if (rc != CPS_OK) return rc;
            F->adam_iterations += 1;
            const double t = (double)F->adam_iterations;   // ResourceApplyAdam, as cps_rpgd_grad_step
            const float lr_t = (float)((double)c.learning_rate * sqrt(1.0 - pow((double)c.adam_beta_2, t)) /
                                       (1.0 - pow((double)c.adam_beta_1, t)));
            if ((rc = cps_grad_fleet_update(h, EK, Q, F->d_G, m, v, lr_t, c.adam_beta_1, c.adam_beta_2, c.adam_epsilon,
                                            c.gradmax_clip)) != CPS_OK)
                return rc;
        }
        // get_action (:182-224): the costs of the improved plans
        rc = neural ? cps_net_grad_fleet(h, (int)E, F->d_s, Q, F->d_costs, F->d_uprev, F->d_J, nullptr)
                    : cps_grad_fleet(h, EK, (int)K, F->d_s, Q, F->d_costs, F->d_uprev, nullptr, nullptr, F->d_J, nullptr, odes);
        if (rc != CPS_OK) return rc;
        const int nxt = F->cur ^ 1;
        a.J = F->d_J; a.Q = Q; a.m = m; a.v = v; a.ages = F->d_ages[F->cur];
        a.Q2 = F->d_Q[nxt]; a.m2 = F->d_m[nxt]; a.v2 = F->d_v[nxt]; a.ages2 = F->d_ages[nxt];
        a.resample = (F->solves % c.resamp_per == 0) ? 1 : 0;
        a.draws = (!philox && a.resample) ? draws_dev + (size_t)j * E * F->nf * h->n_ind : nullptr;
        a.period = (unsigned)F->period;
        a.tp = tp; a.te = te;
        a.record = record_dev ? record_dev + (size_t)j * E * CPS_FLEET_RECORD : nullptr;
        a.J_out = J_out_dev ? J_out_dev + (size_t)j * E * K : nullptr;
        a.Q_opt = Q_opt_out_dev ? Q_opt_out_dev + (size_t)j * E * K * T : nullptr;
        a.time = (double)F->period * dt_control;
        a.Q_out = Q_out_dev ? Q_out_dev + (size_t)j * E : nullptr;
        if (replay_dev) rpgd_relabel_finish_kernel<<<(unsigned)E, 128, F->finish_smem, h->stream>>>(a);
        else rpgd_fleet_finish_kernel<<<(unsigned)E, 128, F->finish_smem, h->stream>>>(a);
        h->launches += 1;
        CUDA_TRY(h, cudaGetLastError());
        F->cur = nxt;
        F->solves += 1;
        F->period += 1;
    }
    return CPS_OK;
}

extern "C" int cps_rpgd_fleet_step(cps_handle *h, int n_periods, const float *tp_dev, const float *te_dev, const float *draws_dev,
                                   float *record_dev, float *J_out_dev, float *Q_opt_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    return rpgd_fleet_launch(h, "cps_rpgd_fleet_step", n_periods, tp_dev, te_dev, draws_dev, record_dev, J_out_dev, Q_opt_out_dev,
                             nullptr, nullptr, nullptr, nullptr);
}

extern "C" int cps_rpgd_fleet_relabel(cps_handle *h, int n_rows, const float *states_dev, const float *tp_dev, const float *te_dev,
                                      const float *L_dev, const float *m_pole_dev, const float *draws_dev, float *Q_out_dev,
                                      float *J_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    if (!states_dev || !Q_out_dev) return fail(h, CPS_ERR_INVALID, "cps_rpgd_fleet_relabel: null pointer");
    return rpgd_fleet_launch(h, "cps_rpgd_fleet_relabel", n_rows, tp_dev, te_dev, draws_dev, nullptr, J_out_dev, nullptr,
                             states_dev, L_dev, m_pole_dev, Q_out_dev);
}

extern "C" int cps_rpgd_fleet_get_states(cps_handle *h, float *s_host, float *u_prev_host) {
    if (!h) return CPS_ERR_INVALID;
    RpgdFleetState *F = h->rfleet;
    if (!F || !F->ready) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_rpgd_fleet_get_states: no RPGD fleet with states "
                                    "(cps_rpgd_fleet_create, cps_rpgd_fleet_set_states)");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc;
    if (s_host && (rc = fleet_states_to_host(h, F->d_s, s_host, F->E, "cps_rpgd_fleet_get_states")) != CPS_OK) return rc;
    if (u_prev_host)
        CUDA_TRY(h, cudaMemcpyAsync(u_prev_host, F->d_uprev, sizeof(float) * (size_t)F->E, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CPS_OK;
}

extern "C" int cps_rpgd_fleet_get_plans(cps_handle *h, float *Q_host, float *m_host, float *v_host, int *ages_host,
                                        long long *adam_iterations, long long *solves) {
    if (!h) return CPS_ERR_INVALID;
    RpgdFleetState *F = h->rfleet;
    if (!F || !F->ready) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_rpgd_fleet_get_plans: no RPGD fleet with states "
                                    "(cps_rpgd_fleet_create, cps_rpgd_fleet_set_states)");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t n = (size_t)F->E * F->K * F->T;
    if (Q_host) CUDA_TRY(h, cudaMemcpyAsync(Q_host, F->d_Q[F->cur], sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
    if (m_host) CUDA_TRY(h, cudaMemcpyAsync(m_host, F->d_m[F->cur], sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
    if (v_host) CUDA_TRY(h, cudaMemcpyAsync(v_host, F->d_v[F->cur], sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
    if (ages_host)
        CUDA_TRY(h, cudaMemcpyAsync(ages_host, F->d_ages[F->cur], sizeof(int) * (size_t)F->E * F->K, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (adam_iterations) *adam_iterations = F->adam_iterations;
    if (solves) *solves = F->solves;
    return CPS_OK;
}

extern "C" long long cps_rpgd_fleet_period(const cps_handle *h) { return (h && h->rfleet) ? h->rfleet->period : -1; }

extern "C" int cps_rpgd_fleet_draws(cps_handle *h, long long period, float *out_dev) {
    if (!h) return CPS_ERR_INVALID;
    RpgdFleetState *F = h->rfleet;
    if (!F) return fail(h, CPS_ERR_NOT_CONFIGURED, "cps_rpgd_fleet_draws: no RPGD fleet (cps_rpgd_fleet_create)");
    if (!out_dev || period < -1) return fail(h, CPS_ERR_INVALID, "cps_rpgd_fleet_draws: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    return draws_launch(h, F, period, out_dev);
}
