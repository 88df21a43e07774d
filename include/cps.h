/*
 * cps.h -- C ABI of the B200-native CartPole MPPI rollout path (libcps_b200.so).
 *
 * This is the drop-in boundary: plain C, opaque handle, raw pointers and sizes, no torch / numpy types.
 * The Python host side (cartpolesimulation_b200/) binds it with ctypes and mirrors the reference's plugin
 * interface (optimizer / predictor / cost-function objects) on top.  Citations are file:line relative to
 * the reference root (SensorsINI/CartPoleSimulation @ a5169e85 with its pinned submodules).
 *
 * Conventions
 *   - "dev" pointers are device pointers on the handle's device; "host" pointers are host memory (pinned
 *     memory makes the copies asynchronous; pageable memory is accepted and merely slower).
 *   - All calls are stream-ordered on the handle's stream (cps_set_stream; default: the legacy default
 *     stream).  *_host entry points synchronise the stream before returning; the others do not.
 *   - One in-flight call per handle (the reference is single-threaded per controller; its GUI may call
 *     step() from a worker thread, GUI/_CartPoleGUI_GuiActions.py:195-209).
 *   - Every function returns CPS_OK (0) or a cps_status error code; cps_last_error() gives the text.
 *     There is no CPU fallback anywhere: without a CUDA device cps_create fails with CPS_ERR_CUDA.
 *   - State vector layout (CartPole/state_utilities.py:5-23):
 *       [0] angle [1] angleD [2] angle_cos [3] angle_sin [4] position [5] positionD
 */
#ifndef CPS_H_
#define CPS_H_

#ifdef __cplusplus
extern "C" {
#endif

#define CPS_ABI_VERSION 1
#define CPS_STATE_DIM 6

typedef struct cps_handle cps_handle;

typedef enum cps_status {
    CPS_OK = 0,
    CPS_ERR_INVALID = 1,        /* bad argument / inconsistent configuration (reference: ValueError) */
    CPS_ERR_CUDA = 2,           /* CUDA runtime error, or no device (reference: n/a) */
    CPS_ERR_UNSUPPORTED = 3,    /* valid in the reference but not implemented here (NotImplementedError) */
    CPS_ERR_NOT_CONFIGURED = 4  /* e.g. cps_net_rollout before cps_net_load */
} cps_status;

/* Integrator variants (SURVEY.md fact 3):
 *  CPS_EULER_V0     predictor_ODE_v0: explicit Euler + edge bounce + fmod wrap
 *                   (CartPole/cartpole_numba.py:56-78, CartPole/cartpole_equations.py:341-364)
 *  CPS_EULER_CROMER predictor_ODE: semi-implicit Euler + atan2 wrap, no bounce
 *                   (CartPole/cartpole_equations.py:214-261,292-308)
 *  CPS_PREDICTOR_NEURAL predictor_autoregressive_neural: GRU / Dense network loaded with cps_net_load
 *                   (SI_Toolkit/src/SI_Toolkit/Predictors/predictor_autoregressive_neural.py:266-352) */
typedef enum cps_integrator { CPS_EULER_V0 = 0, CPS_EULER_CROMER = 1, CPS_PREDICTOR_NEURAL = 2 } cps_integrator;

/* Cost plugins (Control_Toolkit_ASF/Cost_Functions/CartPole/<name>.py) */
typedef enum cps_cost {
    CPS_COST_NONE = -1,
    CPS_COST_DEFAULT = 0,             /* default.py:19-88 */
    CPS_COST_QUADRATIC_BOUNDARY = 1,  /* quadratic_boundary.py:22-87 */
    CPS_COST_QB_GRAD_MINIMAL = 2,     /* quadratic_boundary_grad_minimal.py:17-140 */
    CPS_COST_QB_GRAD = 3,             /* quadratic_boundary_grad.py:17-268 */
    CPS_COST_LEGACY_MPPI = 4          /* q() + phi() of the legacy controller_mppi_cartpole
                                         (Control_Toolkit_ASF/Controllers/controller_mppi_cartpole.py:218-298); only with
                                         the cps_legacy_* entry points and CPS_NOISE_DIRECT */
} cps_cost;

/* Where the MPPI perturbations come from (Control_Toolkit/Optimizers/optimizer_mppi.py:169-178):
 *  CPS_NOISE_INDUCING  standard-normal draws at the n_ind inducing points; the kernel scales them by
 *                      SQRTRHODTINV and interpolates linearly in registers (Interpolator.py:53-106)
 *  CPS_NOISE_DIRECT    delta_u for every horizon step is supplied as is (post-interpolation injection) */
typedef enum cps_noise_mode { CPS_NOISE_INDUCING = 0, CPS_NOISE_DIRECT = 1 } cps_noise_mode;

/* Memory order of per-rollout arrays.
 *  *_ROLLOUT_MAJOR is the reference's order ([K][n_ind] noise, [B][T] controls, [B][T+1][6] trajectories);
 *  *_TIME_MAJOR is the coalesced order the kernels prefer ([n_ind][K], [T][B], [T+1][6][B]). */
typedef enum cps_layout { CPS_ROLLOUT_MAJOR = 0, CPS_TIME_MAJOR = 1 } cps_layout;

/* cps_config.flags.  Default (flags = 0): "rotation" substeps -- (cos, sin) are advanced with the angle-addition
 * formulas by the substep increment h*angleD and re-derived from the (compensated) angle with sincosf once per
 * control step; as accurate as evaluating sincosf every substep (DESIGN.md "rotation mode"), far fewer instructions. */
#define CPS_FLAG_FAST_SINCOS 0x1u     /* with SUBSTEP_SINCOS: MUFU.SIN/COS (__sincosf) instead of the 1-ulp sincosf */
#define CPS_FLAG_EXACT_ATAN2 0x2u     /* with SUBSTEP_SINCOS, Euler-Cromer: wrap by atan2f(sin, cos) as the reference
                                         writes it, instead of the mathematically identical +-2*pi fold */
#define CPS_FLAG_FAST_DIV 0x4u        /* MUFU.RCP without the Newton step in the ODE right-hand side */
#define CPS_FLAG_SUBSTEP_SINCOS 0x8u  /* evaluate sin/cos of the angle in EVERY substep, literally as
                                         cartpole_equations.py:245-248 / cartpole_numba.py:66-76 do */

#define CPS_FLAG_NO_PAIRS 0x40u         /* rollouts, large-K solves, fleets: never use the two-per-thread packed-FP32 kernels
                                           (per rollout they execute the same arithmetic; the flag exists for A/B timing) */
#define CPS_PAIR_MIN_BATCH 262144       /* smallest batch the packed-pair rollout kernel is used for */
#define CPS_MPPI_PAIR_MIN_ROLLOUTS 65536 /* cps_mppi_step: from this K on (even K, native noise order, no logging outputs)
                                           the solve runs two rollouts per thread in packed FP32 */
#define CPS_FLAG_NET_TENSOR_CORES 0x10u /* neural predictor: force the tcgen05 tensor-core kernel (2 x 64 GRU only) */
#define CPS_FLAG_NET_FP32 0x20u         /* neural predictor: force the FP32 CUDA-core kernel (default: tensor cores for 2 x 64 GRU) */

typedef struct cps_config {
    int struct_size;      /* = sizeof(cps_config), ABI check */
    int device;           /* CUDA device ordinal */
    int num_rollouts;     /* K, optimizer_mppi num_rollouts (config_optimizers.yml:91) */
    int horizon;          /* T, mpc_horizon (:89) */
    int substeps;         /* n, intermediate_steps (SI_Toolkit_ASF/config_predictors.yml:21,25) */
    float dt;             /* mpc_timestep (config_optimizers.yml:90); substep h = dt / n */
    int integrator;       /* cps_integrator */
    int cost_id;          /* cps_cost */
    int noise_mode;       /* cps_noise_mode */
    int interp_period;    /* p, period_interpolation_inducing_points (config_optimizers.yml:97) */
    unsigned flags;       /* CPS_FLAG_* */
} cps_config;

/* Physical parameters, fp32-rounded by the caller as CartPole/cartpole_parameters.py:27-29 does.
 * Index order of the p[] vector given to cps_set_physics: */
enum {
    CPS_PH_K = 0, CPS_PH_M_CART, CPS_PH_M_POLE, CPS_PH_G, CPS_PH_J_FRIC, CPS_PH_M_FRIC, CPS_PH_L, CPS_PH_U_MAX,
    CPS_PH_TRACK_HALF_LENGTH, CPS_PH_COUNT
};

/* ---- lifetime -------------------------------------------------------------------------------------- */
/* Replaces the construction done by controller_mpc.configure (Control_Toolkit/Controllers/controller_mpc.py:42-92):
 * optimizer + predictor + cost wrapper for one (K, T, n, integrator, cost) configuration.  Physics defaults to
 * cartpole_physical_parameters.yml:6-17,33-42, cost weights to config_cost_function.yml:5-58 and MPPI parameters
 * to config_optimizers.yml:87-97 until the cps_set_* calls override them.  The handle owns all scratch
 * (block partials, ticket, staging buffers); no allocation happens in the step / rollout calls on device buffers
 * (cps_rollout_host is the exception: its staging buffers grow on first use / on a larger batch, see below). */
int cps_create(const cps_config *cfg, cps_handle **out);
void cps_destroy(cps_handle *h);
/* Text of the last error on this handle (h == NULL: last cps_create failure on the calling thread). */
const char *cps_last_error(const cps_handle *h);
int cps_abi_version(void);
/* Number of inducing points ceil((T-1)/p)+1 (Control_Toolkit/others/Interpolator.py:79-84). */
int cps_num_inducing_points(int horizon, int period);
int cps_set_stream(cps_handle *h, void *cuda_stream /* cudaStream_t */);

/* ---- parameters (cheap; may be called between any two steps) ------------------------------------------- */
/* CartPoleParameters (CartPole/cartpole_parameters.py:8-31). */
int cps_set_physics(cps_handle *h, const float *p, int n /* = CPS_PH_COUNT */);
/* Cost weights in the per-plugin order documented in DESIGN.md "cost parameter vectors"; the hot-reload hook of
 * cost_function_wrapper.update_cost_parameters_from_config (cost_function_wrapper.py:71-74). */
int cps_set_cost_params(cps_handle *h, const float *w, int n);
/* optimizer_mppi.__init__/configure (optimizer_mppi.py:16-138): sqrt_rho_dt_inv = SQRTRHOINV / sqrt(dt) (:130). */
int cps_set_mppi_params(cps_handle *h, float cc_weight, float R, float LBD, float NU, float sqrt_rho_dt_inv,
                        float action_low, float action_high);
/* variable_parameters that may change every control tick (CartPole/__init__.py:512-519):
 * target_position, target_equilibrium for the cost; L and m_pole for the ODE (m_pole is ignored by
 * CPS_EULER_V0, predictors_customization_v0.py:47-54 reads only L). */
int cps_set_variable_parameters(cps_handle *h, float target_position, float target_equilibrium, float L,
                                float m_pole);

/* ---- the hot path: one MPPI solve ------------------------------------------------------------------- */
/* optimizer_mppi._predict_and_cost (optimizer_mppi.py:180-192) as ONE kernel launch: warm-start shift, noise
 * interpolation, clip, K rollouts over T x n substeps, stage + terminal + MPPI-correction cost, exp-weighted update,
 * clip.  s_dev [6]; noise_dev: INDUCING -> n_ind x K standard-normal draws, DIRECT -> T x K delta_u, in
 * `noise_layout` order; u_prev = the last returned control (optimizer_mppi.py:210; 0.0 initially,
 * Optimizers/__init__.py:35); u_nom_dev [T] in/out (the reference's self.u_nom: NOT pre-shifted; the shift
 * happens at the start of the next solve, :183); u_out_dev [1] = u_nom[0] after the update.
 * Optional logging outputs (NULL to skip; optimizer_logging, :205-217): J_out_dev [K],
 * traj_out_dev (K x (T+1) x 6 in traj_layout order), u_run_out_dev ([K][T]). */
int cps_mppi_step(cps_handle *h, const float *s_dev, const float *noise_dev, int noise_layout, float u_prev,
                  float *u_nom_dev, float *u_out_dev, float *J_out_dev, float *traj_out_dev, int traj_layout,
                  float *u_run_out_dev);

/* Host-buffer form of the same call, the one the reference-facing optimizer.step(s) makes: s_host [6] is copied
 * up, the control comes back in *u_out_host; u_nom lives in the handle (cps_mppi_reset zeroes it like
 * optimizer_reset, optimizer_mppi.py:226-230).  noise_dev stays a DEVICE pointer: the draws are produced on the
 * device (the reference draws them inside step() too, :169-175).  Synchronises.  With the ODE predictors this is ONE
 * operation on the stream: the state travels in the kernel's parameter block and the control is written by the kernel
 * into mapped pinned host memory (no copy in either direction). */
int cps_mppi_step_host(cps_handle *h, const float *s_host, const float *noise_dev, int noise_layout, float u_prev,
                       float *u_out_host);
int cps_mppi_reset(cps_handle *h, float u_nom_init);
int cps_mppi_get_u_nom(cps_handle *h, float *u_nom_host /* [T] */);
int cps_mppi_set_u_nom(cps_handle *h, const float *u_nom_host /* [T] */);
float *cps_mppi_u_nom_dev(cps_handle *h);

/* K sharded over several GPUs (SURVEY.md 8e): with cps_mppi_set_shard(h, 1) cps_mppi_step stops after the local
 * reduction and writes the rank's partial (min J, sum w, sum w*noise[.]) = cps_mppi_partial_size() floats to
 * partial_out_dev; the ranks exchange them (all-gather) and each calls cps_mppi_finalize on the gathered
 * [n_ranks][size] array to obtain the identical u_nom / u. */
int cps_mppi_set_shard(cps_handle *h, int enabled, float *partial_out_dev);
int cps_mppi_partial_size(const cps_handle *h);
int cps_mppi_finalize(cps_handle *h, const float *partials_dev, int n_ranks, float *u_nom_dev, float *u_out_dev);

/* The same sharding with the exchange INSIDE the solve launch, over peer memory (NVLink / NVSwitch): every rank owns an
 * exchange buffer of cps_mppi_peer_buffer_floats(h, world) zero-initialised floats that all ranks have mapped (CUDA IPC /
 * virtual-memory handles, e.g. torch.distributed._symmetric_memory); peer_bufs_host[r] is rank r's buffer as mapped on
 * THIS device.  After cps_mppi_set_peers every cps_mppi_step (one launch) pushes the rank's partial record into all
 * ranks' buffers, waits for theirs and finishes the update itself: u_nom / u are bit-identical on all ranks, no
 * collective call and no second launch.  All ranks must call cps_mppi_step the same number of times.  world <= 1 (or
 * peer_bufs_host == NULL) switches the exchange off.  Excludes cps_mppi_set_shard.  The reference has no counterpart
 * (one process per experiment, others/EulerClusterScripts/ParallelDataGeneration.sh). */
#define CPS_MAX_PEERS 8
long long cps_mppi_peer_buffer_floats(const cps_handle *h, int world);
int cps_mppi_set_peers(cps_handle *h, int world, int rank, float *const *peer_bufs_host);
/* Waits on a peer's record that were given up after 10 s (a rank that never called cps_mppi_step); 0 in a healthy run.
 * Synchronises. */
int cps_mppi_peer_timeouts(cps_handle *h, int *count_out);

/* ---- legacy front-end: controller_mppi_cartpole ------------------------------------------------------------ */
/* The repository's original MPPI controller (Control_Toolkit_ASF/Controllers/controller_mppi_cartpole.py), which
 * README.md:46 calls "MPPI with predictor_ODE_v0".  Same rollouts, different bookkeeping (SURVEY.md 8f, row f2):
 *   - delta_u [K][T] is drawn on the host by one of five sampling types (:392-457) and passed in as is;
 *   - the rollouts run on u + delta_u WITHOUT clipping (:190-192);
 *   - cost = SUM over the T stage costs q() (:218-268: dd with a 1e6 track-edge indicator at 0.95, ep, ekp, ekc,
 *     cc = cc_weight*(0.5(1-1/NU) R du^2 + R u du + 0.5 R u^2) on the NOMINAL u, replaced by 1e5 where |u+du| > 1,
 *     ccrc against the PREVIOUS nominal sequence u_prev[t]) + phi() (:271-298);
 *   - u += sum(w du)/sum(w), not clipped (:301-335); the controller returns u[0]; afterwards u_prev <- u and u is
 *     shifted left with a ZERO appended (:534-539).
 * Handle: cost_id = CPS_COST_LEGACY_MPPI, noise_mode = CPS_NOISE_DIRECT.  cps_set_cost_params takes
 * [dd_weight, ep_weight, ekp_weight, ekc_weight, ccrc_weight] (config_controllers.yml:16-21); cc_weight, R, LBD, NU come
 * from cps_set_mppi_params (its sigma and limits are unused: the host draws delta_u and clips the returned control).
 * The handle owns u [T] and u_prev [T] (both zero after cps_create / cps_legacy_reset).
 *
 * One update_every-th iteration (:481-500 + :530-539) as ONE kernel launch.  s_dev [6]; delta_u_dev K x T in `layout`
 * order; u_out_dev [1] = u[0] after the update (before actuator noise and clipping, which stay on the host, :526-528).
 * Optional outputs (NULL to skip): S_out_dev [K] = S_tilde_k; traj_out_dev K x (T+1) x 6 in traj_layout order;
 * u_upd_out_dev [T] = u after the update, before the shift (what LOGS["inputs"] records, :503). */
int cps_legacy_step(cps_handle *h, const float *s_dev, const float *delta_u_dev, int layout, float *u_out_dev,
                    float *S_out_dev, float *traj_out_dev, int traj_layout, float *u_upd_out_dev);
/* Host-buffer form, what controller_mppi_cartpole.step makes per call: s_host [6] and delta_u_host (K x T, `layout`
 * order; pinned memory makes the copy asynchronous) are copied up, *u_out_host = u[0].  Synchronises. */
int cps_legacy_step_host(cps_handle *h, const float *s_host, const float *delta_u_host, int layout, float *u_out_host);
/* The same solve with SAMPLING_TYPE "interpolated" (controller_mppi_cartpole.py:430-451) expanded on the device: knots_host
 * [K][n_knots] are the draws at the horizon indices 0, knot_step, 2 knot_step, ... (already scaled and rounded to float32
 * as the reference's assignment into its float32 array does); the steps between are filled with scipy interp1d's linear
 * formula in float64, bit-identical to the host path.  Moves K n_knots floats instead of K T and takes scipy off the
 * controller's critical path.  cps_legacy_get_perturbations: the [K][T] perturbations of the last host-form step. */
int cps_legacy_step_host_knots(cps_handle *h, const float *s_host, const float *knots_host, int n_knots, int knot_step,
                               float *u_out_host);
int cps_legacy_get_perturbations(cps_handle *h, float *delta_u_host);
/* An iteration that is not a multiple of update_every (:481): no solve; u_out = u[0], u_prev <- u, shift.  u_out_host
 * may be NULL.  Synchronises only if u_out_host is given. */
int cps_legacy_advance(cps_handle *h, float *u_out_host);
int cps_legacy_reset(cps_handle *h);
/* u [T] and u_prev [T]; either pointer may be NULL.  Synchronise. */
int cps_legacy_get_inputs(cps_handle *h, float *u_host, float *u_prev_host);
int cps_legacy_set_inputs(cps_handle *h, const float *u_host, const float *u_prev_host);

/* ---- Legacy controller fleet: E closed-loop experiments under controller_mppi_cartpole ------------------------- */
/* The data generator with the legacy controller (`mppi-cartpole`, Control_Toolkit_ASF/config_controllers.yml:9-30): per
 * controller period every experiment does what one controller_mppi_cartpole_b200.step does from its own state, u [T],
 * u_prev [T] and target position, then the plant advances one period.
 *   - Solve periods ((period - reset period) % update_every == 0): the K x T perturbations of the configured sampling type
 *     from the experiment's raw draws, then the iteration of cps_legacy_step (unclipped rollouts, q() + phi(), the
 *     exp-weighted unclipped update, Q = u[0], u_prev <- u, zero-fill shift).  Other periods: cps_legacy_advance's shift.
 *   - Actuator noise: Q <- fl32(Q (1 + p_Q v)) in float64 with v uniform in [-1, 1), then Q clipped to [-1, 1] (NaN kept).
 *   - The plant period with Q held and the record row of cps_fleet_step with Q_calculated = Q_applied = that Q.
 * Perturbations from the raw draws (stdev = SQRTRHOINV / sqrt(dt), float64; products and sums in float64, rounded to
 * float32 where the reference assigns into its float32 array): IID T normals z, du_t = fl32(stdev z_t); RANDOM_WALK
 * T normals, du_0 = fl32(stdev z_0), du_t = fl32(du_{t-1} + stdev z_t); UNIFORM T uniforms v in [-1, 1), du_t = v_t;
 * REPEATED one normal, du_t = fl32(stdev z); INTERPOLATED ceil(T / 10) + 1 normals, knots fl32(stdev z_j) at t = 0, 10,
 * 20, ... and the linear formula of cps_legacy_step_host_knots between them.
 * Draws: supplied (CPS_FLEET_NOISE_SUPPLIED) raw draws [n_periods][E][K][n_draws] (read in solve periods only) and
 * actuator uniforms [n_periods][E]; or generated from Philox4x32-10 (CPS_FLEET_NOISE_PHILOX, key = seed) in the rollout
 * threads, counter (rollout k, LEGACY tag + group of four draws, period, experiment_offset + e), and for the actuator
 * uniform (0, LEGACY actuator tag, period, experiment_offset + e), disjoint from the other fleets' streams.  A Philox
 * uniform is -1 + 2 ((word >> 8) 2^-24), the multiply and the add rounded separately.
 * One launch per period, whatever E (cps_launch_count): solve periods grid (blocks of cps_legacy_step for K, E), each
 * experiment's partials and merge those of cps_legacy_step; other periods one thread per experiment.
 * The handle: cost CPS_COST_LEGACY_MPPI (any other: CPS_ERR_NOT_CONFIGURED), predictor CPS_EULER_CROMER or CPS_EULER_V0,
 * weights from cps_set_cost_params / cps_set_mppi_params, folded at each cps_legacy_fleet_step; L / m_pole of the
 * controller's model are the handle's.  The legacy cost has no target equilibrium: te_dev is only recorded.
 * n_experiments above 65535, an unknown sampling type, update_every < 1 or dt not a multiple of dt_simulation:
 * CPS_ERR_INVALID; a horizon whose perturbations do not fit shared memory: CPS_ERR_UNSUPPORTED.  Non-finite costs (e.g.
 * from a NaN target) stay in their experiment and are counted (cps_nonfinite_costs). */
enum {
    CPS_LEGACY_SAMPLING_IID = 0,            /* the reference's default branch */
    CPS_LEGACY_SAMPLING_RANDOM_WALK = 1,
    CPS_LEGACY_SAMPLING_UNIFORM = 2,
    CPS_LEGACY_SAMPLING_REPEATED = 3,
    CPS_LEGACY_SAMPLING_INTERPOLATED = 4    /* the shipped SAMPLING_TYPE */
};
typedef struct cps_legacy_fleet_config {
    int struct_size;                 /* = sizeof(cps_legacy_fleet_config) */
    int n_experiments;               /* E on this device, at most 65535 */
    int sim_substeps;                /* plant ticks per controller period */
    int draw_source;                 /* CPS_FLEET_NOISE_SUPPLIED | CPS_FLEET_NOISE_PHILOX */
    double dt_simulation;            /* plant tick, 0.002 s */
    unsigned long long seed;
    long long experiment_offset;     /* global index of local experiment 0 (Philox counters) */
    int sampling_type;               /* CPS_LEGACY_SAMPLING_* */
    int update_every;                /* solve every update_every-th period after a reset */
    double stdev;                    /* SQRTRHOINV * (1 / sqrt(dt)) as the mirror computes it */
    double p_Q;                      /* actuator_noise */
} cps_legacy_fleet_config;
int cps_legacy_fleet_create(cps_handle *h, const cps_legacy_fleet_config *cfg);
/* Every experiment as a freshly configured controller (u = u_prev = 0, the iteration counter restarted so that `period`
 * solves); states s_host [E][6]; the period counter.  Synchronises. */
int cps_legacy_fleet_set_states(cps_handle *h, const float *s_host, long long period);
/* s_host [E][6] and Q_host [E] (each experiment's last control, after the actuator noise); either may be NULL.
 * Synchronises. */
int cps_legacy_fleet_get_states(cps_handle *h, float *s_host, float *Q_host);
/* u_host and u_prev_host [E][T] (u already shifted for the next period); either may be NULL.  Synchronises. */
int cps_legacy_fleet_get_inputs(cps_handle *h, float *u_host, float *u_prev_host);
/* n_periods controller periods, stream-ordered, no synchronisation.  tp_dev / te_dev [n_periods][E] or NULL (0 / +1);
 * draws_dev [n_periods][E][K][n_draws] and act_draws_dev [n_periods][E] as above (NULL on a Philox fleet);
 * record_dev [n_periods][E][CPS_FLEET_RECORD] and S_out_dev [n_periods][E][K] (rollout costs, written in solve periods)
 * may be NULL. */
int cps_legacy_fleet_step(cps_handle *h, int n_periods, const float *tp_dev, const float *te_dev, const float *draws_dev,
                          const float *act_draws_dev, float *record_dev, float *S_out_dev);
/* What a Philox fleet draws in controller period `period`: the raw draws out_dev [E][K][n_draws] (n_draws = T, or 1 for
 * REPEATED, ceil(T / 10) + 1 for INTERPOLATED), the actuator uniforms out_dev [E], and the perturbations out_dev
 * [E][K][T] made from the raw draws by the rollouts' own transform (Philox fleets only). */
int cps_legacy_fleet_draws(cps_handle *h, long long period, float *out_dev);
int cps_legacy_fleet_act_draws(cps_handle *h, long long period, float *out_dev);
int cps_legacy_fleet_perturbations(cps_handle *h, long long period, float *out_dev);
long long cps_legacy_fleet_period(const cps_handle *h);

/* ---- open-loop batched rollouts (the predictor interface) ------------------------------------------------ */
/* predictor.predict_core(s, Q) (SI_Toolkit/src/SI_Toolkit/Predictors/predictor_ODE.py:86-97,
 * predictor_ODE_v0.py:42-74): B rollouts of T control steps x n substeps.  s0_dev: [B][6] if s0_batched else [6]
 * (tiled, predictor_ODE_v0.py:59-60); Q_dev: B x T in q_layout order; traj_out_dev: B x (T+1) x 6 in traj_layout
 * order, row 0 = s0 (may be NULL); final_out_dev: [B][6] last state (may be NULL).  B and T are free per call
 * (B is not tied to cfg.num_rollouts). */
int cps_rollout(cps_handle *h, const float *s0_dev, int s0_batched, const float *Q_dev, int q_layout, int B, int T,
                float *traj_out_dev, int traj_layout, float *final_out_dev);
/* Host-buffer form: copies s0 and Q up, runs, copies the requested outputs back, synchronises.  Uses handle-owned
 * device buffers that grow on demand (the only *_host call that may allocate, on first use / growth). */
int cps_rollout_host(cps_handle *h, const float *s0_host, int s0_batched, const float *Q_host, int q_layout, int B,
                     int T, float *traj_out_host, int traj_layout, float *final_out_host);

/* ---- autoregressive neural predictor (GRU / Dense) ------------------------------------------------------ */
/* What predictor_autoregressive_neural.__init__ derives from the net-info file, the normalisation table and the
 * checkpoint (predictor_autoregressive_neural.py:163-231, Functions/General/Normalising.py:15-186):
 * the network consumes [control, state features in_idx[0..n_state_in)] and produces the state features
 * out_idx[0..n_out); inputs are normalised x = a*v + b, outputs de-normalised v = A*y + B; missing features are
 * zero; angle = atan2(sin, cos) (or sin/cos of a predicted angle) is appended
 * (SI_Toolkit_ASF/ToolkitCustomization/predictors_customization.py:71-139).
 * differential != 0 (outputs named D_*; Predictors/autoregression.py:118-158): the network predicts normalised
 * derivatives; the normalised state advances by diff_p1*y + diff_p2 per step from the normalised initial values
 * out_norm_a*s[out_idx]+out_norm_b, and net input i is fed from integrated output out_to_in[i]. */
#define CPS_NET_MAX_LAYERS 4
#define CPS_NET_GRU 0
#define CPS_NET_DENSE 1
typedef struct cps_net_desc {
    int struct_size;                 /* = sizeof(cps_net_desc) */
    int net_type;                    /* CPS_NET_GRU (torch GRUCell / keras GRU reset_after) | CPS_NET_DENSE (tanh MLP) */
    int n_layers;                    /* hidden layers (<= CPS_NET_MAX_LAYERS); a linear output layer follows */
    int hidden[CPS_NET_MAX_LAYERS];  /* units per hidden layer (each <= 128) */
    int n_state_in;                  /* state features among the net inputs (<= 6); inputs = 1 + n_state_in */
    int in_idx[6];                   /* their indices into the 6-vector state */
    int n_out;                       /* net outputs (<= 6) */
    int out_idx[6];
    float norm_a[7], norm_b[7];      /* [0] control input, [1 + i] state input i */
    float denorm_A[6], denorm_B[6];
    int differential;
    float diff_p1[6], diff_p2[6], out_norm_a[6], out_norm_b[6];
    int out_to_in[6];
} cps_net_desc;

/* Weights, float32, concatenated per hidden layer -- GRU: w_ih [3H][in], w_hh [3H][H], b_ih [3H], b_hh [3H] in torch
 * GRUCell order (gates r, z, n; Functions/Pytorch/Network.py:146-148); Dense: w [H][in], b [H] -- then the output
 * layer w [n_out][H_last], b [n_out].  Copies them to the device in the kernels' layout and zeroes the stored hidden
 * state (net.reset_internal_states(), predictor_autoregressive_neural.py:112-113).  May allocate. */
int cps_net_load(cps_handle *h, const cps_net_desc *desc, const float *weights_host, long long n_weights);
/* predictor.predict_core(s, Q) (predictor_autoregressive_neural.py:266-313): like cps_rollout.  h0_dev: initial
 * hidden state, concatenated over the layers -- NULL: the handle's stored state (memory_states_ref, :291), else
 * [Htot] shared or [B][Htot] if h0_batched.  h_final_dev: optional [B][Htot] hidden state after the T steps. */
int cps_net_rollout(cps_handle *h, const float *s0_dev, int s0_batched, const float *Q_dev, int q_layout, int B, int T,
                    const float *h0_dev, int h0_batched, float *traj_out_dev, int traj_layout, float *h_final_dev);
/* update_internal_state_tf (:332-352): advance the stored hidden state by one network step on the measured state
 * s_dev [6] and the applied control q0_dev [1] (both DEVICE pointers).  No-op for Dense networks.  cps_mppi_step
 * with CPS_PREDICTOR_NEURAL does this itself after the solve (optimizer_mppi.py:191) unless K is sharded. */
int cps_net_update(cps_handle *h, const float *s_dev, const float *q0_dev);
int cps_net_state_size(const cps_handle *h);                       /* Htot (0 for Dense), -1 if no net is loaded */
int cps_net_reset_state(cps_handle *h);
int cps_net_get_state(cps_handle *h, float *state_host /* [Htot] */);
int cps_net_set_state(cps_handle *h, const float *state_host /* [Htot] */);

/* ---- standalone cost plugin (for the other optimizers; CostFunctionWrapper interface) ---------------------- */
/* get_trajectory_cost (Control_Toolkit/Cost_Functions/__init__.py:74-93): traj_dev [K][T+1][6], Q_dev [K][T]
 * (reference order) -> J_dev [K] = mean over the T+1 entries (stage - MAX_COST ..., terminal). */
int cps_trajectory_cost(cps_handle *h, const float *traj_dev, const float *Q_dev, float u_prev, int K, int T,
                        float *J_dev);
/* get_stage_cost (:49-64): states_dev [K][rows][6] with rows = T (the reference passes state_horizon[:, :-1, :]) or
 * T+1 (a whole trajectory, last row ignored) -> stage_dev [K][T]; unshifted != 0 gives _get_stage_cost (no MAX_COST). */
int cps_stage_cost(cps_handle *h, const float *states_dev, int rows, const float *Q_dev, float u_prev, int K, int T,
                   int unshifted, float *stage_dev);

/* get_terminal_cost (default.py:44-68 etc.): states_dev [K][6] -> out_dev [K]. */
int cps_terminal_cost(cps_handle *h, const float *states_dev, int K, float *out_dev);

/* ---- fleet: E independent closed-loop experiments advanced together ---------------------------------------- */
/* BASELINE configs[4] (data_generator: 8192 independent MPPI-controlled cartpoles).  What run_data_generator does
 * for ONE cartpole per process (CartPole/data_generator.py via CartPole/__init__.py:659-739: every dt_controller
 * the controller solves, then the plant -- CartPole.update_state, :283-324 -- advances sim_substeps ticks of
 * dt_simulation with the control held) happens here for E cartpoles per launch, on the device, with no host round
 * trip between periods.  Each experiment owns its state, nominal inputs u_nom[T], last control, targets and noise
 * stream; the handle's (K, T, n, integrator, cost, MPPI parameters) are shared.  The plant uses the handle's physical
 * parameters (cps_set_physics); the controller's model uses L / m_pole from cps_set_variable_parameters.
 * Control disturbance, measurement noise and latency (all off in the shipped configuration,
 * cartpole_physical_parameters.yml:13-24): cps_fleet_set_plant_models below. */
#define CPS_FLEET_NOISE_SUPPLIED 0  /* caller passes standard-normal draws [period][E][n_ind][K] */
#define CPS_FLEET_NOISE_PHILOX 1    /* drawn in the kernel: Philox4x32-10 + Box-Muller, counter = (rollout, draw group,
                                       period, experiment_offset + e), key = seed; cps_fleet_noise materialises them */
#define CPS_FLEET_RECORD 16         /* floats per record row: time, angle, angleD, angleDD, angle_cos, angle_sin, position,
                                       positionD, positionDD, Q_calculated, Q_applied, u, target_position,
                                       target_equilibrium, 0, 0 (the CSV columns of CartPole/__init__.py:221-258) */
typedef struct cps_fleet_config {
    int struct_size;                 /* = sizeof(cps_fleet_config) */
    int n_experiments;               /* E on this device */
    int sim_substeps;                /* plant ticks per controller period: dt.control / dt.simulation (config_data_gen.yml:25-27) */
    int noise_source;                /* CPS_FLEET_NOISE_* */
    double dt_simulation;            /* plant tick, 0.002 s */
    unsigned long long seed;
    long long experiment_offset;     /* global index of local experiment 0 (sharding over GPUs) */
} cps_fleet_config;
/* CPS_ERR_INVALID: n_experiments outside [1, 65535], sim_substeps < 1, dt_simulation <= 0, an unknown noise source, or dt
 * (control) not sim_substeps x dt_simulation. */
int cps_fleet_create(cps_handle *h, const cps_fleet_config *cfg);
/* s_host [E][6]: initial states (angle_cos / angle_sin are taken as given).  Zeroes u_nom and the last control
 * (optimizer_reset + Q_ccrc = 0, CartPole/__init__.py:871) and sets the period counter. */
int cps_fleet_set_states(cps_handle *h, const float *s_host, long long period);
/* Any of the outputs may be NULL: s_host [E][6], u_nom_host [E][T], u_prev_host [E].  Synchronises. */
int cps_fleet_get_states(cps_handle *h, float *s_host, float *u_nom_host, float *u_prev_host);
long long cps_fleet_period(const cps_handle *h);
/* Advance every experiment by n_periods controller periods (one launch each, stream-ordered, no synchronisation).
 * tp_dev / te_dev: [n_periods][E] target position / equilibrium seen by the controller in each period (NULL: 0 / +1;
 * the reference evaluates random_track_f(time) and the up/down flip schedule on the plant tick that precedes the
 * solve, CartPole/__init__.py:360-388); noise_dev: [n_periods][E][n_ind][K] for CPS_FLEET_NOISE_SUPPLIED, else NULL;
 * record_dev: [n_periods][E][CPS_FLEET_RECORD] (row = state at the START of the period with the control chosen for
 * it, what save_csv_routine logs at dt_save = dt_controller) or NULL; J_out_dev: [n_periods][E][K] or NULL. */
int cps_fleet_step(cps_handle *h, int n_periods, const float *tp_dev, const float *te_dev, const float *noise_dev,
                   float *record_dev, float *J_out_dev);
/* Plant-side models between plant and controller (CartPole/__init__.py:336-340, 523-524):
 *   control disturbance  add_control_noise (CartPole/noise_control_signal.py:5-26): the plant is driven by
 *                        Q_applied = Q + mult * n + add (additive, n standard normal, float32, not clipped) or by a draw of
 *                        truncnorm(loc = Q + add, scale = mult) on [-1, 1]; the optimizer's own last control stays Q;
 *   measurement noise    NoiseAdder.add_noise_to_measurement (CartPole/noise_adder.py:69-84): sigma * standard normal on
 *                        angle (then wrapped), position, angleD, positionD of the state handed to the controller;
 *   latency              LatencyAdder (CartPole/latency_adder.py:10-74): the controller sees the state `latency` seconds
 *                        late, linearly interpolated between the two neighbouring plant ticks (ring buffer that starts as
 *                        zeros with cos = 1); cos / sin of the observation are recomputed from its angle.
 * The record rows keep the TRUE state (what the reference's CSV logs) with Q_calculated and Q_applied side by side.
 * Call after cps_fleet_create; cps_fleet_set_states restarts the observation chain: empty latency buffer, and the first
 * solve sees the true state, as the controller call at t = 0 does (CartPole/__init__.py:869-880).  Draws: a Philox fleet generates them in the
 * kernel (counters disjoint from the rollout draws); cps_fleet_step_noisy takes them from the caller -- ctrl_draws_dev
 * [n_periods][E] (standard normal for additive, uniform in (0, 1) for truncnorm), meas_draws_dev
 * [n_periods][sim_substeps][E][4] standard normals per plant tick in the reference's call order (angle, position, angleD,
 * positionD; the draws of the last tick of a period reach the controller); either may be NULL on a Philox fleet. */
typedef struct cps_fleet_plant_models {
    int struct_size;                 /* = sizeof(cps_fleet_plant_models) */
    int control_noise_mode;          /* 0 OFF, 1 additive, 2 truncnorm (controlDisturbance_mode) */
    float control_noise_mult;        /* controlDisturbance */
    float control_noise_add;         /* controlBias */
    int measurement_noise;           /* noise_mode != 'OFF' */
    float sigma_angle, sigma_position, sigma_angleD, sigma_positionD;
    double latency;                  /* seconds */
} cps_fleet_plant_models;
int cps_fleet_set_plant_models(cps_handle *h, const cps_fleet_plant_models *m);
int cps_fleet_get_observed(cps_handle *h, float *obs_host /* [E][6] */);
int cps_fleet_step_noisy(cps_handle *h, int n_periods, const float *tp_dev, const float *te_dev, const float *noise_dev,
                         float *record_dev, float *J_out_dev, const float *ctrl_draws_dev, const float *meas_draws_dev);
/* Offline relabelling (SURVEY 8f row f4): add_control_along_trajectories
 * (SI_Toolkit/src/SI_Toolkit/General/preprocess_data_add_control_along_trajectories.py:53-140) calls controller.step once
 * per recorded row -- `updated_attributes` first, then one solve from the recorded state -- sequentially within a file
 * (the optimizer keeps its warm start and last control) and independently across files (the reference runs a 120-way
 * SLURM array, others/EulerClusterScripts/ControllerAlongTrajectories.sh).  Here E files advance in lockstep, one
 * launch per row: states_dev [n_rows][E][6] recorded states; tp_dev / te_dev / L_dev / m_pole_dev [n_rows][E] the
 * row's attributes (NULL: 0 / +1 / the handle's L / m_pole; ODE_v0 ignores m_pole as the reference does);
 * noise_dev as in cps_fleet_step; Q_out_dev [n_rows][E] the controls; J_out_dev as in cps_fleet_step or NULL.
 * The fleet's plant state is not touched.  Rows of a Monte-Carlo integration over an attribute (:118-128, 64
 * evaluations per recorded row by default) are simply consecutive rows here; the caller averages.
 * cps_fleet_reset: controller.reset() for every file (zero warm start and last control) + the period counter. */
int cps_fleet_relabel(cps_handle *h, int n_rows, const float *states_dev, const float *tp_dev, const float *te_dev,
                      const float *L_dev, const float *m_pole_dev, const float *noise_dev, float *Q_out_dev,
                      float *J_out_dev);
/* The same with a per-row, per-file mask active_dev [n_rows][E] (int; NULL: all active): a file whose entry is 0 sits
 * the row out -- its warm start, last control and Q_out entry stay untouched.  Used by the adaptive quadrature of
 * integration(method='nquad') (:346-362), where every file asks for a different number of controller steps per row. */
int cps_fleet_relabel_masked(cps_handle *h, int n_rows, const float *states_dev, const float *tp_dev, const float *te_dev,
                             const float *L_dev, const float *m_pole_dev, const float *noise_dev, float *Q_out_dev,
                             float *J_out_dev, const int *active_dev);
int cps_fleet_reset(cps_handle *h, long long period);
/* The draws CPS_FLEET_NOISE_PHILOX uses in controller period `period`: out_dev [E][n_ind][K]. */
int cps_fleet_noise(cps_handle *h, long long period, float *out_dev);
/* Fleets with the neural predictor (CPS_PREDICTOR_NEURAL; cps_net_load before cps_fleet_create, else
 * CPS_ERR_NOT_CONFIGURED).  The network lives in the controller only; the plant stays the CartPole ODE.  Each experiment
 * owns a hidden state [Htot] besides its state, warm start and last control.  A period does, per experiment, what
 * cps_mppi_step does with the network -- shifted warm start, its own draws, targets, u_prev and hidden state shared by its K
 * rollouts, merge, then the hidden state advanced one step on (u, s) (optimizer_mppi.py:191,194-196; Dense networks keep
 * it) -- and then the plant period with the record row of fleets on the ODE predictors (Q_applied = Q).  The solve of all
 * experiments is one launch of the network kernel cps_mppi_step would pick (the tensor-core kernel for plain GRUs of up to
 * 2 x 64 units, its rollouts per CTA chosen from E x K; else the FP32 kernel with the single solve's tile for K), so every
 * experiment runs the arithmetic of one cps_mppi_step.  Launches per period: 2 with supplied draws (solve, plant), 3 with
 * CPS_FLEET_NOISE_PHILOX (the draws of cps_fleet_noise into a fleet-owned [E][n_ind][K] workspace first), whatever E.
 * CPS_NOISE_INDUCING only; default / quadratic_boundary need T + 1 < 512.  cps_fleet_set_states also sets every
 * experiment's hidden state to the handle's stored state (zero after cps_net_load, or what cps_net_set_state set); the
 * handle's own stored state is never written by the fleet.  cps_fleet_step re-checks the loaded network: one whose Htot
 * differs from the fleet's gives CPS_ERR_INVALID (recreate the fleet).  cps_fleet_set_plant_models, cps_fleet_step_noisy,
 * cps_fleet_relabel and cps_fleet_relabel_masked give CPS_ERR_UNSUPPORTED on a neural fleet.
 * cps_fleet_get_net_states / cps_fleet_set_net_states: the hidden states [E][Htot] (Htot = cps_net_state_size);
 * synchronise; CPS_ERR_NOT_CONFIGURED on a fleet without the neural predictor. */
int cps_fleet_get_net_states(cps_handle *h, float *out_host);
int cps_fleet_set_net_states(cps_handle *h, const float *in_host);

/* ---- RPGD fleet: E closed-loop experiments under the reference's default optimizer ------------------------------ */
/* The data generator with controller_mpc and optimizer rpgd (Control_Toolkit_ASF/config_controllers.yml:2): per controller
 * period every experiment runs exactly what optimizer_rpgd_tf.step (Control_Toolkit/Optimizers/optimizer_rpgd_tf.py:231-377)
 * does -- first_iter_count Adam steps on the first solve after a reset, outer_its after that (gradient, clip_by_norm per
 * plan, Adam, clip to the control limits), the costs of the improved plans, their stable order, u = Q[best, 0], the plans
 * shifted by shift_previous (last input repeated) and, on resampling solves (solves % resamp_per == 0, the first one
 * included), the K - opt_keep_k worst plans replaced by clip(normal * sample_stdev + sample_mean) at the inducing points,
 * interpolated with Interpolator's tent weights (the kept plans move to rows K - keep.. in cost order with their shifted
 * moments and ages, the fresh ones start with zero moments and age) -- then the plant advances one controller period with
 * Q = u and writes the record row of cps_fleet_step.  u becomes the experiment's u_prev for the next solve's cost.
 * Each experiment owns its plans [K][T], Adam moments, ages, u_prev, state and targets (target_position /
 * target_equilibrium select the folded cost parameters per experiment and period, as in cps_fleet_step); all advance in
 * lockstep, so the solve counter and Adam's iteration count (lr_t) are shared.
 * The handle: predictor CPS_EULER_CROMER (substeps <= 32) or CPS_PREDICTOR_NEURAL, cost CPS_COST_QB_GRAD_MINIMAL or
 * CPS_COST_QB_GRAD, K <= 4096, T, dt; interp_period = period_interpolation_inducing_points; control limits from
 * cps_set_mppi_params (lo, hi).  Anything else: CPS_ERR_UNSUPPORTED.  opt_keep_k outside [1, K], shift_previous < 0 or dt
 * not a multiple of dt_simulation: CPS_ERR_INVALID.
 * CPS_PREDICTOR_NEURAL: the network is loaded before create (cps_net_load; none: CPS_ERR_NOT_CONFIGURED) and must be one
 * cps_plan_cost_grad accepts (not differential, no CPS_FLAG_NET_TENSOR_CORES, fits shared memory with the adjoint's
 * buffers; else CPS_ERR_UNSUPPORTED).  Create sizes the adjoint's workspace for E experiments; step re-checks the network
 * (it may have been reloaded) and grows the workspace if needed.  Every gradient and cost reads the stored hidden state
 * (cps_net_set_state; zero after load) and never writes it, as optimizer_rpgd_tf's predictor does.  The plant stays the
 * CartPole ODE; the network lives only in the controller.
 * Per period 3 + 4 x (Adam steps) launches with CPS_EULER_CROMER, 3 + 2 x (Adam steps) with CPS_PREDICTOR_NEURAL, whatever E
 * (cps_launch_count).
 * Non-finite costs (e.g. from a NaN state or target) are not an error: they sort after every number, as in torch.sort,
 * and every one the fleet's forward passes meet is added to the handle's counter (cps_nonfinite_costs). */
typedef struct cps_rpgd_fleet_config {
    int struct_size;                 /* = sizeof(cps_rpgd_fleet_config) */
    int n_experiments;               /* E on this device */
    int sim_substeps;                /* plant ticks per controller period */
    int draw_source;                 /* CPS_FLEET_NOISE_SUPPLIED | CPS_FLEET_NOISE_PHILOX: the sampling draws */
    double dt_simulation;            /* plant tick, 0.002 s */
    unsigned long long seed;
    long long experiment_offset;     /* global index of local experiment 0 (Philox counters) */
    int outer_its, first_iter_count, resamp_per, opt_keep_k, shift_previous;
    float learning_rate, adam_beta_1, adam_beta_2, adam_epsilon, gradmax_clip, sample_stdev, sample_mean;
} cps_rpgd_fleet_config;
int cps_rpgd_fleet_create(cps_handle *h, const cps_rpgd_fleet_config *cfg);
/* optimizer_reset for every experiment: plans from the draws init_draws_dev [E][K][n_ind] (NULL on a Philox fleet, which
 * draws them itself), zero moments and ages, solve counter and Adam iterations 0, u_prev = 0; states s_host [E][6]
 * (angle_cos / angle_sin taken as given); the period counter. */
int cps_rpgd_fleet_set_states(cps_handle *h, const float *s_host, const float *init_draws_dev, long long period);
/* n_periods controller periods, stream-ordered, no synchronisation.  tp_dev / te_dev [n_periods][E] or NULL (0 / +1);
 * draws_dev [n_periods][E][K - opt_keep_k][n_ind] standard normals (read only in resampling periods; NULL on a Philox
 * fleet); record_dev [n_periods][E][CPS_FLEET_RECORD], J_out_dev [n_periods][E][K] (costs of the improved plans) and
 * Q_opt_out_dev [n_periods][E][K][T] (plans after the Adam steps, before the bookkeeping: optimizer_rpgd_tf's Q_logged)
 * may each be NULL. */
int cps_rpgd_fleet_step(cps_handle *h, int n_periods, const float *tp_dev, const float *te_dev, const float *draws_dev,
                        float *record_dev, float *J_out_dev, float *Q_opt_out_dev);
/* Offline relabelling under RPGD: add_control_along_trajectories
 * (SI_Toolkit/src/SI_Toolkit/General/preprocess_data_add_control_along_trajectories.py:53-140) with optimizer_rpgd_tf as the
 * controller, E recorded files in lockstep (experiment e of the fleet = file e).  controller.reset() of every file is
 * cps_rpgd_fleet_set_states (the states it takes are overwritten by the first row).  Then one row of all files is one
 * controller period of cps_rpgd_fleet_step with the plant stage replaced: each file's state is its recorded row
 * states_dev [n_rows][E][6], the control goes to Q_out_dev [n_rows][E] and to the file's u_prev, nothing is integrated and
 * no record is written.  The arithmetic per file and row is exactly one optimizer_rpgd_b200.step with the row's attributes
 * tp_dev / te_dev / L_dev / m_pole_dev [n_rows][E] (NULL: 0 / +1 / the handle's L / m_pole).  Between rows a file keeps its
 * plans, Adam moments, ages and u_prev; the solve counter and Adam's iteration count are shared (lockstep).  L / m_pole
 * change the controller's model on CPS_EULER_CROMER (folded on the device per row and file with fold_ode's expressions,
 * so the handle's own values give the handle's constants bit for bit); the neural predictor reads neither, so there they
 * are accepted and change nothing.  draws_dev [n_rows][E][K - opt_keep_k][n_ind] as in cps_rpgd_fleet_step (NULL on a
 * Philox fleet, whose counters use the period counter and experiment_offset: the draws are those cps_rpgd_fleet_draws
 * returns, whatever the split of the files over handles); J_out_dev [n_rows][E][K] or NULL.  Launches per row as per
 * period: 3 + 4 x (Adam steps) with CPS_EULER_CROMER, 3 + 2 x (Adam steps) with CPS_PREDICTOR_NEURAL, whatever E.  After
 * the call the fleet's states are the last row's recorded states. */
int cps_rpgd_fleet_relabel(cps_handle *h, int n_rows, const float *states_dev, const float *tp_dev, const float *te_dev,
                           const float *L_dev, const float *m_pole_dev, const float *draws_dev, float *Q_out_dev,
                           float *J_out_dev);
/* s_host [E][6], u_prev_host [E]; either may be NULL.  Synchronises. */
int cps_rpgd_fleet_get_states(cps_handle *h, float *s_host, float *u_prev_host);
/* Optimizer state: Q_host, m_host, v_host [E][K][T], ages_host [E][K], the shared Adam iteration and solve counters; any
 * may be NULL.  Synchronises. */
int cps_rpgd_fleet_get_plans(cps_handle *h, float *Q_host, float *m_host, float *v_host, int *ages_host,
                             long long *adam_iterations, long long *solves);
long long cps_rpgd_fleet_period(const cps_handle *h);
/* The draws a Philox fleet uses: period >= 0 the resampling draws of that period [E][K - opt_keep_k][n_ind]; period = -1
 * the draws of a reset [E][K][n_ind].  Counters (plan row, tag + draw group, period, experiment_offset + e): disjoint
 * from the MPPI fleet's rollout and plant-side draws. */
int cps_rpgd_fleet_draws(cps_handle *h, long long period, float *out_dev);

/* ---- CEM fleet: E closed-loop experiments under optimizer_cem_tf ------------------------------------------------ */
/* The data generator with controller_mpc and optimizer cem-tf (Control_Toolkit_ASF/config_controllers.yml;
 * Control_Toolkit/Optimizers/optimizer_cem_tf.py:12-117): per controller period every experiment runs exactly what one
 * cps_cem_step does from its own state -- first_iter_count outer iterations on the first period after
 * cps_cem_fleet_set_states (warmup_iterations with warmup, else cem_outer_it), outer_its after that; per iteration
 * Q = clip(mean + eps * stdev) with separately rounded multiply and add (:66-68), the costs of the K plans from the
 * experiment's state with its u_prev and targets (:57-61), the best_k cheapest plans (ties to the lowest index, NaN costs
 * last) and their mean / population stdev per step (:63-83); after the last iteration stdev is clipped to
 * [stdev_min, 1e8], both vectors are shifted by one step (tail: initial_stdev, mid-range mean) and u = elite_Q[0, 0]
 * (:96-99) -- then the plant advances one controller period with Q = u and writes the record row of cps_fleet_step.
 * u becomes the experiment's u_prev for the next period's costs.  Each experiment owns its distribution (mean, stdev
 * [T]), u_prev, state and targets (target_position / target_equilibrium select the folded cost parameters per experiment
 * and period, as in cps_fleet_step); all advance in lockstep, so the solve counter is shared.
 * Draws: standard normals [n_it][E][T][K] per period (K fastest; n_it that period's iteration count), consecutive periods
 * back to back in one cps_cem_fleet_step call (CPS_FLEET_NOISE_SUPPLIED), or generated in the rollout threads
 * (CPS_FLEET_NOISE_PHILOX): counter (plan k, CEM tag + it x ceil(T / 4) + group of four steps, period,
 * experiment_offset + e), key = seed, disjoint from the MPPI and RPGD fleets' streams; cps_cem_fleet_draws materialises
 * them.  Launches per period: n_it x (1, or 2 when best_k x T > 2048: the elite statistics then run as a second kernel
 * with one block per (step, experiment)) + 1 for the plant, whatever E (cps_launch_count).
 * The handle: predictor CPS_EULER_CROMER or CPS_EULER_V0, one of the four cost plugins, K <= 8192 (the single-block
 * selection of cps_cem_step), control limits from cps_set_mppi_params (lo, hi); or CPS_PREDICTOR_NEURAL as under
 * cps_plan_cost.  No cost plugin or the legacy cost, CPS_FLAG_SUBSTEP_SINCOS / CPS_FLAG_FAST_DIV, K > 8192 or a horizon whose buffers do not fit shared
 * memory: CPS_ERR_UNSUPPORTED.  best_k outside [1, K], a negative stdev, outer_its or first_iter_count < 1, dt not a
 * multiple of dt_simulation: CPS_ERR_INVALID.
 * Non-finite costs (e.g. from a NaN state or target) are not an error: they sort after every number, stay in their
 * experiment, and every one is added to the handle's counter (cps_nonfinite_costs). */
typedef struct cps_cem_fleet_config {
    int struct_size;                 /* = sizeof(cps_cem_fleet_config) */
    int n_experiments;               /* E on this device, at most 65535 */
    int sim_substeps;                /* plant ticks per controller period */
    int draw_source;                 /* CPS_FLEET_NOISE_SUPPLIED | CPS_FLEET_NOISE_PHILOX: the sampling draws */
    double dt_simulation;            /* plant tick, 0.002 s */
    unsigned long long seed;
    long long experiment_offset;     /* global index of local experiment 0 (Philox counters) */
    int outer_its, first_iter_count; /* cem_outer_it; the first period's count (warmup_iterations or cem_outer_it) */
    int best_k;                      /* cem_best_k */
    float initial_stdev, stdev_min;  /* cem_initial_action_stdev, cem_stdev_min */
} cps_cem_fleet_config;
int cps_cem_fleet_create(cps_handle *h, const cps_cem_fleet_config *cfg);
/* optimizer_reset for every experiment (mean mid-range, stdev initial_stdev, as cps_cem_reset), u_prev = 0, solve counter
 * 0; states s_host [E][6] (angle_cos / angle_sin taken as given); the period counter.  Synchronises. */
int cps_cem_fleet_set_states(cps_handle *h, const float *s_host, long long period);
/* s_host [E][6], u_prev_host [E]; either may be NULL.  Synchronises. */
int cps_cem_fleet_get_states(cps_handle *h, float *s_host, float *u_prev_host);
/* The sampling distribution of every experiment: mean_host, stdev_host [E][T]; either may be NULL.  Synchronises. */
int cps_cem_fleet_get_distribution(cps_handle *h, float *mean_host, float *stdev_host);
/* n_periods controller periods, stream-ordered, no synchronisation.  tp_dev / te_dev [n_periods][E] or NULL (0 / +1);
 * draws_dev: the periods' draws back to back (see above; NULL on a Philox fleet); record_dev [n_periods][E][CPS_FLEET_RECORD],
 * J_out_dev [n_periods][E][K] and Q_out_dev [n_periods][E][T][K] (costs and plans of each period's last iteration) may each
 * be NULL. */
int cps_cem_fleet_step(cps_handle *h, int n_periods, const float *tp_dev, const float *te_dev, const float *draws_dev,
                       float *record_dev, float *J_out_dev, float *Q_out_dev);
/* The draws a Philox fleet uses in controller period `period`: out_dev [n_it][E][T][K], n_it = first_iter_count for the
 * period set by cps_cem_fleet_set_states, else outer_its. */
int cps_cem_fleet_draws(cps_handle *h, long long period, float *out_dev);
long long cps_cem_fleet_period(const cps_handle *h);

/* ---- CEM-GMM and random-action fleets: E closed-loop experiments under optimizer_cem_gmm_tf / optimizer_random_action_tf */
/* The data generator with controller_mpc and optimizer cem-gmm-tf or random-action-tf (Control_Toolkit_ASF/
 * config_controllers.yml; Control_Toolkit/Optimizers/optimizer_cem_gmm_tf.py:14-140, optimizer_random_action_tf.py:12-86).
 * CEM-GMM: per controller period every experiment runs exactly what one cps_cem_gmm_step with outer_its iterations does
 * from its own state, mixture (loc[2][T], scale[2][T], p1), u_prev, targets and draws -- per iteration component
 * c = 0 iff u01 < p1 and Q = clip(loc[c][t] + scale[c][t] eps_c) with separately rounded multiply and add, the costs, the
 * best_k cheapest plans (ties to the lowest index, NaN costs last), the two clusters around the two cheapest elites
 * (nearer in the Euclidean norm, ties to the cheapest), their per-step mean and population stdev clipped to
 * [stdev_min, 1e4] and p1 = n1 / best_k; after the last iteration u = elite_Q[0, 0] and loc / scale shifted by one step
 * with the last entry repeated.  Random action: every experiment evaluates K plans uniform in [lo, hi) from its state,
 * u_prev and targets and takes u = Q[argmin J, 0] (ties to the lowest index).  Then, for both, the plant advances one
 * controller period with Q = u and writes the record row of cps_fleet_step; u becomes the experiment's u_prev.
 * Targets select the folded cost parameters per experiment and period, as in cps_fleet_step.
 * Draws, supplied (CPS_FLEET_NOISE_SUPPLIED; consecutive periods back to back in one _step call) or generated from
 * Philox4x32-10 (CPS_FLEET_NOISE_PHILOX, key = seed, counters disjoint from the other fleets' streams; _draws materialises
 * them): CEM-GMM standard normals eps [outer_its][E][2][T][K] and uniforms u01 [outer_its][E][T][K] per period, counter
 * (plan k, GMM tag + 3 it ceil(T / 4) + {0, ceil(T / 4)} + group of four steps, period, experiment_offset + e) for the two
 * components' normals and + 2 ceil(T / 4) + group for the uniforms; random action plans [E][T][K] per period, counter
 * (plan k, RA tag + group of four steps, period, experiment_offset + e).  A Philox uniform is (word >> 8) 2^-24 in [0, 1)
 * from one 32-bit word; a random-action plan entry is lo + (hi - lo) u with the multiply and the add rounded separately.
 * Launches per period: 2 outer_its + 1 (CEM-GMM), 2 (random action), whatever E (cps_launch_count).
 * The handle: predictor CPS_EULER_CROMER or CPS_EULER_V0, one of the four cost plugins, K <= 8192, control limits from
 * cps_set_mppi_params (lo, hi); or CPS_PREDICTOR_NEURAL as under cps_plan_cost.  No cost plugin or the legacy cost, CPS_FLAG_SUBSTEP_SINCOS /
 * CPS_FLAG_FAST_DIV, K > 8192 or a horizon whose buffers do not fit shared memory: CPS_ERR_UNSUPPORTED.  CEM-GMM best_k
 * outside [2, K], a negative stdev, outer_its < 1, more than 65535 experiments or dt not a multiple of dt_simulation:
 * CPS_ERR_INVALID.  Non-finite costs sort after every number, stay in their experiment and are counted
 * (cps_nonfinite_costs). */
typedef struct cps_cem_gmm_fleet_config {
    int struct_size;                 /* = sizeof(cps_cem_gmm_fleet_config) */
    int n_experiments;               /* E on this device, at most 65535 */
    int sim_substeps;                /* plant ticks per controller period */
    int draw_source;                 /* CPS_FLEET_NOISE_SUPPLIED | CPS_FLEET_NOISE_PHILOX */
    double dt_simulation;            /* plant tick, 0.002 s */
    unsigned long long seed;
    long long experiment_offset;     /* global index of local experiment 0 (Philox counters) */
    int outer_its;                   /* cem_outer_it */
    int best_k;                      /* cem_best_k */
    float initial_stdev, stdev_min;  /* cem_initial_action_stdev, cem_stdev_min */
} cps_cem_gmm_fleet_config;
int cps_cem_gmm_fleet_create(cps_handle *h, const cps_cem_gmm_fleet_config *cfg);
/* optimizer_reset for every experiment (both components at mid-range with initial_stdev, p1 = 0.5, as cps_cem_gmm_reset),
 * u_prev = 0; states s_host [E][6]; the period counter.  Synchronises. */
int cps_cem_gmm_fleet_set_states(cps_handle *h, const float *s_host, long long period);
/* s_host [E][6], u_prev_host [E]; either may be NULL.  Synchronises. */
int cps_cem_gmm_fleet_get_states(cps_handle *h, float *s_host, float *u_prev_host);
/* Every experiment's mixture: loc_host, scale_host [E][2][T], p1_host [E]; any may be NULL.  Synchronises. */
int cps_cem_gmm_fleet_get_distribution(cps_handle *h, float *loc_host, float *scale_host, float *p1_host);
/* n_periods controller periods, stream-ordered, no synchronisation.  tp_dev / te_dev [n_periods][E] or NULL (0 / +1);
 * eps_dev / u01_dev the periods' draws back to back (NULL on a Philox fleet); record_dev [n_periods][E][CPS_FLEET_RECORD],
 * J_out_dev [n_periods][E][K] and Q_out_dev [n_periods][E][T][K] (costs and plans of each period's last iteration) may
 * each be NULL. */
int cps_cem_gmm_fleet_step(cps_handle *h, int n_periods, const float *tp_dev, const float *te_dev, const float *eps_dev,
                           const float *u01_dev, float *record_dev, float *J_out_dev, float *Q_out_dev);
/* The draws a Philox fleet uses in controller period `period`: eps_out_dev [outer_its][E][2][T][K], u01_out_dev
 * [outer_its][E][T][K]; either may be NULL. */
int cps_cem_gmm_fleet_draws(cps_handle *h, long long period, float *eps_out_dev, float *u01_out_dev);
long long cps_cem_gmm_fleet_period(const cps_handle *h);

typedef struct cps_random_action_fleet_config {
    int struct_size;                 /* = sizeof(cps_random_action_fleet_config) */
    int n_experiments;               /* E on this device, at most 65535 */
    int sim_substeps;                /* plant ticks per controller period */
    int draw_source;                 /* CPS_FLEET_NOISE_SUPPLIED | CPS_FLEET_NOISE_PHILOX */
    double dt_simulation;            /* plant tick, 0.002 s */
    unsigned long long seed;
    long long experiment_offset;     /* global index of local experiment 0 (Philox counters) */
} cps_random_action_fleet_config;
int cps_random_action_fleet_create(cps_handle *h, const cps_random_action_fleet_config *cfg);
/* u_prev = 0; states s_host [E][6]; the period counter.  Synchronises. */
int cps_random_action_fleet_set_states(cps_handle *h, const float *s_host, long long period);
int cps_random_action_fleet_get_states(cps_handle *h, float *s_host, float *u_prev_host);
/* As cps_cem_gmm_fleet_step; plans_dev [n_periods][E][T][K] (NULL on a Philox fleet); Q_out_dev receives the plans. */
int cps_random_action_fleet_step(cps_handle *h, int n_periods, const float *tp_dev, const float *te_dev, const float *plans_dev,
                                 float *record_dev, float *J_out_dev, float *Q_out_dev);
/* The plans a Philox fleet evaluates in controller period `period`: out_dev [E][T][K]. */
int cps_random_action_fleet_draws(cps_handle *h, long long period, float *out_dev);
long long cps_random_action_fleet_period(const cps_handle *h);

/* ---- forward-only planners: predict_and_cost and the selection step (SURVEY 8f row f3) ----------------------- */
/* optimizer_random_action_tf / optimizer_cem_tf / optimizer_cem_gmm_tf evaluate K candidate input plans from one state
 * with predictor.predict_core(s, Q) followed by cost_function.get_trajectory_cost(trajectory, Q, u_prev)
 * (Control_Toolkit/Optimizers/optimizer_random_action_tf.py:42-49, optimizer_cem_tf.py:57-61,
 * optimizer_cem_gmm_tf.py:53-54) and select on the sorted costs.  Here evaluation and selection are one launch; the
 * trajectory tensor is only written when asked for.  ODE predictors and the four cost plugins; plans are clipped by
 * the caller (random action) or in the kernel (CEM) to the control limits of cps_set_mppi_params (lo, hi).
 *
 * cps_plan_cost: J_out_dev[k] = get_trajectory_cost(predict_core(s, Q), Q, u_prev)[k] for K plans of length T
 * (any K, T; Q_dev [K][T] CPS_ROLLOUT_MAJOR or [T][K] CPS_TIME_MAJOR); traj_out_dev as in cps_mppi_step or NULL.
 * cps_plan_cost also takes CPS_PREDICTOR_NEURAL: the plain (not D_*) network loaded with cps_net_load, started from the
 * handle's stored hidden state (read, never written), with quadratic_boundary_grad_minimal or quadratic_boundary_grad, the
 * forward pass of cps_plan_cost_grad (the same J bit for bit; trajectories those of cps_net_rollout on the FP32 kernel).
 * No network loaded: CPS_ERR_NOT_CONFIGURED; differential networks, other cost plugins, CPS_FLAG_NET_TENSOR_CORES or a
 * network whose shared-memory image exceeds 227 KB: CPS_ERR_UNSUPPORTED.
 *
 * The planners below (cps_plan_random_action*, cps_cem_*, cps_cem_gmm_*) and their fleets take CPS_PREDICTOR_NEURAL
 * too, with the network loaded before configure / create.  In the reference their predict_and_cost is predict_core +
 * get_trajectory_cost (optimizer_random_action_tf.py:42-49, optimizer_cem_tf.py:57-61), so, as RPGD: every rollout starts
 * from the stored hidden state (cps_net_set_state; zero after loading), no solve writes it, and fleets keep no hidden
 * state per experiment.  Scope: that of cps_plan_cost on a network (refusals as above, at configure / create and at
 * every solve) and K <= 8192 (the single-block selection; above: CPS_ERR_UNSUPPORTED).  The plans are sampled into
 * memory (CEM clip(mean + eps stdev), CEM-GMM as cps_cem_gmm_step, random action the caller's plans or the fleets'
 * Philox uniforms, from the draws and Philox counters of the ODE path), their costs are those of cps_plan_cost on them bit
 * for bit, and the selection / update runs as a separate one-block kernel (one block per experiment on a fleet), with
 * the ODE path's arithmetic and NaN handling.  Launches: random action 2 per solve; CEM 3 per iteration (4 when
 * best_k x T > 2048); CEM-GMM 3 per iteration, as before.  Fleets per period, whatever E: CEM n_it x (3, or 4) + 1,
 * CEM-GMM 3 outer_its + 1, random action 4.  The host forms copy the state to the device (one extra copy). */
int cps_plan_cost(cps_handle *h, const float *s_dev, const float *Q_dev, int q_layout, int K, int T, float u_prev,
                  float *J_out_dev, float *traj_out_dev, int traj_layout);
/* optimizer_random_action_tf.step (:52-79) for the handle's (K, T): u_out_dev[0] = Q[argmin J, 0], ties to the lowest
 * index.  J_out_dev [K] and best_out_dev [1] (index of the cheapest plan) may be NULL. */
int cps_plan_random_action(cps_handle *h, const float *s_dev, const float *Q_dev, int q_layout, float u_prev,
                           float *u_out_dev, float *J_out_dev, int *best_out_dev);
int cps_plan_random_action_host(cps_handle *h, const float *s_host, const float *Q_dev, int q_layout, float u_prev,
                                float *u_out_host);
/* optimizer_cem_tf (:12-117).  cps_cem_configure: cem_best_k, cem_initial_action_stdev, cem_stdev_min; allocates the
 * sampling distribution (mean, stdev per horizon step) and resets it as optimizer_reset does (:112-116).
 * cps_cem_step: n_iterations outer iterations (cem_outer_it, or warmup_iterations on the first call), one launch each
 * (two when cem_best_k * T > 2048: the elite statistics then run as a second kernel with one block per step; three
 * above 8192 rollouts: the selection then runs as a cooperative kernel with one block per SM):
 * Q = clip(mean + eps * stdev), predict_and_cost, the cem_best_k cheapest plans (ties to the lowest index), mean and
 * population stdev of the elites per step (update_distribution, :63-83); after the last iteration stdev is clipped to
 * [cem_stdev_min, 1e8], both vectors are shifted by one step (tail: initial stdev, mid-range mean) and
 * u_out_dev[0] = elite_Q[0, 0] (:96-99).  eps_dev: standard-normal draws [n_iterations][K][T] (or [n_iterations][T][K]
 * with CPS_TIME_MAJOR); Q_out_dev (same layout, one iteration) receives the LAST iteration's plans, J_out_dev [K] its
 * costs; both may be NULL. */
int cps_cem_configure(cps_handle *h, int best_k, float initial_stdev, float stdev_min);
int cps_cem_reset(cps_handle *h);
int cps_cem_step(cps_handle *h, const float *s_dev, const float *eps_dev, int eps_layout, int n_iterations, float u_prev,
                 float *u_out_dev, float *Q_out_dev, float *J_out_dev);
int cps_cem_step_host(cps_handle *h, const float *s_host, const float *eps_dev, int eps_layout, int n_iterations,
                      float u_prev, float *u_out_host);
/* dist_mue / stdev [T]; either pointer may be NULL.  Synchronise. */
int cps_cem_get_distribution(cps_handle *h, float *mean_host, float *stdev_host);
int cps_cem_set_distribution(cps_handle *h, const float *mean_host, const float *stdev_host);

/* optimizer_cem_gmm_tf (Control_Toolkit/Optimizers/optimizer_cem_gmm_tf.py:58-140): CEM whose sampling distribution is a
 * two-component Gaussian mixture per horizon step.  Per outer iteration (three launches, nothing returns to the host):
 * Q = clip(loc[t, c] + scale[t, c] * eps_c) with the component c of every (rollout, step) chosen independently
 * (c = 0 iff u01 < p1; MixtureSameFamily over the [T, 1] batch, :60-61); predict_and_cost (plan_kernel); the cem_best_k
 * cheapest plans (ties to the lowest index); every elite but the two cheapest joins the nearer of those two in the
 * Euclidean norm over the horizon (:72-77); the clusters' per-step mean and population stdev clipped to
 * [cem_stdev_min, 1e4] become the components, the first cluster's share of the elites its weight p1 (:79-93).  After the
 * last iteration u_out_dev[0] = elite_Q[0, 0] and loc / scale are shifted by one step with the last entry repeated
 * (:108-118).  cps_cem_gmm_reset: both components at mid-range with the initial stdev, p1 = 0.5 (:133-139).
 * Draws: eps_dev standard normals for BOTH components, [n_iterations][K][T][2] (the reference's sample shape) or
 * [n_iterations][2][T][K] with CPS_TIME_MAJOR; u01_dev uniforms in [0, 1), [n_iterations][K][T] or [n_iterations][T][K].
 * Q_out_dev ([K][T] or [T][K]) receives the last iteration's plans, J_out_dev [K] its costs; both may be NULL.
 * Distribution: loc[2][T], scale[2][T] (component-major), p1. */
int cps_cem_gmm_configure(cps_handle *h, int best_k, float initial_stdev, float stdev_min);
int cps_cem_gmm_reset(cps_handle *h);
int cps_cem_gmm_step(cps_handle *h, const float *s_dev, const float *eps_dev, const float *u01_dev, int layout,
                     int n_iterations, float u_prev, float *u_out_dev, float *Q_out_dev, float *J_out_dev);
int cps_cem_gmm_step_host(cps_handle *h, const float *s_host, const float *eps_dev, const float *u01_dev, int layout,
                          int n_iterations, float u_prev, float *u_out_host);
int cps_cem_gmm_get_distribution(cps_handle *h, float *loc_host, float *scale_host, float *p1_host);
int cps_cem_gmm_set_distribution(cps_handle *h, const float *loc_host, const float *scale_host, const float *p1_host);

/* Roofline denominators for the compute-bound rollout kernels, measured on this device with two microbenchmarks
 * (dense FFMA chains; MUFU.EX2 chains): FP32 TFLOP/s (FMA = 2 flops) and MUFU Gop/s.  Synchronises. */
int cps_measure_peaks(cps_handle *h, double *fp32_tflops, double *mufu_gops);

/* Self-test of the rotation kernels' once-per-control-step sin / cos (the math library's small-argument path without its
 * large-argument branch; the reference takes np.sin / np.cos of the wrapped angle, CartPole/cartpole_equations.py:297-299):
 * compares it bit for bit with sincosf and cosf on every float of [-pi, pi]; *mismatches_out = number of differing
 * results (0 expected).  One launch, ~2e9 evaluations; synchronises. */
int cps_selftest_sincos(cps_handle *h, long long *mismatches_out);

/* ---- gradient of predict_and_cost; RPGD ----------------------------------------------------------------- */
/* The reference's gradient-based optimizers take d(traj_cost)/dQ with a tf.GradientTape around predict_and_cost
 * (Control_Toolkit/Optimizers/optimizer_rpgd_tf.py:167-175; RPGD is the shipped default optimizer,
 * Control_Toolkit_ASF/config_controllers.yml:2).  cps_plan_cost_grad is that derivative on the device: forward rollout with a
 * checkpoint per control step, the control steps' transposed Jacobians (hand-derived adjoint of the Euler-Cromer substep) in
 * parallel over (step, plan), reverse sweep over the steps with the cost plugin's partial derivatives (two launches).  Q_dev [K][T] (or [T][K] with CPS_TIME_MAJOR) for the handle's K and T; J_out_dev [K] (or NULL) the costs,
 * G_out_dev the gradient in the layout of Q.  Predictor "ODE" with cos / sin from the angle every substep (the arithmetic
 * the reference differentiates), cost quadratic_boundary_grad_minimal (the shipped RPGD configuration) or
 * quadratic_boundary_grad (u_prev enters its control-change term; its kinetic term's target is under stop_gradient, as in
 * the plugin); anything else: CPS_ERR_UNSUPPORTED.
 * CPS_PREDICTOR_NEURAL (predictor_autoregressive_neural): one launch per gradient, a tile of 16 or 32 plans per CTA runs the
 * FP32 network forward over the horizon and then the reverse sweep through the GRU / Dense layers, the normalised-output
 * feedback, de-normalisation, angle augmentation and the cost plugin (records in a handle-owned workspace that grows on
 * demand, (T+1) x Htot x K floats and a little more).  All plans start from the handle's stored hidden state, which the call
 * reads and never writes (no gradient flows into it or into s); the same two cost plugins.  No network loaded:
 * CPS_ERR_NOT_CONFIGURED; differential (D_*) networks, CPS_FLAG_NET_TENSOR_CORES (that flag forces a kernel without a
 * gradient) or a network whose shared-memory image with the adjoint's buffers exceeds 227 KB: CPS_ERR_UNSUPPORTED.
 * cps_rpgd_grad_step is grad_step (:166-180) on the device (either predictor, as cps_plan_cost_grad; with the neural one the
 * stored hidden state is left as it is): the gradient, tf.clip_by_norm over each plan (gradmax_clip), one
 * Adam step (Keras legacy Adam: lr_t = lr sqrt(1 - b2^t) / (1 - b1^t), m, v per element, handle-owned, t = iterations since
 * cps_rpgd_reset) and the clip to the control limits, in place on Q_dev [K][T].  cps_rpgd_adam_state exposes the device
 * buffers of m and v ([K][T]) and the iteration count for the warm-start bookkeeping of step() (:297-356). */
int cps_plan_cost_grad(cps_handle *h, const float *s_dev, const float *Q_dev, int q_layout, float u_prev, float *J_out_dev,
                       float *G_out_dev);
int cps_rpgd_reset(cps_handle *h);
int cps_rpgd_grad_step(cps_handle *h, const float *s_dev, float *Q_dev, float u_prev, float learning_rate, float beta_1,
                       float beta_2, float epsilon, float gradmax_clip, float *J_out_dev);
int cps_rpgd_adam_state(cps_handle *h, float **m_dev, float **v_dev, long long *iterations);
int cps_rpgd_set_iterations(cps_handle *h, long long iterations);
/* get_action and the per-solve bookkeeping of optimizer_rpgd_tf.step (:182-224, :297-356) on the device: the stable order of
 * the K costs J_dev, u_nom = the cheapest plan (copied to u_nom_host [T]; synchronises), every plan shifted by
 * shift_previous (last input repeated), the Adam moments shifted by one step, ages_dev [K] (int32, or NULL) + 1.  With
 * fresh_dev != NULL ([K - keep][T], a resampling solve) the `keep` cheapest plans move to the rows K - keep.. in cost order
 * with their moments and ages, rows 0..K - keep - 1 take the fresh plans with zero moments and age.  In place on Q_dev
 * [K][T]; K <= 4096 (ranks by counting), else CPS_ERR_UNSUPPORTED and the caller does it with tensor operations. */
int cps_rpgd_finish(cps_handle *h, const float *J_dev, float *Q_dev, const float *fresh_dev, int keep, int shift_previous,
                    int *ages_dev, float *u_nom_host);

/* ---- diagnostics ------------------------------------------------------------------------------------- */
/* Number of kernels this handle has launched so far (bench.py's gpu_launches claim). */
long long cps_launch_count(const cps_handle *h);
/* Which network kernel the last cps_net_rollout / neural cps_mppi_step of this handle launched: 0 none yet, 1 the FP32
 * CUDA-core kernel (net_kernel), 2 the tensor-core kernel (net_tc_kernel; the default for plain 2 x 64 GRU networks).
 * The reference has no counterpart (its predictor is one torch module, SI_Toolkit/Predictors/predictor_autoregressive_neural.py:266-313). */
int cps_net_last_kernel(const cps_handle *h);
/* Which kernel the last cps_rollout / cps_rollout_host chunk of this handle launched: 0 none yet, 1 rollout_kernel (one
 * cartpole per thread), 2 rollout_pair_kernel (two per thread, packed FP32; large time-major batches). */
int cps_rollout_last_kernel(const cps_handle *h);
/* Cumulative count of non-finite trajectory costs seen by cps_mppi_step, cps_plan_cost_grad / cps_rpgd_grad_step,
 * cps_rpgd_fleet_step and cps_cem_fleet_step since cps_create (the reference propagates NaN silently; this library does the same arithmetic but
 * counts it).  Synchronises. */
int cps_nonfinite_costs(cps_handle *h, int *count_out);

#ifdef __cplusplus
}
#endif
#endif /* CPS_H_ */
