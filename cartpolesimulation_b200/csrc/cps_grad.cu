// cps_grad.cu -- the gradient of predict_and_cost with respect to the input plans, and the RPGD update built on it.
//
// The reference's gradient-based optimizers (RPGD is its shipped default, Control_Toolkit_ASF/config_controllers.yml:2;
// Control_Toolkit/Optimizers/optimizer_rpgd_tf.py:167-180) wrap
//     rollout_trajectory = predictor.predict_core(s, Q);  traj_cost = cost_function.get_trajectory_cost(traj, Q, u)
// in a tf.GradientTape and take d(traj_cost)/dQ [K][T]: reverse-mode differentiation through T x n Euler-Cromer substeps
// (SI_Toolkit/Predictors/predictor_ODE.py, CartPole/cartpole_equations.py:71-99, 245-262) and the cost plugin, with the
// [K][T+1][6] trajectory and the tape in between.  Here it is three launches, and only the first and the cheap last one are
// sequential in time:
//   forward   (thread per plan) integrates it (cos / sin from the angle every substep, as the reference's graph does),
//             accumulates the cost and leaves a checkpoint (angle, angleD, position, positionD) per control step in a
//             [T][4][K] workspace (coalesced: consecutive plans are consecutive addresses);
//   jacobians (thread per (control step, plan), T times the parallelism): re-integrates the n substeps of the step from its
//             checkpoint and sweeps the four unit adjoints backwards through them with the hand-derived adjoint of the
//             substep (oracle/oracle.py:plan_cost_grad is the same derivation in numpy, checked against torch autograd
//             through the unmodified reference modules, tests/golden/grad_*.npz): the step's transposed Jacobian;
//   reverse   (thread per plan) walks the control steps backwards: one 4 x 4 matrix-vector product per step plus the cost
//             plugin's partial derivatives at the control-step boundaries.
// (The first version did all of it in one thread per plan: 3 T n sequential substep evaluations, 0.124 ms for 16 plans.)
// rpgd_update_kernel is the rest of grad_step (:176-180): tf.clip_by_norm per plan, the Adam step (Keras legacy Adam =
// ResourceApplyAdam) and the clip to the control limits.
// Cost plugins: quadratic_boundary_grad_minimal (the plugin the shipped RPGD configuration uses) and quadratic_boundary_grad;
// predictor "ODE" here, the neural predictor in cps_net_grad.cu (cps_plan_cost_grad hands it over; the RPGD update and
// bookkeeping below serve both).
#include <cuda_runtime.h>

#include <cmath>
#include <cstring>
#include <new>

#include "cps_grad_partials.cuh"
#include "cps_internal.cuh"

#define CPS_GRAD_MAX_SUBSTEPS 32

struct GradState {
    float *d_ck;        // [T][4][K] checkpoints
    float *d_jac;       // [T][CPS_GRAD_REC][K] transposed Jacobians of the control steps + boundary terms
    float *d_J;         // [K]
    float *d_G;         // [K][T]
    float *d_m, *d_v;   // Adam moments [K][T]
    float *d_Q2, *d_m2, *d_v2, *d_unom;   // cps_rpgd_finish: permuted copies [K][T], the cheapest plan [T]
    int *d_ages2;
    float *h_unom;      // pinned [T]
    long long adam_iterations;
};

struct GradArgs {
    OdeParams ode;
    CostParams cost;
    const float *s;
    const float *Q;
    long long qs_k, qs_t;
    int K, T;
    int full;        // cost plugin: 0 quadratic_boundary_grad_minimal, 1 quadratic_boundary_grad
    float u_prev;    // the input applied before the plan (quadratic_boundary_grad's control-change term)
    float inv_T1;
    float *ck, *jac, *J, *G;
    long long gs_k, gs_t;
    int *nonfinite;
};

// The fleet variants' per-experiment inputs (cps_rpgd_fleet.cu): plan k belongs to experiment k / kpe.
struct FleetGradExt {
    const CostParams *costs;   // [E] folded for each experiment's targets of the period
    const float *u_prev;       // [E]
    int kpe;                   // plans per experiment
};
struct FleetGradArgs {
    GradArgs g;                // K = E * kpe plans [E * kpe][T]; s = the fleet's states [E][8]
    FleetGradExt x;
};
// The same with the controller's model per experiment (cps_rpgd_fleet_relabel with per-row L / m_pole): experiment e
// integrates with odes[e] instead of g.ode.
struct FleetGradOdeArgs {
    GradArgs g;
    FleetGradExt x;
    const OdeParams *odes;     // [E]
};

namespace {

struct Sub { float th, w, v, sn, c; };

// One Euler-Cromer substep of predictor_ODE with cos / sin taken from the angle (cartpole_equations.py:71-99, 245-262).
// Returns the substep's inputs (angle, angleD, positionD, sin, cos) for the reverse sweep.
__device__ __forceinline__ Sub grad_substep(const OdeParams &P, float &th, float &w, float &x, float &v, float uk) {
    Sub in;
    in.th = th; in.w = w; in.v = v;
    sincos_th(th, in.sn, in.c);
    const float sn = in.sn, c = in.c;
    const float rA = rcp_pos<false>(fmaf(-P.m_p, c * c, P.KM));
    const float t1 = fmaf(-P.c2, w * w, P.c1 * c);
    const float num = fmaf(sn, t1, fmaf(-(P.c3 * w), c, fmaf(-P.c5, v, uk)));
    const float xDD = num * rA;
    const float thDD = fmaf(P.d1, sn, fmaf(P.d2 * xDD, c, -P.d3 * w));
    w = fmaf(thDD, P.h, w);
    v = fmaf(xDD, P.h, v);
    th = fold_angle(fmaf(w, P.h, th));
    x = fmaf(v, P.h, x);
    return in;
}

// ---- forward: one thread per plan; cost and a checkpoint per control step ---------------------------------------------------
// The integration and the cost are plan_kernel's (control_step with the rotation substeps, stage_cost): J is bit-identical
// to cps_plan_cost's, and the sequential part of the gradient runs at the solve kernels' speed.
// FLEET (cps_rpgd_fleet.cu): the plans of E experiments in one launch, plan k of experiment k / fx.kpe with that experiment's
// state, u_prev and cost parameters (fx); a null a.ck skips the checkpoints (costs only).  Per plan the arithmetic is the same.
// ODE_E (FLEET only): the model constants of experiment e from odes[e] rather than a.ode.
template <int NSUB, bool FLEET, bool ODE_E = false>
__device__ __forceinline__ void grad_fwd(const GradArgs &a, const FleetGradExt &fx, const OdeParams *odes = nullptr) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= a.K) return;
    const int e = FLEET ? k / fx.kpe : 0;
    const CostParams &C = FLEET ? fx.costs[e] : a.cost;
    const int T = a.T, K = a.K;
    const bool want_ck = !FLEET || a.ck != nullptr;
    State z = load_state(FLEET ? a.s + (long long)e * 8 : a.s);
    const OdeParams ode = pin_params(ODE_E ? odes[e] : a.ode, z.th);
    float c_cost = cosf(z.th);
    const float *q = a.Q + (long long)k * a.qs_k;
    float *ck = want_ck ? a.ck + k : nullptr;   // costs only (fleet): no checkpoint buffer
    float Jacc = 0.0f, up = FLEET ? fx.u_prev[e] : a.u_prev;
    float qn = q[0];
#pragma unroll 1
    for (int t = 0; t < T; ++t) {
        const float u = qn;
        if (t + 1 < T) qn = q[(long long)(t + 1) * a.qs_t];   // prefetch under the integration
        if (want_ck) {
            ck[((long long)t * 4 + 0) * K] = z.th; ck[((long long)t * 4 + 1) * K] = z.w;
            ck[((long long)t * 4 + 2) * K] = z.x;  ck[((long long)t * 4 + 3) * K] = z.v;
        }
        Jacc += a.full ? stage_cost<COST_GRAD>(C, c_cost, z.w, z.x, u, up) : stage_cost<COST_GRADMIN>(C, c_cost, z.w, z.x, u, 0.0f);
        control_step<1, SC_ROTATE, false, false, false, NSUB>(ode, z, u);
        c_cost = z.c;
        up = u;
    }
    const float J = __fdiv_rn(Jacc, (float)(T + 1));   // the plugin's terminal cost is zero
    if (a.J) a.J[k] = J;
    if (!isfinite(J)) atomicAdd(a.nonfinite, 1);
}
template <int NSUB>
__global__ void __launch_bounds__(128) plan_grad_fwd_kernel(const __grid_constant__ GradArgs a) {
    grad_fwd<NSUB, false>(a, FleetGradExt());
}
template <int NSUB>
__global__ void __launch_bounds__(128) fleet_grad_fwd_kernel(const __grid_constant__ FleetGradArgs f) {
    grad_fwd<NSUB, true>(f.g, f.x);
}
template <int NSUB>
__global__ void __launch_bounds__(128) fleet_grad_fwd_ode_kernel(const __grid_constant__ FleetGradOdeArgs f) {
    grad_fwd<NSUB, true, true>(f.g, f.x, f.odes);
}

// ---- transposed Jacobian of every control step, in parallel over (control step, plan) ------------------------------------
// The reverse sweep is linear in the adjoint (a_th, a_w, a_x, a_v), so a control step acts on it as a 4 x 4 matrix that
// depends only on the step's forward states: thread (t, k) re-integrates the n substeps of step t from its checkpoint and
// pushes the four unit adjoints back through them together (the coefficients of a substep are computed once for the four).
// Output per (t, k): M[3][4] -- rows (a_th, a_w, a_v) at the start of the step as combinations of the adjoint at its end
// (a_x passes through unchanged: the position enters no right-hand side) --, r[4], the row that gives d/d(uk), and the
// terms the cost adds at the step's boundary.
// Sequential work per plan shrinks from T x n reverse substeps to T small matrix-vector products (plan_grad_rev_kernel).
template <int NSUB, bool FLEET = false, bool ODE_E = false>
__device__ __forceinline__ void step_record(const GradArgs &a, int t, int k, float *o, long long stride,
                                            const FleetGradExt &fx = FleetGradExt(), const OdeParams *odes = nullptr) {
    const int K = a.K;
    const int e = FLEET ? k / fx.kpe : 0;
    const CostParams &C = FLEET ? fx.costs[e] : a.cost;
    const OdeParams &P = ODE_E ? odes[e] : a.ode;
    const int n = NSUB ? NSUB : P.n;
    const float *ck = a.ck + k;
    float th = ck[((long long)t * 4 + 0) * K], w = ck[((long long)t * 4 + 1) * K];
    float x = ck[((long long)t * 4 + 2) * K], v = ck[((long long)t * 4 + 3) * K];
    const float th0 = th, w0 = w, x0 = x;
    const float u = a.Q[(long long)k * a.qs_k + (long long)t * a.qs_t];
    const float uk = P.u_scale * u;
    Sub sub[NSUB ? NSUB : CPS_GRAD_MAX_SUBSTEPS];
#pragma unroll
    for (int i = 0; i < (NSUB ? NSUB : CPS_GRAD_MAX_SUBSTEPS); ++i)
        if (i < n) sub[i] = grad_substep(P, th, w, x, v, uk);
    // seed j = unit adjoint in component j (th, w, x, v) at the end of the step
    float A_th[4] = {1.0f, 0.0f, 0.0f, 0.0f}, A_w[4] = {0.0f, 1.0f, 0.0f, 0.0f}, A_v[4] = {0.0f, 0.0f, 0.0f, 1.0f};
    float A_uk[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
    for (int ii = 0; ii < (NSUB ? NSUB : CPS_GRAD_MAX_SUBSTEPS); ++ii) {
        const int i = n - 1 - ii;
        if (i < 0) continue;
        const float wi = sub[i].w, vi = sub[i].v, sn = sub[i].sn, c = sub[i].c;
        const float rA = rcp_pos<false>(fmaf(-P.m_p, c * c, P.KM));
        const float t1 = fmaf(-P.c2, wi * wi, P.c1 * c), t4 = P.c3 * wi;
        const float num = fmaf(sn, t1, fmaf(-t4, c, fmaf(-P.c5, vi, uk)));
        const float xDD = num * rA;
        const float d2c = P.d2 * c, d2x = P.d2 * xDD, krA = 2.0f * P.m_p * c * rA * rA, kw = -2.0f * P.c2 * wi;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float a_x = (j == 2) ? 1.0f : 0.0f;
            const float a_v2 = fmaf(P.h, a_x, A_v[j]);             // x' = x + h v'
            const float a_w2 = fmaf(P.h, A_th[j], A_w[j]);         // th' = th + h w'
            const float a_thDD = P.h * a_w2;                       // w' = w + h thDD
            const float a_xDD = fmaf(d2c, a_thDD, P.h * a_v2);     // v' = v + h xDD; thDD = d1 s + d2 xDD c - d3 w
            float a_s = P.d1 * a_thDD;
            float a_c = d2x * a_thDD;
            float a_win = fmaf(-P.d3, a_thDD, a_w2);
            const float a_num = rA * a_xDD, a_rA = num * a_xDD;    // xDD = num rA
            a_c = fmaf(krA, a_rA, a_c);                            // rA = 1 / (KM - m_p c^2)
            a_s = fmaf(t1, a_num, a_s);                            // num = s t1 - t4 c + (uk - c5 v)
            const float a_t1 = sn * a_num, a_t4 = -c * a_num;
            a_c = fmaf(-t4, a_num, a_c);
            a_c = fmaf(P.c1, a_t1, a_c);                           // t1 = c1 c - c2 w^2
            a_win = fmaf(kw, a_t1, fmaf(P.c3, a_t4, a_win));
            A_uk[j] += a_num;
            A_v[j] = fmaf(-P.c5, a_num, a_v2);
            A_th[j] = fmaf(c, a_s, fmaf(-sn, a_c, A_th[j]));       // c = cos th, s = sin th
            A_w[j] = a_win;
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        o[(0 + j) * stride] = A_th[j];
        o[(4 + j) * stride] = A_w[j];
        o[(8 + j) * stride] = A_v[j];
        o[(12 + j) * stride] = A_uk[j];
    }
    // what the reverse sweep adds at this control-step boundary: the cost plugin's partial derivatives at the step's first
    // state and its control term, with the 1 / (T + 1) of the mean
    float d_th, d_w, d_x, d_u;
    if (a.full) {
        grad_partials(C, th0, w0, x0, d_th, d_w, d_x);
        // cc u_t^2 + ccrc (u_t - u_{t-1})^2 of this stage and ccrc (u_{t+1} - u_t)^2 of the next (_control_change_rate_cost, :174-180)
        const float *q = a.Q + (long long)k * a.qs_k;
        const float up = (t > 0) ? q[(long long)(t - 1) * a.qs_t] : (FLEET ? fx.u_prev[e] : a.u_prev);
        d_u = 2.0f * C.w[5] * u + 2.0f * C.w[6] * (u - up);
        if (t + 1 < a.T) d_u -= 2.0f * C.w[6] * (q[(long long)(t + 1) * a.qs_t] - u);
    } else {
        gradmin_partials(C, th0, w0, x0, d_th, d_w, d_x);
        d_u = 2.0f * C.w[4] * u;
    }
    o[16 * stride] = a.inv_T1 * d_th;
    o[17 * stride] = a.inv_T1 * d_w;
    o[18 * stride] = a.inv_T1 * d_x;
    o[19 * stride] = a.inv_T1 * d_u;
}

// records to global memory (horizons too long for the fused kernel below)
template <int NSUB>
__global__ void __launch_bounds__(128) plan_grad_jac_kernel(const __grid_constant__ GradArgs a) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int K = a.K;
    if (gid >= (long long)K * a.T) return;
    const int k = (int)(gid % K), t = (int)(gid / K);
    step_record<NSUB>(a, t, k, a.jac + (long long)t * CPS_GRAD_REC * K + k, K);
}
// (six blocks per SM as plan_grad_jac_kernel<10>: the per-experiment cost parameters would otherwise lift it to 96 registers)
template <int NSUB>
__global__ void __launch_bounds__(128, 6) fleet_grad_jac_kernel(const __grid_constant__ FleetGradArgs f) {
    const GradArgs &a = f.g;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int K = a.K;
    if (gid >= (long long)K * a.T) return;
    const int k = (int)(gid % K), t = (int)(gid / K);
    step_record<NSUB, true>(a, t, k, a.jac + (long long)t * CPS_GRAD_REC * K + k, K, f.x);
}
// the same with experiment e's model constants read from f.odes[e]: they occupy registers, where the kernel above reads
// them from the parameter bank.  Five blocks per SM (96 registers): at six (80) the NSUB = 10 variant spills 76 bytes.
template <int NSUB>
__global__ void __launch_bounds__(128, 5) fleet_grad_jac_ode_kernel(const __grid_constant__ FleetGradOdeArgs f) {
    const GradArgs &a = f.g;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int K = a.K;
    if (gid >= (long long)K * a.T) return;
    const int k = (int)(gid % K), t = (int)(gid / K);
    step_record<NSUB, true, true>(a, t, k, a.jac + (long long)t * CPS_GRAD_REC * K + k, K, f.x, f.odes);
}

// One control step of the reverse sweep from its record r.
__device__ __forceinline__ void load_record(const float *m, long long stride, float (&r)[CPS_GRAD_REC]) {
#pragma unroll
    for (int j = 0; j < CPS_GRAD_REC; ++j) r[j] = m[j * stride];
}
__device__ __forceinline__ void apply_record(const float (&r)[CPS_GRAD_REC], float us, float &a_th, float &a_w, float &a_x, float &a_v,
                                             float &g_out) {
    const float a_uk = fmaf(r[12], a_th, fmaf(r[13], a_w, fmaf(r[14], a_x, r[15] * a_v)));
    const float n_th = fmaf(r[0], a_th, fmaf(r[1], a_w, fmaf(r[2], a_x, r[3] * a_v)));
    const float n_w = fmaf(r[4], a_th, fmaf(r[5], a_w, fmaf(r[6], a_x, r[7] * a_v)));
    const float n_v = fmaf(r[8], a_th, fmaf(r[9], a_w, fmaf(r[10], a_x, r[11] * a_v)));
    g_out = fmaf(us, a_uk, r[19]);
    a_th = n_th + r[16];
    a_w = n_w + r[17];
    a_x = a_x + r[18];
    a_v = n_v;
}
__device__ __forceinline__ void reverse_step(const float *m, long long stride, float us, float &a_th, float &a_w, float &a_x,
                                             float &a_v, float &g_out) {
    float r[CPS_GRAD_REC];
    load_record(m, stride, r);
    apply_record(r, us, a_th, a_w, a_x, a_v, g_out);
}

// Fused: a block takes P plans, thread (t, plan) leaves its record in shared memory ([T][CPS_GRAD_REC][P]), then the first P
// threads walk the control steps backwards from there -- no round trip through global memory under the sequential part.
template <int NSUB>
__global__ void __launch_bounds__(512) plan_grad_jacrev_kernel(const __grid_constant__ GradArgs a, int P) {
    extern __shared__ float s_rec[];
    const int tid = threadIdx.x, kk = tid % P, t = tid / P;
    const int k = blockIdx.x * P + kk;
    if (t < a.T && k < a.K) step_record<NSUB>(a, t, k, s_rec + (long long)t * CPS_GRAD_REC * P + kk, P);
    __syncthreads();
    if (tid < P && k < a.K) {
        float *g = a.G + (long long)k * a.gs_k;
        float a_th = 0.0f, a_w = 0.0f, a_x = 0.0f, a_v = 0.0f;
#pragma unroll 2
        for (int tt = a.T - 1; tt >= 0; --tt) {
            float go;
            reverse_step(s_rec + (long long)tt * CPS_GRAD_REC * P + kk, P, a.ode.u_scale, a_th, a_w, a_x, a_v, go);
            g[(long long)tt * a.gs_t] = go;
        }
    }
}

// ---- reverse from global records (horizons too long for the fused kernel): one thread per plan -----------------------------
__global__ void __launch_bounds__(128) plan_grad_rev_kernel(const __grid_constant__ GradArgs a) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= a.K) return;
    const int T = a.T, K = a.K;
    float *g = a.G + (long long)k * a.gs_k;
    float a_th = 0.0f, a_w = 0.0f, a_x = 0.0f, a_v = 0.0f;
    // the records do not depend on the adjoint: the next one is read while this one is applied
    float r[CPS_GRAD_REC], rn[CPS_GRAD_REC];
    load_record(a.jac + (long long)(T - 1) * CPS_GRAD_REC * K + k, K, r);
#pragma unroll 1
    for (int t = T - 1; t >= 0; --t) {
        if (t > 0) load_record(a.jac + (long long)(t - 1) * CPS_GRAD_REC * K + k, K, rn);
        float go;
        apply_record(r, a.ode.u_scale, a_th, a_w, a_x, a_v, go);
        g[(long long)t * a.gs_t] = go;
#pragma unroll
        for (int j = 0; j < CPS_GRAD_REC; ++j) r[j] = rn[j];
    }
}

// grad_step after the tape (optimizer_rpgd_tf.py:176-180): clip_by_norm over the plan, Adam, clip to the limits.
// One warp per plan.
struct RpgdArgs {
    float *Q; const float *G; float *m, *v;
    int K, T;
    float clip_norm, lr_t, beta1, beta2, eps, lo, hi;
};
__global__ void __launch_bounds__(128) rpgd_update_kernel(const __grid_constant__ RpgdArgs a) {
    const int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (k >= a.K) return;
    const float *g = a.G + (long long)k * a.T;
    float ss = 0.0f;
    for (int t = lane; t < a.T; t += 32) ss = fmaf(g[t], g[t], ss);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    const float l2 = sqrtf(ss);
    const float scale = a.clip_norm / fmaxf(l2, a.clip_norm);   // tf.clip_by_norm: t * clip_norm / max(l2norm, clip_norm)
    for (int t = lane; t < a.T; t += 32) {
        const long long i = (long long)k * a.T + t;
        const float gi = g[t] * scale;
        const float m = fmaf(a.beta1, a.m[i], (1.0f - a.beta1) * gi);
        const float v = fmaf(a.beta2, a.v[i], (1.0f - a.beta2) * gi * gi);
        a.m[i] = m; a.v[i] = v;
        const float qn = a.Q[i] - a.lr_t * m / (sqrtf(v) + a.eps);
        a.Q[i] = fminf(fmaxf(qn, a.lo), a.hi);
    }
}

// get_action + the bookkeeping of step(): one block per plan.
struct FinishArgs {
    const float *J, *Q, *m, *v, *fresh;
    const int *ages;
    float *Q2, *m2, *v2, *u_nom;
    int *ages2;
    int K, T, keep, sp;
};
__global__ void __launch_bounds__(64) rpgd_finish_kernel(const __grid_constant__ FinishArgs a) {
    __shared__ int s_cnt[2];
    const int i = blockIdx.x, tid = threadIdx.x, K = a.K, T = a.T;
    const float Ji = a.J[i];
    int cnt = 0;   // plans in front of plan i in the stable ascending order (torch.sort(J, stable=True), :186)
    for (int j = tid; j < K; j += 64) {
        const float Jj = a.J[j];
        cnt += (Jj < Ji || (Jj == Ji && j < i)) ? 1 : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((tid & 31) == 0) s_cnt[tid >> 5] = cnt;
    __syncthreads();
    const int rank = s_cnt[0] + s_cnt[1];
    const bool resample = a.fresh != nullptr;
    const int dest = resample ? (rank < a.keep ? (K - a.keep) + rank : -1) : i;
    const float *q = a.Q + (long long)i * T, *m = a.m + (long long)i * T, *v = a.v + (long long)i * T;
    if (rank == 0)
        for (int t = tid; t < T; t += 64) a.u_nom[t] = q[t];
    if (dest >= 0) {
        for (int t = tid; t < T; t += 64) {
            const long long o = (long long)dest * T + t;
            a.Q2[o] = q[min(t + a.sp, T - 1)];
            a.m2[o] = (t + 1 < T) ? m[t + 1] : 0.0f;
            a.v2[o] = (t + 1 < T) ? v[t + 1] : 0.0f;
        }
        if (a.ages && tid == 0) a.ages2[dest] = a.ages[i] + 1;
    }
    if (resample && i < K - a.keep) {
        for (int t = tid; t < T; t += 64) {
            const long long o = (long long)i * T + t;
            a.Q2[o] = a.fresh[o];
            a.m2[o] = 0.0f;
            a.v2[o] = 0.0f;
        }
        if (a.ages && tid == 0) a.ages2[i] = 1;
    }
}
__global__ void __launch_bounds__(256) rpgd_copyback_kernel(float *Q, float *m, float *v, int *ages, const float *Q2, const float *m2,
                                                            const float *v2, const int *ages2, int K, int T) {
    const int n = K * T;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        Q[i] = Q2[i]; m[i] = m2[i]; v[i] = v2[i];
        if (ages && i < K) ages[i] = ages2[i];
    }
}

}  // namespace

void cps_grad_free(cps_handle *h) {
    GradState *G = h->grad;
    if (!G) return;
    cudaFree(G->d_ck); cudaFree(G->d_jac); cudaFree(G->d_J); cudaFree(G->d_G); cudaFree(G->d_m); cudaFree(G->d_v);
    cudaFree(G->d_Q2); cudaFree(G->d_m2); cudaFree(G->d_v2); cudaFree(G->d_unom); cudaFree(G->d_ages2);
    if (G->h_unom) cudaFreeHost(G->h_unom);
    delete G;
    h->grad = nullptr;
}

static int grad_state(cps_handle *h, GradState **out) {
    if (h->grad) { *out = h->grad; return CPS_OK; }
    const bool neural = h->cfg.integrator == CPS_PREDICTOR_NEURAL;
    if (h->cfg.integrator != CPS_EULER_CROMER && !neural)
        return fail(h, CPS_ERR_UNSUPPORTED, "cps_plan_cost_grad: the adjoint is built for predictor \"ODE\" (Euler-Cromer) and the "
                    "neural predictor");
    if (h->cfg.cost_id != CPS_COST_QB_GRAD_MINIMAL && h->cfg.cost_id != CPS_COST_QB_GRAD)
        return fail(h, CPS_ERR_UNSUPPORTED, "cps_plan_cost_grad: the adjoint is built for the quadratic_boundary_grad_minimal and quadratic_boundary_grad plugins");
    if (!neural && h->cfg.substeps > CPS_GRAD_MAX_SUBSTEPS)
        return fail(h, CPS_ERR_UNSUPPORTED, "cps_plan_cost_grad: at most 32 substeps per control step");
    GradState *G = new (std::nothrow) GradState();
    if (!G) return fail(h, CPS_ERR_INVALID, "cps_plan_cost_grad: out of host memory");
    memset(G, 0, sizeof(*G));
    const size_t K = h->cfg.num_rollouts, T = h->cfg.horizon;
    cudaError_t e = cudaSuccess;
    if (!neural) {   // the neural adjoint keeps its records in the network's workspace (cps_net_grad.cu)
        e = cudaMalloc(&G->d_ck, sizeof(float) * 4 * K * T);
        if (e == cudaSuccess) e = cudaMalloc(&G->d_jac, sizeof(float) * CPS_GRAD_REC * K * T);
    }
    if (e == cudaSuccess) e = cudaMalloc(&G->d_J, sizeof(float) * K);
    if (e == cudaSuccess) e = cudaMalloc(&G->d_G, sizeof(float) * K * T);
    if (e == cudaSuccess) e = cudaMalloc(&G->d_m, sizeof(float) * K * T);
    if (e == cudaSuccess) e = cudaMalloc(&G->d_v, sizeof(float) * K * T);
    if (e == cudaSuccess) e = cudaMemset(G->d_m, 0, sizeof(float) * K * T);
    if (e == cudaSuccess) e = cudaMemset(G->d_v, 0, sizeof(float) * K * T);
    if (e != cudaSuccess) {
        cudaFree(G->d_ck); cudaFree(G->d_jac); cudaFree(G->d_J); cudaFree(G->d_G); cudaFree(G->d_m); cudaFree(G->d_v);
        delete G;
        return fail(h, CPS_ERR_CUDA, "cps_plan_cost_grad: allocating the workspace: %s", cudaGetErrorString(e));
    }
    h->grad = G;
    *out = G;
    return CPS_OK;
}

extern "C" int cps_plan_cost_grad(cps_handle *h, const float *s_dev, const float *Q_dev, int q_layout, float u_prev,
                                  float *J_out_dev, float *G_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    if (!s_dev || !Q_dev || !G_out_dev) return fail(h, CPS_ERR_INVALID, "cps_plan_cost_grad: null pointer");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    GradState *G;
    int rc = grad_state(h, &G);
    if (rc != CPS_OK) return rc;
    const int K = h->cfg.num_rollouts, T = h->cfg.horizon;
    if (h->cfg.integrator == CPS_PREDICTOR_NEURAL)
        return cps_net_plan_cost_grad(h, s_dev, Q_dev, q_layout, u_prev, J_out_dev ? J_out_dev : G->d_J, G_out_dev);
    GradArgs a;
    memset(&a, 0, sizeof(a));
    a.ode = h->ode; a.cost = h->cost;
    a.s = s_dev;
    a.Q = Q_dev;
    if (q_layout == CPS_TIME_MAJOR) { a.qs_k = 1; a.qs_t = K; a.gs_k = 1; a.gs_t = K; }
    else { a.qs_k = T; a.qs_t = 1; a.gs_k = T; a.gs_t = 1; }
    a.K = K; a.T = T;
    a.full = h->cfg.cost_id == CPS_COST_QB_GRAD ? 1 : 0;
    a.u_prev = u_prev;   // enters quadratic_boundary_grad's control-change term only
    a.inv_T1 = 1.0f / (float)(T + 1);
    a.ck = G->d_ck; a.jac = G->d_jac; a.J = J_out_dev ? J_out_dev : G->d_J; a.G = G_out_dev;
    a.nonfinite = h->d_nonfinite;
    const int block = (K <= 148 * 32) ? 32 : 128;   // small K: one warp per block spreads the plans over the SMs
    const int grid = (K + block - 1) / block;
    const long long pairs = (long long)K * T;
    const int jblock = (pairs <= 148 * 32 * 4) ? 32 : 128;
    if (a.ode.n == 10) plan_grad_fwd_kernel<10><<<grid, block, 0, h->stream>>>(a);
    else plan_grad_fwd_kernel<0><<<grid, block, 0, h->stream>>>(a);
    if (T <= 512 && pairs <= 148LL * 1024) {   // beyond about one resident wave the 128-thread Jacobian kernel's occupancy wins
        // plans per block: small blocks (the Jacobian threads hold ~100 registers: 20 warps per SM whatever the block size, and
        // finer blocks leave a shorter tail) as long as there are at least four blocks per SM
        int P = 1;
        while (2 * P * T <= 512 && 2 * P <= 32 && K / (2 * P) >= 592) P *= 2;
        const int threads = ((P * T + 31) / 32) * 32;
        const size_t smem = sizeof(float) * CPS_GRAD_REC * (size_t)P * T;
        void (*fn)(const GradArgs, int) = (a.ode.n == 10) ? plan_grad_jacrev_kernel<10> : plan_grad_jacrev_kernel<0>;
        if (smem > 48 * 1024) CUDA_TRY(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        fn<<<(K + P - 1) / P, threads, smem, h->stream>>>(a, P);
        h->launches += 2;
    } else {
        if (a.ode.n == 10) plan_grad_jac_kernel<10><<<(unsigned)((pairs + jblock - 1) / jblock), jblock, 0, h->stream>>>(a);
        else plan_grad_jac_kernel<0><<<(unsigned)((pairs + jblock - 1) / jblock), jblock, 0, h->stream>>>(a);
        plan_grad_rev_kernel<<<grid, block, 0, h->stream>>>(a);
        h->launches += 3;
    }
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

extern "C" int cps_rpgd_reset(cps_handle *h) {
    if (!h) return CPS_ERR_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    GradState *G;
    int rc = grad_state(h, &G);
    if (rc != CPS_OK) return rc;
    const size_t n = (size_t)h->cfg.num_rollouts * h->cfg.horizon;
    CUDA_TRY(h, cudaMemsetAsync(G->d_m, 0, sizeof(float) * n, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(G->d_v, 0, sizeof(float) * n, h->stream));
    G->adam_iterations = 0;
    return CPS_OK;
}

extern "C" int cps_rpgd_grad_step(cps_handle *h, const float *s_dev, float *Q_dev, float u_prev, float learning_rate, float beta_1,
                                  float beta_2, float epsilon, float gradmax_clip, float *J_out_dev) {
    if (!h) return CPS_ERR_INVALID;
    if (!s_dev || !Q_dev) return fail(h, CPS_ERR_INVALID, "cps_rpgd_grad_step: null pointer");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    GradState *G;
    int rc = grad_state(h, &G);
    if (rc != CPS_OK) return rc;
    if ((rc = cps_plan_cost_grad(h, s_dev, Q_dev, CPS_ROLLOUT_MAJOR, u_prev, J_out_dev, G->d_G)) != CPS_OK) return rc;
    G->adam_iterations += 1;
    const double t = (double)G->adam_iterations;
    RpgdArgs a;
    a.Q = Q_dev; a.G = G->d_G; a.m = G->d_m; a.v = G->d_v;
    a.K = h->cfg.num_rollouts; a.T = h->cfg.horizon;
    a.clip_norm = gradmax_clip;
    a.lr_t = (float)((double)learning_rate * sqrt(1.0 - pow((double)beta_2, t)) / (1.0 - pow((double)beta_1, t)));   // ResourceApplyAdam
    a.beta1 = beta_1; a.beta2 = beta_2; a.eps = epsilon;
    a.lo = h->mppi_in[5]; a.hi = h->mppi_in[6];
    rpgd_update_kernel<<<(a.K + 3) / 4, 128, 0, h->stream>>>(a);
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

extern "C" int cps_rpgd_finish(cps_handle *h, const float *J_dev, float *Q_dev, const float *fresh_dev, int keep, int shift_previous,
                               int *ages_dev, float *u_nom_host) {
    if (!h) return CPS_ERR_INVALID;
    if (!J_dev || !Q_dev || !u_nom_host) return fail(h, CPS_ERR_INVALID, "cps_rpgd_finish: null pointer");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    GradState *G;
    int rc = grad_state(h, &G);
    if (rc != CPS_OK) return rc;
    const int K = h->cfg.num_rollouts, T = h->cfg.horizon;
    if (K > 4096) return fail(h, CPS_ERR_UNSUPPORTED, "cps_rpgd_finish: at most 4096 plans (ranks by counting)");
    if (keep < 1 || keep > K || shift_previous < 0) return fail(h, CPS_ERR_INVALID, "cps_rpgd_finish: bad keep / shift_previous");
    if (!G->d_Q2) {   // first use
        const size_t n = (size_t)K * T;
        cudaError_t e = cudaMalloc(&G->d_Q2, sizeof(float) * n);
        if (e == cudaSuccess) e = cudaMalloc(&G->d_m2, sizeof(float) * n);
        if (e == cudaSuccess) e = cudaMalloc(&G->d_v2, sizeof(float) * n);
        if (e == cudaSuccess) e = cudaMalloc(&G->d_unom, sizeof(float) * T);
        if (e == cudaSuccess) e = cudaMalloc(&G->d_ages2, sizeof(int) * K);
        if (e == cudaSuccess) e = cudaHostAlloc(&G->h_unom, sizeof(float) * T, cudaHostAllocDefault);
        if (e != cudaSuccess) return fail(h, CPS_ERR_CUDA, "cps_rpgd_finish: allocating the workspace: %s", cudaGetErrorString(e));
    }
    FinishArgs a;
    a.J = J_dev; a.Q = Q_dev; a.m = G->d_m; a.v = G->d_v; a.fresh = fresh_dev; a.ages = ages_dev;
    a.Q2 = G->d_Q2; a.m2 = G->d_m2; a.v2 = G->d_v2; a.u_nom = G->d_unom; a.ages2 = G->d_ages2;
    a.K = K; a.T = T; a.keep = keep; a.sp = shift_previous;
    rpgd_finish_kernel<<<K, 64, 0, h->stream>>>(a);
    const int n = K * T;
    rpgd_copyback_kernel<<<(n + 255) / 256 < 592 ? (n + 255) / 256 : 592, 256, 0, h->stream>>>(Q_dev, G->d_m, G->d_v, ages_dev, G->d_Q2, G->d_m2,
                                                                                                G->d_v2, G->d_ages2, K, T);
    h->launches += 2;
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaMemcpyAsync(G->h_unom, G->d_unom, sizeof(float) * T, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    memcpy(u_nom_host, G->h_unom, sizeof(float) * T);
    return CPS_OK;
}

extern "C" int cps_rpgd_adam_state(cps_handle *h, float **m_dev, float **v_dev, long long *iterations) {
    if (!h) return CPS_ERR_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    GradState *G;
    int rc = grad_state(h, &G);
    if (rc != CPS_OK) return rc;
    if (m_dev) *m_dev = G->d_m;
    if (v_dev) *v_dev = G->d_v;
    if (iterations) *iterations = G->adam_iterations;
    return CPS_OK;
}

extern "C" int cps_rpgd_set_iterations(cps_handle *h, long long iterations) {
    if (!h || iterations < 0) return CPS_ERR_INVALID;
    GradState *G;
    int rc = grad_state(h, &G);
    if (rc != CPS_OK) return rc;
    G->adam_iterations = iterations;
    return CPS_OK;
}

// ---- cps_rpgd_fleet.cu: the plans of E experiments in one launch per kernel ------------------------------------------------
// G != nullptr: the gradient -- forward with checkpoints, Jacobians to global records, reverse (the global-record path of
// cps_plan_cost_grad for every E: the launches per period do not depend on E; the records and the arithmetic per plan are the
// same as the fused kernel's, so J and G match cps_plan_cost_grad bit for bit).  G == nullptr: the costs only, J [n_plans].
// odes_dev [n_plans / kpe] or nullptr: each experiment's model constants (the _ode kernels), else the handle's.
int cps_grad_fleet(cps_handle *h, int n_plans, int kpe, const float *s_dev, const float *Q_dev, const CostParams *costs_dev,
                   const float *u_prev_dev, float *ck, float *jac, float *J, float *G, const OdeParams *odes_dev) {
    const int T = h->cfg.horizon;
    FleetGradArgs f;
    memset(&f, 0, sizeof(f));
    GradArgs &a = f.g;
    a.ode = h->ode;
    a.s = s_dev;
    a.Q = Q_dev;
    a.qs_k = T; a.qs_t = 1; a.gs_k = T; a.gs_t = 1;
    a.K = n_plans; a.T = T;
    a.full = h->cfg.cost_id == CPS_COST_QB_GRAD ? 1 : 0;
    a.inv_T1 = 1.0f / (float)(T + 1);
    a.ck = G ? ck : nullptr; a.jac = jac; a.J = J; a.G = G;
    a.nonfinite = h->d_nonfinite;
    f.x.costs = costs_dev; f.x.u_prev = u_prev_dev; f.x.kpe = kpe;
    FleetGradOdeArgs fo;
    fo.g = f.g; fo.x = f.x; fo.odes = odes_dev;
    const int block = 128, grid = (n_plans + block - 1) / block;
    if (odes_dev) {
        if (a.ode.n == 10) fleet_grad_fwd_ode_kernel<10><<<grid, block, 0, h->stream>>>(fo);
        else fleet_grad_fwd_ode_kernel<0><<<grid, block, 0, h->stream>>>(fo);
    } else {
        if (a.ode.n == 10) fleet_grad_fwd_kernel<10><<<grid, block, 0, h->stream>>>(f);
        else fleet_grad_fwd_kernel<0><<<grid, block, 0, h->stream>>>(f);
    }
    h->launches += 1;
    if (G) {
        const long long pairs = (long long)n_plans * T;
        const unsigned jgrid = (unsigned)((pairs + 127) / 128);
        if (odes_dev) {
            if (a.ode.n == 10) fleet_grad_jac_ode_kernel<10><<<jgrid, 128, 0, h->stream>>>(fo);
            else fleet_grad_jac_ode_kernel<0><<<jgrid, 128, 0, h->stream>>>(fo);
        } else {
            if (a.ode.n == 10) fleet_grad_jac_kernel<10><<<jgrid, 128, 0, h->stream>>>(f);
            else fleet_grad_jac_kernel<0><<<jgrid, 128, 0, h->stream>>>(f);
        }
        plan_grad_rev_kernel<<<grid, block, 0, h->stream>>>(a);
        h->launches += 2;
    }
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}

// rpgd_update_kernel over n_plans plans [n_plans][T] (one warp each); lr_t computed by the caller
int cps_grad_fleet_update(cps_handle *h, int n_plans, float *Q_dev, const float *G_dev, float *m_dev, float *v_dev, float lr_t,
                          float beta_1, float beta_2, float epsilon, float gradmax_clip) {
    RpgdArgs a;
    a.Q = Q_dev; a.G = G_dev; a.m = m_dev; a.v = v_dev;
    a.K = n_plans; a.T = h->cfg.horizon;
    a.clip_norm = gradmax_clip; a.lr_t = lr_t;
    a.beta1 = beta_1; a.beta2 = beta_2; a.eps = epsilon;
    a.lo = h->mppi_in[5]; a.hi = h->mppi_in[6];
    rpgd_update_kernel<<<(a.K + 3) / 4, 128, 0, h->stream>>>(a);
    h->launches += 1;
    CUDA_TRY(h, cudaGetLastError());
    return CPS_OK;
}
