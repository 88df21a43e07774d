// cps_plant.cuh -- code shared by the fleets (cps_fleet.cu: MPPI on the ODE or the network, cps_rpgd_fleet.cu: RPGD): the
// plant in the reference's mixed float32 / float64 arithmetic, the record row, the counter-based normal draws and the
// device-side fold of the controller's model constants, with the host functions that fill their parameter blocks.
#pragma once
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>

#include "cps_device.cuh"
#include "cps_internal.cuh"

using namespace cps;

struct PlantParams {
    float k, m_cart, g, J_fric, M_fric, u_max, thl;
    double L, m_pole, dt;
    int n_sim;
};

// The plant of the handle's physical constants, n_sim ticks of dt_simulation per controller period
static inline PlantParams plant_params(const cps_handle *h, double dt_simulation, int sim_substeps) {
    PlantParams P;
    P.k = h->phys[CPS_PH_K]; P.m_cart = h->phys[CPS_PH_M_CART]; P.g = h->phys[CPS_PH_G]; P.J_fric = h->phys[CPS_PH_J_FRIC];
    P.M_fric = h->phys[CPS_PH_M_FRIC]; P.u_max = h->phys[CPS_PH_U_MAX]; P.thl = h->phys[CPS_PH_TRACK_HALF_LENGTH];
    P.L = (double)h->phys[CPS_PH_L]; P.m_pole = (double)h->phys[CPS_PH_M_POLE];
    P.dt = dt_simulation; P.n_sim = sim_substeps;
    return P;
}

// What fold_ode_device reads besides L and m_pole: the physical constants, the substep and the handle's L / m_pole "for
// controller" (used when a fleet is given only one of the per-row arrays).
struct FoldInputs {
    float k, m_cart, g, J_fric, M_fric, u_max;
    float m_pole_fixed;         // ODE_v0 takes only L from the variable parameters
    float L_default, mp_default;
    double h_step;              // substep dt / n in double
};

static inline FoldInputs fold_inputs(const cps_handle *h) {
    FoldInputs f;
    f.k = h->phys[CPS_PH_K]; f.m_cart = h->phys[CPS_PH_M_CART]; f.g = h->phys[CPS_PH_G]; f.J_fric = h->phys[CPS_PH_J_FRIC];
    f.M_fric = h->phys[CPS_PH_M_FRIC]; f.u_max = h->phys[CPS_PH_U_MAX];
    f.m_pole_fixed = h->phys[CPS_PH_M_POLE];
    f.L_default = h->L_var; f.mp_default = h->m_pole_var;
    f.h_step = (double)h->cfg.dt / (double)h->cfg.substeps;
    return f;
}

// fold_ode (cps_lib.cu) on the device, same double-precision expressions: the controller's model constants for a
// per-experiment pole length / mass (add_control_along_trajectories feeds L per recorded row).
template <int INTEG>
__device__ __forceinline__ void fold_ode_device(const FoldInputs &a, double L, double mp_in, OdeParams &o) {
    const double k = a.k, mc = a.m_cart, g = a.g, J = a.J_fric, M = a.M_fric, umax = a.u_max;
    const double mp = (INTEG == 0) ? (double)a.m_pole_fixed : mp_in;
    const double kp1 = k + 1.0, Lh = L / 2.0;
    o.KM = (float)(kp1 * (mc + mp));
    o.m_p = (float)mp;
    o.c1 = (float)(mp * g);
    o.c2 = (float)(kp1 * mp * Lh);
    o.c3 = (float)(J / Lh);
    o.c5 = (float)(kp1 * M);
    o.d1 = (float)(g / (kp1 * Lh));
    o.d2 = (float)(1.0 / (kp1 * Lh));
    o.d3 = (float)(J / (mp * Lh * kp1 * Lh));
    o.bounce = (float)(2.0 / (0.5 * L));
    const double hh = a.h_step;
    const double hd2 = hh * (1.0 / (kp1 * Lh));
    o.yc1 = (float)(hd2 * (mp * g));
    o.yc2 = (float)(hd2 * (kp1 * mp * Lh));
    o.yc3 = (float)(hd2 * (J / Lh));
    o.yc5 = (float)(hd2 * (kp1 * M));
    o.yu_scale = (float)(hd2 * (kp1 * umax));
    o.v_y = (float)(kp1 * Lh);
    o.hd1 = (float)(hh * (g / (kp1 * Lh)));
    o.hd3 = (float)(hh * (J / (mp * Lh * kp1 * Lh)));
    // the rotation constants and w_rot_max depend on the step only: the handle's fold stands
}

// experiment e's cost parameters for its targets (null: 0 / +1)
__device__ __forceinline__ CostParams fold_cost_e(const CostParams &up, const CostParams &dn, const float *tp, const float *te,
                                                  int e) {
    const float tpe = tp ? tp[e] : 0.0f, tee = te ? te[e] : 1.0f;
    CostParams c = (tee == 1.0f) ? up : dn;   // quadratic_boundary_grad selects its weight set on the target equilibrium
    c.target_position = tpe;
    c.target_equilibrium = tee;
    return c;
}

// ---- Philox4x32-10 (Salmon et al., SC'11), the counter-based generator torch / TF / cuRAND also use ---------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

// Two standard normals from two 32-bit words (Box-Muller on 24-bit uniforms in (0, 1)).
__device__ __forceinline__ void box_muller(unsigned a, unsigned b, float &n0, float &n1) {
    const float u1 = ((float)(a >> 8) + 0.5f) * 5.9604644775390625e-8f;  // 2^-24
    const float u2 = ((float)(b >> 8) + 0.5f) * 5.9604644775390625e-8f;
    const float r = sqrtf(-2.0f * logf(u1));
    float sn, cs;
    sincospif(2.0f * u2, &sn, &cs);
    n0 = r * cs;
    n1 = r * sn;
}

// Standard normals i = 0..n_ind-1, dst[i * stride], four per counter (w0, w1 + i / 4, period, e_global).  The fleets'
// streams: the MPPI rollout draws have w0 = rollout, w1 = 0 (second word = draw group < 2^28); the RPGD plan draws have
// w0 = plan row, w1 = RPGD_DRAWS_RESAMPLE (the resampling solve of `period`) or RPGD_DRAWS_RESET (period 0, the plans of
// a reset); the CEM draws of outer iteration `it` have w0 = plan, w1 = CEM_DRAWS + it * ceil(T / 4) (second word below
// CEM_DRAWS + 2^28: cps_cem_fleet_create bounds the iterations); the plant-side draws of cps_fleet.cu have second word
// 0xFFFFFFFF.  The second words keep them disjoint.
#define RPGD_DRAWS_RESAMPLE 0xA0000000u
#define RPGD_DRAWS_RESET 0xB0000000u
#define CEM_DRAWS 0xC0000000u
__device__ __forceinline__ void philox_normals(unsigned long long seed, unsigned w0, unsigned w1, unsigned period,
                                               unsigned e_global, int n_ind, float *dst, long long stride) {
    const uint2 key = make_uint2((unsigned)seed, (unsigned)(seed >> 32));
    for (int g = 0; 4 * g < n_ind; ++g) {
        const uint4 r = philox4x32_10(make_uint4(w0, w1 + (unsigned)g, period, e_global), key);
        float n[4];
        box_muller(r.x, r.y, n[0], n[1]);
        box_muller(r.z, r.w, n[2], n[3]);
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (4 * g + q < n_ind) dst[(long long)(4 * g + q) * stride] = n[q];
    }
}

// ---- the plant (device restatement of oracle/cps_oracle.c: ode_plant, plant_integrate; no FMA contraction) ------------
__device__ __forceinline__ void plant_ode(const PlantParams &P, float ca, float sa, float angleD, float positionD, float u,
                                          double &angleDD, double &positionDD) {
    const double kp1 = (double)__fadd_rn(P.k, 1.0f);
    const float ca2 = __fmul_rn(ca, ca), aD2 = __fmul_rn(angleD, angleD);
    const double A = __dsub_rn(__dmul_rn(kp1, __dadd_rn((double)P.m_cart, P.m_pole)), __dmul_rn(P.m_pole, (double)ca2));
    const float F_fric = __fmul_rn(-P.M_fric, positionD);
    const float T_fric = __fmul_rn(-P.J_fric, angleD);
    const double L_half = P.L / 2.0;
    const double grav = __dmul_rn(__dmul_rn(__dmul_rn(P.m_pole, (double)P.g), (double)sa), (double)ca);
    const double fric = (double)__fmul_rn(T_fric, ca) / L_half;
    const double centr = -__dmul_rn(__dmul_rn(__dmul_rn(P.m_pole, L_half), (double)aD2), (double)sa);
    const double inner = __dadd_rn(__dadd_rn(centr, (double)F_fric), (double)u);
    const double pDD = __dadd_rn(__dadd_rn(grav, fric), __dmul_rn(kp1, inner)) / A;
    positionDD = pDD;
    const double num = __dadd_rn(__dadd_rn((double)__fmul_rn(P.g, sa), __dmul_rn(pDD, (double)ca)),
                                 (double)T_fric / __dmul_rn(P.m_pole, L_half));
    angleDD = num / __dmul_rn(kp1, L_half);
}

__device__ __forceinline__ double plant_wrap(double angle) {
    const double two_pi = 6.283185307179586, pi = 3.141592653589793;
    const double m = fmod(angle, two_pi);
    if (m < -pi) return m + two_pi;
    if (m > pi) return m - two_pi;
    return m;
}

__device__ __forceinline__ void plant_tick(const PlantParams &P, float *s, double aDD, double pDD) {
    const float angle = s[IDX_ANGLE], angleD = s[IDX_ANGLED], position = s[IDX_POS], positionD = s[IDX_POSD];
    const double angleD_next = __dadd_rn((double)angleD, __dmul_rn(aDD, P.dt));
    const double positionD_next = __dadd_rn((double)positionD, __dmul_rn(pDD, P.dt));
    const double angle_next = __dadd_rn((double)angle, __dmul_rn(angleD_next, P.dt));
    const double position_next = __dadd_rn((double)position, __dmul_rn(positionD_next, P.dt));
    s[IDX_ANGLE] = (float)angle_next; s[IDX_ANGLED] = (float)angleD_next;
    s[IDX_POS] = (float)position_next; s[IDX_POSD] = (float)positionD_next;
    if (s[IDX_POS] >= P.thl || -s[IDX_POS] >= P.thl) {  // edge_bounce (cartpole_equations.py:341-347)
        const float a = s[IDX_ANGLE], aD = s[IDX_ANGLED], p = s[IDX_POS], pD = s[IDX_POSD];
        const float ca = cosf(a);
        const double aD2 = __dsub_rn((double)aD, __dmul_rn(2.0, (double)__fmul_rn(pD, ca)) / __dmul_rn(0.5, P.L));
        const double a2 = __dadd_rn((double)a, __dmul_rn(aD2, P.dt));
        const float pD2 = -pD;
        const double p2 = __dadd_rn((double)p, __dmul_rn((double)pD2, P.dt));
        s[IDX_ANGLE] = (float)a2; s[IDX_ANGLED] = (float)aD2; s[IDX_POS] = (float)p2; s[IDX_POSD] = pD2;
    }
    s[IDX_COS] = cosf(s[IDX_ANGLE]);   // of the UNWRAPPED angle (CartPole/__init__.py:329-334)
    s[IDX_SIN] = sinf(s[IDX_ANGLE]);
    s[IDX_ANGLE] = (float)plant_wrap((double)s[IDX_ANGLE]);
}

// The fleets' record row of one controller period (include/cps.h CPS_FLEET_RECORD): the state the controller was called
// on with its second derivatives, Qc = the controller's control, Q = the applied one (after control noise), u = u_max Q,
// and the targets.
__device__ __forceinline__ void plant_record(float *r, double time, const float *s, double aDD, double pDD, float Qc, float Q,
                                             float u, float tp, float te) {
    r[0] = (float)time;
    r[1] = s[IDX_ANGLE]; r[2] = s[IDX_ANGLED]; r[3] = (float)aDD; r[4] = s[IDX_COS]; r[5] = s[IDX_SIN];
    r[6] = s[IDX_POS]; r[7] = s[IDX_POSD]; r[8] = (float)pDD;
    r[9] = Qc; r[10] = Q; r[11] = u; r[12] = tp; r[13] = te; r[14] = 0.0f; r[15] = 0.0f;
}

// The plant period of fleets whose solve leaves each experiment's control in an [E] array (the neural MPPI fleet of
// cps_fleet.cu, the CEM fleet of cps_cem_fleet.cu): fleet_net_plant_kernel, one thread per experiment, writes the record
// row with Q_applied = Q and advances the state.  fleet_plant_launch (cps_fleet.cu) launches it on the handle's stream.
struct NetPlantArgs {
    PlantParams plant;
    float *s;                   // [E][8]
    const float *u;             // [E] the controls the solve just chose
    const float *tp, *te;       // [E] targets of this period (null: 0 / +1)
    float *record;              // [E][CPS_FLEET_RECORD] of this period, or null
    double time;                // period * dt_control
    int E;
};
int fleet_plant_launch(cps_handle *h, const NetPlantArgs &a);

// The n_sim ticks of one controller period with u held (CartPole/__init__.py:283-324): (aDD, pDD) enter as the second
// derivatives of s and leave as those of the new state; on_tick(i) runs after tick i.  The caller computes the first pair
// (plant_ode) itself: folding that and the record row in here changes how fleet_kernel's solve is scheduled.
template <class Tick>
__device__ __forceinline__ void plant_ticks(const PlantParams &P, float *s, float u, double &aDD, double &pDD, Tick on_tick) {
    for (int i = 0; i < P.n_sim; ++i) {
        plant_tick(P, s, aDD, pDD);
        plant_ode(P, s[IDX_COS], s[IDX_SIN], s[IDX_ANGLED], s[IDX_POSD], u, aDD, pDD);
        on_tick(i);
    }
}
