// cps_plant.cuh -- device code shared by the two fleets (cps_fleet.cu: MPPI, cps_rpgd_fleet.cu: RPGD): the plant in the
// reference's mixed float32 / float64 arithmetic and the counter-based normal draws.
#pragma once
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>

#include "cps_device.cuh"

using namespace cps;

struct PlantParams {
    float k, m_cart, g, J_fric, M_fric, u_max, thl;
    double L, m_pole, dt;
    int n_sim;
};

// fold_ode (cps_lib.cu) on the device, same double-precision expressions: the controller's model constants for a
// per-experiment pole length / mass (add_control_along_trajectories feeds L per recorded row).  `a` is any argument block
// with the physical constants k, m_cart, g, J_fric, M_fric, u_max, m_pole_fixed and the substep h_step (FleetArgs of
// cps_fleet.cu, RpgdRowArgs of cps_rpgd_fleet.cu).
template <int INTEG, class A>
__device__ __forceinline__ void fold_ode_device(const A &a, double L, double mp_in, OdeParams &o) {
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

// Draws i = 0..n_ind-1 of rollout k, experiment e_global, controller period `period`; dst[i * stride].
__device__ __forceinline__ void fleet_draws(unsigned long long seed, unsigned period, unsigned e_global, unsigned k,
                                            int n_ind, float *dst, long long stride) {
    const uint2 key = make_uint2((unsigned)seed, (unsigned)(seed >> 32));
    for (int g = 0; 4 * g < n_ind; ++g) {
        const uint4 r = philox4x32_10(make_uint4(k, (unsigned)g, period, e_global), key);
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

// The RPGD fleet's sampling draws (cps_rpgd_fleet.cu): draws i = 0..n_ind-1 of plan row `row`, dst[i * stride].  Counter
// (row, tag + draw group, period, global experiment): the tag in the second word keeps them apart from the rollout draws
// above (second word = draw group < 2^28) and from the plant-side draws (second word 0xFFFFFFFF).  tag: RPGD_DRAWS_RESAMPLE
// for the resampling solve of `period`, RPGD_DRAWS_RESET (period 0) for the plans of a reset.
// Deliberately a copy of fleet_draws' loop rather than a shared one with a tag argument: fleet_draws is inlined into
// fleet_kernel, whose code must not change with the RPGD fleet (its SASS is checked byte for byte).
#define RPGD_DRAWS_RESAMPLE 0xA0000000u
#define RPGD_DRAWS_RESET 0xB0000000u
__device__ __forceinline__ void rpgd_draws(unsigned long long seed, unsigned tag, unsigned period, unsigned e_global, unsigned row,
                                           int n_ind, float *dst, long long stride) {
    const uint2 key = make_uint2((unsigned)seed, (unsigned)(seed >> 32));
    for (int g = 0; 4 * g < n_ind; ++g) {
        const uint4 r = philox4x32_10(make_uint4(row, tag + (unsigned)g, period, e_global), key);
        float n[4];
        box_muller(r.x, r.y, n[0], n[1]);
        box_muller(r.z, r.w, n[2], n[3]);
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (4 * g + q < n_ind) dst[(long long)(4 * g + q) * stride] = n[q];
    }
}
