// cps_grad_partials.cuh -- partial derivatives of the gradient cost plugins' stage cost, shared by the adjoints of the
// ODE predictor (cps_grad.cu) and of the neural predictor (cps_net_grad.cu).
#pragma once
#include "cps_internal.cuh"

// sincosf / cosf for the angles a rollout produces: fold_angle leaves every angle after the first substep in [-pi, pi], where
// sincos_folded is bit-identical to the math library (cps_selftest_sincos); anything else (a caller-supplied unwrapped
// initial angle) takes the library call, out of line.
static __device__ __noinline__ void sincos_library(float a, float *s, float *c) { sincosf(a, s, c); }
__device__ __forceinline__ void sincos_th(float th, float &s, float &c) {
    if (__builtin_expect(fabsf(th) <= CPS_PI_F, 1)) sincos_folded(th, s, c);
    else sincos_library(th, &s, &c);
}

// Partial derivatives of the stage cost with respect to (angle, angleD, position).
// quadratic_boundary_grad_minimal (Control_Toolkit_ASF/Cost_Functions/CartPole/quadratic_boundary_grad_minimal.py:62-130);
// w: [dd_q, db, ep, ekp, cc*R, bf = f thl, 1/((1-f) thl)] as in stage_cost<COST_GRADMIN>.
__device__ __forceinline__ void gradmin_partials(const CostParams &C, float th, float w, float x, float &d_th, float &d_w,
                                                 float &d_x) {
    float sn, c;
    sincos_th(th, sn, c);
    const float dist = (x - C.target_position) * C.inv_2thl;
    const float apos = fabsf(x);
    const float over = (apos > C.w[5]) ? (apos - C.w[5]) * C.w[6] : 0.0f;
    d_x = fmaf(C.w[0] * 2.0f * dist, C.inv_2thl, C.w[1] * 2.0f * over * C.w[6] * copysignf(1.0f, x));
    d_th = C.w[2] * 2.0f * (1.0f - C.target_equilibrium * c) * (C.target_equilibrium * sn);
    d_w = 2.0f * C.w[3] * w;
}
// quadratic_boundary_grad (quadratic_boundary_grad.py:62-142, 202-240); w as in stage_cost<COST_GRAD>:
// [dd_q, dd_lin, db, ep, ekp, cc*R, ccrc, bf, 1/((1-f) thl), tmax, cos(admissible angle)].  The kinetic term is
// |angleD^2 - tmax scaling(angle)| with the target under stop_gradient (:133-139): no derivative with respect to the angle.
__device__ __forceinline__ float sgnf(float x) { return (float)(x > 0.0f) - (float)(x < 0.0f); }   // d|x|/dx with 0 at 0, as autograd
__device__ __forceinline__ void grad_partials(const CostParams &C, float th, float w, float x, float &d_th, float &d_w,
                                              float &d_x) {
    float sn, c;
    sincos_th(th, sn, c);
    const float e = C.target_equilibrium;
    const float dist = (x - C.target_position) * C.inv_2thl;
    const float apos = fabsf(x);
    const float over = (apos > C.w[7]) ? (apos - C.w[7]) * C.w[8] : 0.0f;
    d_x = fmaf(C.w[0] * 2.0f * dist, C.inv_2thl, C.w[2] * 2.0f * over * C.w[8] * copysignf(1.0f, x)) + C.w[1] * sgnf(dist) * C.inv_2thl;
    d_th = C.w[3] * 2.0f * (2.0f - e * c) * (e * sn);
    const float scaling = (e * (c - C.w[10]) > 0.0f) ? 0.0f : 0.5f * (1.0f - e * c);
    d_w = C.w[4] * sgnf(fmaf(w, w, -C.w[9] * scaling)) * 2.0f * w;
}
