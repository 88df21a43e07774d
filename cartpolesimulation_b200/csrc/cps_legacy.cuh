// cps_legacy.cuh -- what the legacy front-end (cps_legacy.cu) and the legacy controller fleet (cps_legacy_fleet.cu) share:
// the stage cost q() and the handle check.
#pragma once
#include "cps_internal.cuh"

// q() for one rollout and one horizon step (controller_mppi_cartpole.py:218-268).  ca = cos(angle); un = nominal input,
// du = perturbation, up = previous iteration's nominal input of this step.  Terms are added in the reference's order.
__device__ __forceinline__ float legacy_stage(const CostParams &C, const MppiParams &mp, float ca, float angleD, float x,
                                              float xD, float un, float du, float up) {
    const float dist = (x - C.target_position) * C.inv_2thl;
    const float dd = C.w[0] * fmaf(dist, dist, (fabsf(x) > C.w[5]) ? 1.0e6f : 0.0f);  // distance_difference_cost (:138-143)
    const float ep = C.w[1] * sq(1.0f - ca);                                           // E_pot_cost (:131-135)
    const float ekp = C.w[2] * (angleD * angleD);                                      // E_kin_pol (:125-128)
    const float ekc = C.w[3] * (xD * xD);                                              // E_kin_cart (:119-122)
    const float Q = un + du;
    float cc = fmaf(mp.cc_half_nu * du, du, fmaf(mp.cc_R * un, du, mp.cc_half_R * (un * un)));  // (:254-256)
    if (fabsf(Q) > 1.0f) cc = 1.0e5f;                                                  // input-constraint penalty (:263)
    const float ccrc = C.w[4] * sq(Q - up);                                            // control_change_rate_cost (:146-149)
    return ((((dd + ep) + ekp) + ekc) + cc) + ccrc;
}

static inline int legacy_check(cps_handle *h, const char *who) {
    if (h->cfg.cost_id != CPS_COST_LEGACY_MPPI)
        return fail(h, CPS_ERR_NOT_CONFIGURED, "%s: handle was not created with CPS_COST_LEGACY_MPPI", who);
    return CPS_OK;
}
