// kfpos_t6.cuh -- KalmanFilterTOA (6-state constant-velocity iterated EKF on
// rangings), per-thread formulation.  Reference: algorithms/KalmanFilterTOA.cpp.
#pragma once
#include "kfpos_math.cuh"
#include "kfpos_solve.cuh"

namespace kfpos {

// P^- = F P F^T + Q for F = [[I, tI],[0, I]] and the per-axis Q of
// predictionErrorCovariance (TOA.cpp:362-391), in place on the packed matrix.
KF_DEV void t6_predict_cov(Sym<6> &P, double t, double accel_noise) {
    const double t2 = t * t / 2, a2 = accel_noise * accel_noise;
    // pp block first (needs the old pv and vv blocks)
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            const double bij = P.get(3 + j, i), bji = P.get(3 + i, j), cij = P.get(3 + i, 3 + j);
            P.at(i, j) = fma(t, (bij + bji) + t * cij, P.get(i, j));
        }
    // pv block: B + t C
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) P.at(3 + j, i) = fma(t, P.get(3 + i, 3 + j), P.get(3 + j, i));
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        P.at(i, i) += a2 * t2 * t2;
        P.at(3 + i, i) += a2 * t2 * t;
        P.at(3 + i, 3 + i) += a2 * t * t;
    }
}

// Result of one IEKF update in factored form: x = x^- + dx (position part; the
// velocity increment is never used, TOA.cpp:159-183) and P = P^- - B M B^T with
// B = P^-[:, 0:3] and M symmetric 3x3 (packed Sym<3> order xx, xy, yy, xz, yz, zz).
struct T6Result {
    double dx[3];
    double M[6];
    double cost;
};

// kalmanStep3DIgnoreAnchor (TOA.cpp:242-338) on the slots in `mask`.
//   xp : predicted position (predicted velocity is 0: TOA.cpp:110-120)
//   Pm : P^- (shared-memory column, read only)
// Returns ML_SINGULAR when a solve failed (the reference's catch at TOA.cpp:151
// then skips the update), else 0.  `out.cost` = last assigned IEKF cost.
//
// Formulation (validated against the dense oracle).  Every ranging row is
// [h_i^T 0] with h_i the unit vector anchor -> tag, and R is diagonal, so with
// A = P^-[0:3,0:3], B = P^-[:,0:3], G = J^T R^-1 J (3x3) and b = J^T R^-1 (eps - J delta):
//   K (eps - J delta) = B (I + G A)^-1 b        (push-through identity: no inverse of P^-, no m x m inverse)
//   (I - K J) P^-     = P^- - B (I + G A)^-1 G B^T
// so one IEKF iteration is ONE pass over the anchors that accumulates the cost, b and G
// (independent FMAs, no serial rank-1 chain) followed by a 3x3 solve.  I + G A has
// eigenvalues >= 1 (G, A positive semi-definite): it is never singular, also for the
// rank-3 first step P^- = Q.  The prior term delta^T pinv(P^-) delta of the cost equals
// w . dx with w = b - G dx (delta = -P^- w lies in the range of P^-).
// wmask != 0: the lanes in wmask all call this function together; they are re-converged
// after the Newton loop (whose trip count differs per lane) so that the IEKF loop is issued
// once per warp and not once per group of lanes that left the Newton loop together.
// COSTFIRST: the evaluations that usually end the Newton and the IEKF loop form the cost alone first (plain replay only)
template <bool PME, int MT, bool COSTFIRST = false>
KF_DEV int t6_update(const AnchorTable &A, const EpochT<PME, MT> &ep, unsigned mask, const double (&xp)[3],
                     const Col &Pm, T6Result &out, StepStats &st, unsigned wmask = 0u, const Col *cyc_ref = nullptr,
                     unsigned long long *cnt = nullptr) {
    // ---- inner ML solve from the predicted position (TOA.cpp:268-273)
    double pml[3] = {xp[0], xp[1], xp[2]};
    double sse, sse_xp = 0.0;
    // scalar errorEstimation: the Newton solver's pass at its start point x^- is also the IEKF's first
    // pass: cost = sse_xp / R, b = -g_xp / R (eps - J delta = eps at delta = 0), G = Gu_xp / R
    double g_xp[3] = {0.0, 0.0, 0.0}, Gu_xp[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    int rc;
    if constexpr (PME) rc = ml_solve3<PME, MT>(A, ep, mask, pml, sse, st.ml_iters, nullptr, &sse_xp, 10000u, nullptr, cyc_ref);
    else rc = ml_solve3_ekf<MT, COSTFIRST>(A, ep, mask, pml, sse, st.ml_iters, sse_xp, g_xp, Gu_xp, *cyc_ref, cnt);
    if (wmask) __syncwarp(wmask);
    if (rc == ML_FEW) st.status |= 2u;
    if (rc == ML_SINGULAR) return ML_SINGULAR;
    if (isnan(pml[0]) || isnan(pml[1]) || isnan(pml[2])) { // TOA.cpp:270-272: back to xp
        st.status |= 16u;
        sse = sse_xp;
    }
    if (mask == 0u) sse = -1.0; // estimationError of an empty list (ML.cpp:265-267)

    // R_ii = max(mlRangingError, errorEstimation_i) (TOA.cpp:281).  An epoch without rangings has no
    // rows at all: the reference's update is then x = x^-, P = P^- (K empty), whatever errorEstimation is
    // (the C++ mirror forwards such epochs with err_scalar = 0) -- the weight must be an exact 0, not 1/0.
    const double invR0 = mask ? fast_rcp(fmax(sse, ep.e0)) : 0.0;
    double a[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) a[k] = Pm[k]; // position block of P^-

    double dx[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int k = 0; k < 6; ++k) out.M[k] = 0.0;
    double cost = 1e20;
    double prior = 0.0; // delta^T pinv(P^-) delta
    bool broke = false;
    // the sums of the first iteration (scalar errorEstimation: those of the Newton solver's first pass) as the initial
    // values of the loop-carried ones, not copied in the loop (~40 moves inside the replay loop)
    double c = sse_xp, b[3] = {-g_xp[0], -g_xp[1], -g_xp[2]}, G[6] = {Gu_xp[0], Gu_xp[1], Gu_xp[2], Gu_xp[3], Gu_xp[4], Gu_xp[5]};
    for (int iter = 0; iter < 10; ++iter) {
        // ---- one pass: cost at the current iterate (TOA.cpp:297-305) and the
        //      information-form accumulators of the rows linearised there (TOA.cpp:313-320)
        if (PME || iter > 0) {
            if constexpr (COSTFIRST && !PME && MT > 0) {
                if (iter >= 2) { // the evaluation that usually ends the loop: the cost alone first (iekf_cost_only)
                    const double c2 = iekf_cost_only<MT>(A, ep, mask, xp[0] + dx[0], xp[1] + dx[1], xp[2] + dx[2]);
                    if (rel_change_lt(cost, fma(c2, invR0, prior), 1e-3)) {
                        st.cost_evals += 1;
                        broke = true;
                        break;
                    }
                }
            }
            iekf_pass<PME, MT, 3>(A, ep, mask, sse, xp[0] + dx[0], xp[1] + dx[1], xp[2] + dx[2], dx, c, b, G);
        }
        const double newCost = PME ? c + prior : fma(c, invR0, prior);
        st.cost_evals += 1;
        if (rel_change_lt(cost, newCost, 1e-3)) { broke = true; break; }
        cost = newCost;
        st.gain_evals += 1;
        if (!PME) {
#pragma unroll
            for (int k = 0; k < 3; ++k) b[k] *= invR0;
#pragma unroll
            for (int k = 0; k < 6; ++k) G[k] *= invR0;
        }
        double sgain[3];
        prior = info_gain3(a, b, G, dx, out.M, sgain);
    }
    if (!broke) st.status |= 32u;
    out.dx[0] = dx[0]; out.dx[1] = dx[1]; out.dx[2] = dx[2];
    out.cost = cost;
    return 0;
}

} // namespace kfpos
