// kfpos_solve.cuh -- per-thread ML (Newton) multilateration and the information-form
// ranging pass of the iterated EKFs: the B200 formulation of
// MLLocation::estimatePosition / estimatePosition2D (ML.cpp:48-257) and of the ranging
// rows of kalmanStep3D* (TOA.cpp:293-326, KF.cpp:451-495, TOAIMU.cpp:303-334).
//
// One thread owns one filter / epoch.  The SM sub-partition dispatches one FP64
// instruction every ~2.3 cycles and any other instruction in 1 (profiles/README.md), so the
// kernels are bound by  2.3 * (#FP64 instr) + (#other instr):  everything here is written
// to minimise that sum --
//   * MT > 0: the anchor count is a compile-time constant, the anchor loops are fully
//     unrolled, the anchor coordinates fold into the DADD operands as constant-bank
//     references, the epoch's ranges live in registers, and a missing ranging is handled
//     by zeroing its 1/d and r (two predicated moves) instead of a branch;
//   * MT == 0: run-time anchor count, rolled loops, ranges in a shared-memory column;
//   * one Newton iteration = ONE pass over the anchors (stop cost, SSE, gradient,
//     Hessian together; the reference evaluates the distances three times);
//   * one IEKF iteration = ONE pass (cost, b = J^T R^-1 y, G = J^T R^-1 J) + a 3x3 / 2x2 solve;
//   * reciprocal / reciprocal square root = MUFU seed + one cubic correction.
#pragma once
#include "kfpos_math.cuh"

namespace kfpos {

// Valid rangings of one epoch in metres.  PME = per-measurement errorEstimation column
// `e` (shared memory); otherwise the scalar e0 applies to every ranging.
template <bool PME, int MT = 0>
struct EpochT {
    Col z; // MT == 0: shared-memory column
    Col e;
    double zr[MT > 0 ? MT : 1]; // MT > 0: registers
    double e0;
    unsigned valid;
    int m_slots;
    KF_DEV int m() const { return MT > 0 ? MT : m_slots; }
    KF_DEV double r(int i) const { return MT > 0 ? zr[i] : z[i]; }
    // run-time index (MT > 0: a select chain over the register copy)
    KF_DEV double z_at(int i) const {
        if (MT == 0) return z[i];
        double v = 0.0;
#pragma unroll
        for (int k = 0; k < (MT > 0 ? MT : 1); ++k) v = (k == i) ? zr[k] : v;
        return v;
    }
    KF_DEV double err(int i) const { return PME ? e[i] : e0; }
};

// fabs(cost - newCost) / cost > 1e-3  (ML.cpp:67,165), bit-exact without the division
// unless the quotient is within 1e-9 of the threshold.
// (the division itself out of line: it is reached when the quotient is within 1e-9 of the threshold or the cost is
// not positive, and inlined it costs ~40 instructions at each of a dozen call sites of kernels whose code is
// several times the instruction cache)
static __device__ __noinline__ double rel_change_quotient(double q, double cost) { return q / cost; }
// (likewise the counters of rare events inside the replay loops)
static __device__ __noinline__ void count_rare_event(unsigned long long *c) { atomicAdd(c, 1ull); }
// (and the jump over whole periods when Brent's cycle detection fires: an integer modulo)
static __device__ __noinline__ unsigned skip_whole_periods(unsigned iter, unsigned per) { return 10000u - (10000u - iter) % per; }
// (the same with its rare-event counter, for the EKFs' inner solver: one call site in the Newton loop instead of two)
static __device__ __noinline__ unsigned skip_whole_periods_counted(unsigned iter, unsigned per, unsigned long long *cnt) {
    if (cnt) atomicAdd(cnt + CNT_ML_CYCLES, 1ull);
    return 10000u - (10000u - iter) % per;
}
KF_DEV bool rel_change_gt(double cost, double newCost) {
    const double q = fabs(cost - newCost);
    if (cost > 0.0) {
        const double t = 1e-3 * cost;
        if (q > t * 1.000000001) return true;
        if (q < t * 0.999999999) return false;
    }
    return rel_change_quotient(q, cost) > 1e-3;
}
// fabs(cost - newCost) / cost < tol  (TOA.cpp:307, KF.cpp:470, TOAIMU.cpp:312)
KF_DEV bool rel_change_lt(double cost, double newCost, double tol) {
    const double q = fabs(cost - newCost);
    if (cost > 0.0) {
        const double t = tol * cost;
        if (q < t * 0.999999999) return true;
        if (q > t * 1.000000001) return false;
    }
    return rel_change_quotient(q, cost) < tol;
}

// Exact shortcut for Newton iterations that never meet the stop test.  The iteration is a
// deterministic map p -> F(p) (the stop test is a function of two successive points), and in floating
// point an oscillating sequence almost always becomes EXACTLY periodic after a few hundred steps.
// Brent's cycle detection compares the iterate with a reference point that is refreshed at powers of
// two; a bit-for-bit match after `lam` steps proves that the sequence repeats with period lam and --
// having just gone once around without stopping -- that it will run to the reference's cap of 10000
// iterations (ML.cpp:67,165).  The caller then skips whole periods: the remaining
// (10000 - iter) mod lam iterations end in exactly the state the full run would reach.  Used by the
// EKFs' inner solver, where one such solve would hold a warp of the persistent replay kernel for
// milliseconds (the ML kernel parks long solves instead, kfpos_mlk.cu).
// (implemented inline in ml_solve3_ekf: the reference point lives in three shared-memory words, the
// iteration counter is the clock, so the common 2-4 step solve pays one load and one compare a step)

struct MlPass3 {
    double wcost, sse;
    double g[3];
    double H[6]; // packed Sym<3>: xx, xy, yy, xz, yz, zz
};

// gradient / Hessian / costs at p over the slots in `mask` (ML.cpp:171-222).
// With a scalar errorEstimation the weight 1/e is common to g and H and cancels in
// the Newton step, so only the stop-test cost carries it.
// ACCG (scalar errorEstimation only): also accumulate Gu = sum u u^T of the unit vectors, packed
// xx, xy, yy, xz, yz, zz -- with sse and g of the same pass that is everything the FIRST iteration of
// the IEKF needs at this point (cost = sse / R, b = -g / R, G = Gu / R), see t6_update.
template <bool PME, int MT, bool ACCG = false>
KF_DEV void ml_pass3(const AnchorTable &A, const EpochT<PME, MT> &ep, unsigned mask, int nvalid,
                     const double (&p)[3], MlPass3 &o, double *Gu = nullptr) {
    double wc = 0.0, sse = 0.0, g0 = 0.0, g1 = 0.0, g2 = 0.0;
    double h0 = 0.0, h1 = 0.0, h2 = 0.0, h3 = 0.0, h4 = 0.0, h5 = 0.0, c1s = 0.0;
    double u0 = 0.0, u1 = 0.0, u2 = 0.0, u3 = 0.0, u4 = 0.0, u5 = 0.0;
#pragma unroll(MT > 0 ? MT : 2)
    for (int i = 0; i < ep.m(); ++i) {
        const bool on = (mask >> i) & 1u;
        if (MT == 0 && !on) continue;
        const double dx = A.x[i] - p[0], dy = A.y[i] - p[1], dz = A.z[i] - p[2];
        const double d2 = fma(dz, dz, fma(dy, dy, dx * dx));
        double invd = MT > 0 ? fast_rsqrt_masked(d2, on) : fast_rsqrt(d2); // a missing ranging contributes exact zeros
        double r = ep.r(i);
        if (MT > 0) r = on ? r : 0.0;
        const double res = fma(-d2, invd, r);
        const double rid = r * invd;
        if (PME) {
            const double w = fast_rcp(ep.e[i]);
            sse = fma(res, res, sse);
            wc = fma(res * res, w, wc);
            const double t = res * invd * w;
            g0 = fma(t, dx, g0); g1 = fma(t, dy, g1); g2 = fma(t, dz, g2);
            c1s = fma(1.0 - rid, w, c1s);
            const double c2 = rid * invd * invd * w;
            const double cx = c2 * dx, cy = c2 * dy, cz = c2 * dz;
            h0 = fma(cx, dx, h0); h1 = fma(cx, dy, h1); h2 = fma(cy, dy, h2);
            h3 = fma(cx, dz, h3); h4 = fma(cy, dz, h4); h5 = fma(cz, dz, h5);
        } else {
            sse = fma(res, res, sse);
            const double t = res * invd;
            g0 = fma(t, dx, g0); g1 = fma(t, dy, g1); g2 = fma(t, dz, g2);
            c1s += rid; // sum of (1 - r/d) = nvalid - sum r/d
            const double w2 = invd * invd;
            const double c2 = rid * w2;
            const double cx = c2 * dx, cy = c2 * dy;
            h0 = fma(cx, dx, h0); h1 = fma(cx, dy, h1); h2 = fma(cy, dy, h2);
            h3 = fma(cx, dz, h3); h4 = fma(cy, dz, h4);
            // the zz sums follow from the unit length of (dx, dy, dz) / d after the loop
            if (ACCG) {
                const double wx = w2 * dx, wy = w2 * dy;
                u0 = fma(wx, dx, u0); u1 = fma(wx, dy, u1); u2 = fma(wy, dy, u2);
                u3 = fma(wx, dz, u3); u4 = fma(wy, dz, u4);
            }
        }
    }
    if (!PME) {
        // sum_i (r_i/d_i) u_i u_i^T has trace sum_i r_i/d_i and sum_i u_i u_i^T has trace nvalid (u_i = unit
        // vector, 0 for a missing ranging): the zz entries cost two subtractions instead of a
        // multiply and an FMA per anchor
        h5 = (c1s - h0) - h2;
        if (ACCG) u5 = ((double)nvalid - u0) - u2;
        c1s = (double)nvalid - c1s;
    }
    if (ACCG) { Gu[0] = u0; Gu[1] = u1; Gu[2] = u2; Gu[3] = u3; Gu[4] = u4; Gu[5] = u5; }
    o.sse = sse;
    o.wcost = PME ? wc : sse * fast_rcp(ep.e0);
    o.g[0] = g0; o.g[1] = g1; o.g[2] = g2;
    o.H[0] = h0 + c1s; o.H[1] = h1; o.H[2] = h2 + c1s; o.H[3] = h3; o.H[4] = h4; o.H[5] = h5 + c1s;
}

// return codes of the ML solvers
#define ML_OK 0
#define ML_FEW 1       // fewer than minRangings: position = start (ML.cpp:54-58,158-161)
#define ML_SINGULAR -1 // arma::solve / inv would throw

// covariance of the 3-D estimate, ML.cpp:229-254: J_i = (p - b_i)/d_i ; W = diag(max(e_i, SSE)) ;
// cov = inv(J^T W^-1 J), packed Sym<3>
template <bool PME, int MT>
KF_DEV int ml_cov3(const AnchorTable &A, const EpochT<PME, MT> &ep, unsigned mask, const double (&p)[3], double sse,
                   double *cov) {
    double M[6] = {0, 0, 0, 0, 0, 0};
    if (MT > 0) {
        // compile-time anchor count: unrolled, a missing ranging weighs 0, one MUFU-seeded reciprocal per ranging
        // (<= 1 ulp, kfpos_math.cuh) instead of two IEEE divisions with their slow-path branches -- the eight
        // chains interleave (the rolled form below waits ~200 cycles per ranging on its own divisions)
#pragma unroll
        for (int i = 0; i < (MT > 0 ? MT : 1); ++i) {
            const bool on = (mask >> i) & 1u;
            const double dx = p[0] - A.x[i], dy = p[1] - A.y[i], dz = p[2] - A.z[i];
            const double d2 = fma(dz, dz, fma(dy, dy, dx * dx));
            const double wr = fast_rcp(d2 * fmax(ep.err(i), sse));
            const double w = on ? wr : 0.0;
            M[0] = fma(w * dx, dx, M[0]);
            M[1] = fma(w * dx, dy, M[1]);
            M[2] = fma(w * dy, dy, M[2]);
            M[3] = fma(w * dx, dz, M[3]);
            M[4] = fma(w * dy, dz, M[4]);
            M[5] = fma(w * dz, dz, M[5]);
        }
    }
    for (int i = 0; i < (MT > 0 ? 0 : ep.m_slots); ++i) {
        if (!((mask >> i) & 1u)) continue;
        const double dx = p[0] - A.x[i], dy = p[1] - A.y[i], dz = p[2] - A.z[i];
        const double id2 = 1.0 / (dx * dx + dy * dy + dz * dz);
        const double w = id2 / fmax(ep.err(i), sse);
        M[0] = fma(w * dx, dx, M[0]);
        M[1] = fma(w * dx, dy, M[1]);
        M[2] = fma(w * dy, dy, M[2]);
        M[3] = fma(w * dx, dz, M[3]);
        M[4] = fma(w * dy, dz, M[4]);
        M[5] = fma(w * dz, dz, M[5]);
    }
    double I[6];
    if (!inv_sym3(M, I)) return ML_SINGULAR;
#pragma unroll
    for (int k = 0; k < 6; ++k) cov[k] = I[k];
    return ML_OK;
}

// covariance of the 2-D estimate, ML.cpp:118-141 (xx, xy, yy)
template <bool PME, int MT>
KF_DEV int ml_cov2(const AnchorTable &A, const EpochT<PME, MT> &ep, unsigned mask, const double (&p)[3], double sse,
                   double *cov) {
    double m00 = 0, m01 = 0, m11 = 0;
    if (MT > 0) { // unrolled, one MUFU-seeded reciprocal per ranging (see ml_cov3)
#pragma unroll
        for (int i = 0; i < (MT > 0 ? MT : 1); ++i) {
            const bool on = (mask >> i) & 1u;
            const double dx = p[0] - A.x[i], dy = p[1] - A.y[i], dz = p[2] - A.z[i];
            const double d2 = fma(dz, dz, fma(dy, dy, dx * dx));
            const double wr = fast_rcp(d2 * fmax(ep.err(i), sse));
            const double w = on ? wr : 0.0;
            m00 = fma(w * dx, dx, m00);
            m01 = fma(w * dx, dy, m01);
            m11 = fma(w * dy, dy, m11);
        }
    }
    for (int i = 0; i < (MT > 0 ? 0 : ep.m_slots); ++i) {
        if (!((mask >> i) & 1u)) continue;
        const double dx = p[0] - A.x[i], dy = p[1] - A.y[i], dz = p[2] - A.z[i];
        const double id2 = 1.0 / (dx * dx + dy * dy + dz * dz);
        const double w = id2 / fmax(ep.err(i), sse);
        m00 = fma(w * dx, dx, m00);
        m01 = fma(w * dx, dy, m01);
        m11 = fma(w * dy, dy, m11);
    }
    const double det = m00 * m11 - m01 * m01;
    if (!usable_det(det)) return ML_SINGULAR;
    const double id = 1.0 / det;
    cov[0] = m11 * id;
    cov[1] = -m01 * id;
    cov[2] = m00 * id;
    return ML_OK;
}

// estimatePosition (3-D), ML.cpp:153-257.  p: in = start, out = estimate.
// sse_out = estimationError at the returned point, sse_start = at the start point.
// The covariance inv(J^T W^-1 J) (ML.cpp:229-254) is produced only when cov != nullptr.
// iter_cap < 10000 makes the solver resumable: when `iter_cap` iterations were not enough it
// returns ML_MORE with (cost, iter) in `rs` and the current point in p; calling it again with
// that `rs` continues the same iteration sequence (the ML kernel parks such epochs in a
// queue so that a few slow epochs do not hold their whole warp for 10000 iterations).
struct MlResume {
    double cost;
    unsigned iter; // 0 = fresh start
};
#define ML_MORE 2

template <bool PME, int MT>
KF_DEV int ml_solve3(const AnchorTable &A, const EpochT<PME, MT> &ep, unsigned mask, double (&p)[3],
                     double &sse_out, unsigned &iters, double *cov /* packed Sym<3> or null */,
                     double *sse_start = nullptr, unsigned iter_cap = 10000u, MlResume *rs = nullptr,
                     const Col *cyc_ref = nullptr /* EKF callers: arms the cycle detection (see below) */) {
    const int nvalid = __popc(mask);
    MlPass3 ps;
    double cost = 1e20, newCost = 1.0;
    unsigned iter = 0;
    bool first = true;
    if (rs && rs->iter) { // resume: the pass below recomputes newCost at p
        cost = rs->cost;
        iter = rs->iter;
        first = false;
    }
    for (;;) {
        ml_pass3<PME, MT>(A, ep, mask, nvalid, p, ps);
        if (first) {
            first = false;
            if (sse_start) *sse_start = ps.sse;
            if (nvalid < 4) { sse_out = ps.sse; return ML_FEW; }
            // scalar errorEstimation == 0: the reference divides gradient and Hessian by it, its solver
            // rejects the non-finite normal matrix (here the weight cancels, so say so explicitly)
            if (!PME && ep.e0 == 0.0) { sse_out = ps.sse; return ML_SINGULAR; }
        } else {
            newCost = ps.wcost;
        }
        if (!(rel_change_gt(cost, newCost) && iter < 10000u)) break;
        if (iter >= iter_cap) {
            rs->cost = cost;
            rs->iter = iter;
            return ML_MORE;
        }
        iter += 1;
        cost = newCost;
        double s[3];
        if (!solve_sym3(ps.H, ps.g, s)) { iters += iter; return ML_SINGULAR; }
        // newPos = solve(H, H pos - g)  ==  pos - H^-1 g
        p[0] -= s[0]; p[1] -= s[1]; p[2] -= s[2];
        if (cyc_ref) { // Brent's cycle detection, as in ml_solve3_ekf
            const Col &c = *cyc_ref;
            if ((iter & (iter - 1u)) == 0u) {
                c[0] = p[0]; c[1] = p[1]; c[2] = p[2];
            } else if (p[0] == c[0] && p[1] == c[1] && p[2] == c[2]) {
                const unsigned per = iter - (1u << (31 - __clz(iter)));
                iter = skip_whole_periods(iter, per);
            }
        }
    }
    iters += iter;
    sse_out = ps.sse;
    if (cov) return ml_cov3<PME, MT>(A, ep, mask, p, ps.sse, cov);
    return ML_OK;
}

// The same solver for the EKFs' inner ML (scalar errorEstimation, no covariance, no resume): its
// pass at the START point -- the predicted position, where the IEKF's first iteration also
// linearises -- additionally returns g and Gu = sum u u^T, which give that iteration's
// b = -g / R and G = Gu / R without another pass over the anchors (its cost is sse_start / R).
template <int MT>
KF_DEV double iekf_cost_only(const AnchorTable &A, const EpochT<false, MT> &ep, unsigned mask, double px, double py,
                             double pz);
#ifndef ML_EKF_COST_FIRST
#define ML_EKF_COST_FIRST 4u
#endif

// COSTFIRST: see below (the plain replay only: in the leave-one-out instantiation, whose code is far beyond the
// instruction cache anyway, the extra code measured 5 % slower)
template <int MT, bool COSTFIRST = false>
KF_DEV int ml_solve3_ekf(const AnchorTable &A, const EpochT<false, MT> &ep, unsigned mask, double (&p)[3],
                         double &sse_out, unsigned &iters, double &sse_start, double (&g_start)[3],
                         double (&Gu_start)[6], const Col &cyc_ref, unsigned long long *cnt = nullptr) {
    const int nvalid = __popc(mask);
    MlPass3 ps;
    ml_pass3<false, MT, true>(A, ep, mask, nvalid, p, ps, Gu_start);
    sse_start = ps.sse;
    sse_out = ps.sse;
    g_start[0] = ps.g[0]; g_start[1] = ps.g[1]; g_start[2] = ps.g[2];
    if (nvalid < 4) return ML_FEW;
    if (ep.e0 == 0.0) return ML_SINGULAR; // see ml_solve3
    double cost = 1e20, newCost = 1.0;
    unsigned iter = 0;
    while (rel_change_gt(cost, newCost) && iter < 10000u) {
        iter += 1;
        cost = newCost;
        double s[3];
        if (!solve_sym3(ps.H, ps.g, s)) { iters += iter; return ML_SINGULAR; }
        p[0] -= s[0]; p[1] -= s[1]; p[2] -= s[2];
        // from the fourth Newton iteration on the pass usually ends the solve: its cost alone first (the same sum of
        // squared residuals, bit for bit), the full pass when the stop test fails (measured: from the third iteration on
        // +0.3 %, from the fourth +1.6 %)
        if (COSTFIRST && MT > 0 && iter >= ML_EKF_COST_FIRST) {
            const double sse2 = iekf_cost_only<MT>(A, ep, mask, p[0], p[1], p[2]);
            const double wc2 = sse2 * fast_rcp(ep.e0);
            if (!(rel_change_gt(newCost, wc2) && iter < 10000u)) {
                ps.sse = sse2;
                break;
            }
        }
        ml_pass3<false, MT>(A, ep, mask, nvalid, p, ps);
        newCost = ps.wcost;
        // Brent's cycle detection (see CycleDetect) with the reference point in shared memory and the
        // iteration count as its clock: refreshed when iter is a power of two
        if ((iter & (iter - 1u)) == 0u) {
            cyc_ref[0] = p[0]; cyc_ref[1] = p[1]; cyc_ref[2] = p[2];
        } else if (p[0] == cyc_ref[0] && p[1] == cyc_ref[1] && p[2] == cyc_ref[2]) {
            const unsigned per = iter - (1u << (31 - __clz(iter)));
            iter = skip_whole_periods_counted(iter, per, cnt);
        }
    }
    if (cnt && iter >= 10000u) count_rare_event(cnt + CNT_ML_CAPPED);
    iters += iter;
    sse_out = ps.sse;
    return ML_OK;
}

struct MlPass2 {
    double sse;
    double g[2];
    double H[3]; // xx, xy, yy
};

// 2-D pass: distances are 3-D with z fixed, derivatives in x,y only (ML.cpp:74-95)
template <bool PME, int MT>
KF_DEV void ml_pass2(const AnchorTable &A, const EpochT<PME, MT> &ep, unsigned mask, int nvalid, double px,
                     double py, double pz, MlPass2 &o) {
    double sse = 0.0, g0 = 0.0, g1 = 0.0, h0 = 0.0, h1 = 0.0, h2 = 0.0, c1s = 0.0;
#pragma unroll(MT > 0 ? MT : 2)
    for (int i = 0; i < ep.m(); ++i) {
        const bool on = (mask >> i) & 1u;
        if (MT == 0 && !on) continue;
        const double dx = A.x[i] - px, dy = A.y[i] - py, dz = A.z[i] - pz;
        const double d2 = fma(dz, dz, fma(dy, dy, dx * dx));
        double invd = MT > 0 ? fast_rsqrt_masked(d2, on) : fast_rsqrt(d2);
        double r = ep.r(i);
        if (MT > 0) r = on ? r : 0.0;
        const double res = fma(-d2, invd, r);
        const double rid = r * invd;
        sse = fma(res, res, sse);
        if (PME) {
            const double w = fast_rcp(ep.e[i]);
            const double t = res * invd * w;
            g0 = fma(t, dx, g0); g1 = fma(t, dy, g1);
            c1s = fma(1.0 - rid, w, c1s);
            const double c2 = rid * invd * invd * w;
            const double cx = c2 * dx, cy = c2 * dy;
            h0 = fma(cx, dx, h0); h1 = fma(cx, dy, h1); h2 = fma(cy, dy, h2);
        } else {
            const double t = res * invd;
            g0 = fma(t, dx, g0); g1 = fma(t, dy, g1);
            c1s += rid;
            const double c2 = rid * (invd * invd);
            const double cx = c2 * dx, cy = c2 * dy;
            h0 = fma(cx, dx, h0); h1 = fma(cx, dy, h1); h2 = fma(cy, dy, h2);
        }
    }
    if (!PME) c1s = (double)nvalid - c1s;
    o.sse = sse;
    o.g[0] = g0; o.g[1] = g1;
    o.H[0] = h0 + c1s; o.H[1] = h1; o.H[2] = h2 + c1s;
}

// estimatePosition2D, ML.cpp:48-143.  z stays at its start value.  The damping
// `step` of the reference never takes effect: a rejected step leaves
// newCost == cost, so the while-test fails on the next evaluation (ML.cpp:109-116).
// B-1 (SURVEY App. B): the tentative cost is evaluated at z = start z (the evident intent);
// zero_tz = true evaluates it at z = 0 instead, which is what a build of the reference that
// zero-initialises ML.cpp:64's `tentativePos` computes (used to replay the reference's golden vectors).
template <bool PME, int MT>
KF_DEV double sse_at(const AnchorTable &A, const EpochT<PME, MT> &ep, unsigned mask, double px, double py, double pz) {
    double sse = 0.0;
    for (int i = 0; i < ep.m_slots; ++i) {
        if (!((mask >> i) & 1u)) continue;
        const double dx = A.x[i] - px, dy = A.y[i] - py, dz = A.z[i] - pz;
        const double d2 = fma(dz, dz, fma(dy, dy, dx * dx));
        const double res = fma(-d2, fast_rsqrt(d2), ep.z_at(i));
        sse = fma(res, res, sse);
    }
    return sse;
}

template <bool PME, int MT>
KF_DEV int ml_solve2(const AnchorTable &A, const EpochT<PME, MT> &ep, unsigned mask, double (&p)[3],
                     double &sse_out, unsigned &iters, double *cov /* xx, xy, yy or null */,
                     double *sse_start = nullptr, bool zero_tz = false) {
    const int nvalid = __popc(mask);
    MlPass2 ps, pt;
    double cost = 1e20, newCost = 0.0;
    double nx = p[0], ny = p[1];
    unsigned iter = 0;
    bool first = true;
    for (;;) {
        ml_pass2<PME, MT>(A, ep, mask, nvalid, nx, ny, p[2], pt);
        if (first) {
            first = false;
            ps = pt;
            newCost = pt.sse;
            if (sse_start) *sse_start = pt.sse;
            if (nvalid < 3) { sse_out = pt.sse; return ML_FEW; }
            if (!PME && ep.e0 == 0.0) { sse_out = pt.sse; return ML_SINGULAR; } // see ml_solve3
        } else {
            // only the generic (MT = 0) instantiations carry the test mode; the launchers route it there
            const double tc = (MT == 0 && zero_tz) ? sse_at<PME, MT>(A, ep, mask, nx, ny, 0.0) : pt.sse;
            if (tc > cost) break; // step /= 2; position kept; the while-test then fails
            newCost = tc;
            p[0] = nx; p[1] = ny;
            ps = pt;
        }
        if (!(rel_change_gt(cost, newCost) && iter < 10000u)) break;
        iter += 1;
        cost = newCost;
        double s0, s1;
        if (!solve_sym2(ps.H[0], ps.H[1], ps.H[2], ps.g[0], ps.g[1], s0, s1)) {
            iters += iter;
            return ML_SINGULAR;
        }
        nx = p[0] - s0; ny = p[1] - s1;
    }
    iters += iter;
    sse_out = ps.sse;
    if (cov) return ml_cov2<PME, MT>(A, ep, mask, p, ps.sse, cov);
    return ML_OK;
}

// estimatePositionIgnoreN's selection (ML.cpp:307-347): removes from `used` the `drop` rangings with
// the largest squared residual at `pos` -- the tail of the ascending std::sort order; ties keep the
// lower index (SURVEY App. B-11).
// near_tie (optional): set when the smallest dropped and the largest kept squared residual are within
// ML_TIE_MARGIN of each other (or not comparable) -- the decision then belongs to the exact-order solver.
template <bool PME, int MT>
KF_DEV unsigned drop_worst(const AnchorTable &A, const EpochT<PME, MT> &ep, unsigned used, const double (&pos)[3],
                           int drop, bool *near_tie = nullptr) {
    double worst = -1.0;
    int dcount = 0;
    for (; dcount < drop; ++dcount) {
        worst = -1.0;
        int wi = -1;
        for (int i = 0; i < ep.m_slots; ++i) {
            if (!((used >> i) & 1u)) continue;
            const double ex = A.x[i] - pos[0], ey = A.y[i] - pos[1], ez = A.z[i] - pos[2];
            const double d = sqrt(ex * ex + ey * ey + ez * ez);
            const double zi = ep.z_at(i);
            const double q = (d - zi) * (d - zi);
            if (q >= worst) { worst = q; wi = i; }
        }
        if (wi < 0) break; // all residuals NaN
        used &= ~(1u << wi);
    }
    if (near_tie && drop > 0) {
        // `worst` = the smallest dropped residual (each round removed the largest one left)
        double kept = -1.0;
        bool odd = dcount < drop;
        for (int i = 0; i < ep.m_slots; ++i) {
            if (!((used >> i) & 1u)) continue;
            const double ex = A.x[i] - pos[0], ey = A.y[i] - pos[1], ez = A.z[i] - pos[2];
            const double d = sqrt(ex * ex + ey * ey + ez * ez);
            const double zi = ep.z_at(i);
            const double q = (d - zi) * (d - zi);
            if (!(q == q)) odd = true;
            kept = fmax(kept, q);
        }
        *near_tie = odd || !(worst - kept > ML_TIE_MARGIN * worst);
    }
    return used;
}

// estimatePositionBestGroup's scan (ML.cpp:351-414): all C(n,k) subsets of the valid rangings in
// prev_permutation (= lexicographic) order, each solved from `start`; the subset with the smallest
// criterion wins, `<=` keeps the LAST minimum.  App. B-3: subset = measurements with mask true;
// B-4: 2-D criterion = cov(0,0)+cov(1,1); best_mode 1 = cov(2,2) (3-D only).  Returns the subset
// index (>= 0) and its mask / position / covariance / solver code; -1 when n < k.
template <bool PME, int MT>
KF_DEV int best_group(const AnchorTable &A, const EpochT<PME, MT> &ep, unsigned valid, bool use2d, int best_mode,
                      const double (&start)[3], unsigned &iters, double (&pos)[3], double (&cov)[6],
                      unsigned &used, int &rc, bool zero_tz = false) {
    const int k = use2d ? 3 : 4, n = __popc(valid);
    if (n < k) return -1;
    // on entry pos / cov hold the all-ranging estimate (ML.cpp:353-358); it is what remains when a
    // subset's solve fails -- the reference's solver then throws out of the scan, nothing is selected
    const double pos_all[3] = {pos[0], pos[1], pos[2]};
    double cov_all[6];
#pragma unroll
    for (int q = 0; q < 6; ++q) cov_all[q] = cov[q];
    unsigned char slot[32];
    int c = 0;
    for (int i = 0; i < ep.m_slots; ++i)
        if ((valid >> i) & 1u) slot[c++] = (unsigned char)i;
    double minErr = 0.0;
    int minIdx = -1, gi = 0;
    int a[4] = {0, 1, 2, 3};
    while (true) {
        unsigned gm = 0u;
        for (int j = 0; j < k; ++j) gm |= 1u << slot[a[j]];
        double gp[3] = {start[0], start[1], start[2]}, gc[6] = {0, 0, 0, 0, 0, 0}, gs;
        int grc;
        if (use2d) {
            double c2[3] = {0, 0, 0};
            grc = ml_solve2<PME, MT>(A, ep, gm, gp, gs, iters, c2, nullptr, zero_tz);
            gc[0] = c2[0]; gc[1] = c2[1]; gc[2] = c2[2];
        } else {
            grc = ml_solve3<PME, MT>(A, ep, gm, gp, gs, iters, gc);
        }
        double cur;
        if (use2d) cur = gc[0] + gc[2];
        else if (best_mode == 1) cur = gc[5];
        else cur = gc[0] + gc[2] + gc[5];
        if (grc != ML_OK) {
            pos[0] = pos_all[0]; pos[1] = pos_all[1]; pos[2] = pos_all[2];
#pragma unroll
            for (int q = 0; q < 6; ++q) cov[q] = cov_all[q];
            used = valid;
            rc = ML_SINGULAR;
            return -1;
        }
        if (minIdx == -1 || cur <= minErr) {
            minIdx = gi;
            minErr = cur;
            pos[0] = gp[0]; pos[1] = gp[1]; pos[2] = gp[2];
#pragma unroll
            for (int q = 0; q < 6; ++q) cov[q] = gc[q];
            used = gm;
            rc = grc;
        }
        ++gi;
        // next combination in lexicographic order
        int j = k - 1;
        while (j >= 0 && a[j] == n - k + j) --j;
        if (j < 0) break;
        ++a[j];
        for (int q = j + 1; q < k; ++q) a[q] = a[q - 1] + 1;
    }
    return minIdx;
}

// ---- information-form ranging pass of one IEKF iteration at the iterate p = x^- + dx:
//   c = sum eps_i^2 / R_i,  b = sum h_i y_i / R_i,  G = sum h_i h_i^T / R_i   (packed xx,xy,yy,xz,yz,zz)
// with h_i = (p - a_i)/d_i, eps_i = r_i - d_i, y_i = eps_i + h_i . dx  (= eps - J delta, delta = -dx)
// and R_i = max(sse, e_i).  With a scalar errorEstimation R is common: the sums are returned
// UNSCALED and the caller multiplies by 1/R once.  D = 3: all three components; D = 2: the
// rows only touch x,y (K8; z is the fixed tag height), G packed xx,xy,yy.
template <bool PME, int MT, int D>
KF_DEV void iekf_pass(const AnchorTable &A, const EpochT<PME, MT> &ep, unsigned mask, double sse, double px,
                      double py, double pz, const double (&dx)[3], double &c_out, double (&b)[3], double (&G)[6]) {
    double c = 0.0, b0 = 0.0, b1 = 0.0, b2 = 0.0;
    double G0 = 0.0, G1 = 0.0, G2 = 0.0, G3 = 0.0, G4 = 0.0, G5 = 0.0;
#pragma unroll(MT > 0 ? MT : 2)
    for (int i = 0; i < ep.m(); ++i) {
        const bool on = (mask >> i) & 1u;
        if (MT == 0 && !on) continue;
        const double ex = px - A.x[i], ey = py - A.y[i], ez = pz - A.z[i];
        const double d2 = fma(ez, ez, fma(ey, ey, ex * ex));
        double id = MT > 0 ? fast_rsqrt_masked(d2, on) : fast_rsqrt(d2);
        double r = ep.r(i);
        if (MT > 0) r = on ? r : 0.0;
        const double e = fma(-d2, id, r);
        const double h0 = ex * id, h1 = ey * id, h2 = D == 3 ? ez * id : 0.0;
        // b = sum h (eps + h . dx) / R = sum h eps / R + G dx: the second term is added after the loop
        const double y = e;
        if (PME) {
            const double iR = fast_rcp(fmax(sse, ep.e[i]));
            c = fma(e * e, iR, c);
            const double yr = y * iR;
            const double h0r = h0 * iR, h1r = h1 * iR;
            b0 = fma(h0, yr, b0); b1 = fma(h1, yr, b1);
            G0 = fma(h0r, h0, G0); G1 = fma(h0r, h1, G1); G2 = fma(h1r, h1, G2);
            if (D == 3) {
                b2 = fma(h2, yr, b2);
                G3 = fma(h0r, h2, G3); G4 = fma(h1r, h2, G4); G5 = fma(h2 * iR, h2, G5);
            }
        } else {
            c = fma(e, e, c);
            b0 = fma(h0, y, b0); b1 = fma(h1, y, b1);
            G0 = fma(h0, h0, G0); G1 = fma(h0, h1, G1); G2 = fma(h1, h1, G2);
            if (D == 3) {
                b2 = fma(h2, y, b2);
                G3 = fma(h0, h2, G3); G4 = fma(h1, h2, G4);
            }
        }
    }
    // unit rows: trace(sum h h^T) = number of rangings (a missing one has h = 0)
    if (!PME && D == 3) G5 = ((double)__popc(mask) - G0) - G2;
    c_out = c;
    if (D == 3) {
        b0 = fma(G0, dx[0], fma(G1, dx[1], fma(G3, dx[2], b0)));
        b1 = fma(G1, dx[0], fma(G2, dx[1], fma(G4, dx[2], b1)));
        b2 = fma(G3, dx[0], fma(G4, dx[1], fma(G5, dx[2], b2)));
    } else {
        b0 = fma(G0, dx[0], fma(G1, dx[1], b0));
        b1 = fma(G1, dx[0], fma(G2, dx[1], b1));
    }
    b[0] = b0; b[1] = b1; b[2] = b2;
    G[0] = G0; G[1] = G1; G[2] = G2; G[3] = G3; G[4] = G4; G[5] = G5;
}

// The cost of iekf_pass alone: sum of squared residuals at (px, py, pz), scalar errorEstimation, compile-time anchor
// count -- the same operations on the same values as iekf_pass's `c`, without the rows' b and G.  The IEKF of T6 meets its
// break test at the third evaluation for 99.95 % of the updates, so that evaluation first forms only the cost (14 instead
// of 25 FP64 instructions per ranging) and the full pass runs when the test fails.
template <int MT>
KF_DEV double iekf_cost_only(const AnchorTable &A, const EpochT<false, MT> &ep, unsigned mask, double px, double py,
                             double pz) {
    double c = 0.0;
#pragma unroll
    for (int i = 0; i < (MT > 0 ? MT : 1); ++i) {
        const bool on = (mask >> i) & 1u;
        const double ex = px - A.x[i], ey = py - A.y[i], ez = pz - A.z[i];
        const double d2 = fma(ez, ez, fma(ey, ey, ex * ex));
        const double id = fast_rsqrt_masked(d2, on);
        const double r = on ? ep.r(i) : 0.0;
        const double e = fma(-d2, id, r);
        c = fma(e, e, c);
    }
    return c;
}

// Solves one information-form IEKF gain step for 3-D ranging rows:
//   N = I + G A;  s = N^-1 b;  dx = A s (position part of B s);  M = N^-1 G;
//   returns w . dx with w = b - G dx
// A = position block of P^- (packed xx, yx, yy, zx, zy, zz), G packed the same way.
KF_DEV double info_gain3(const double (&a)[6], const double (&b)[3], const double (&G)[6], double (&dx)[3],
                         double (&M)[6], double (&s)[3]) {
    const double a00 = a[0], a10 = a[1], a11 = a[2], a20 = a[3], a21 = a[4], a22 = a[5];
    const double G0 = G[0], G1 = G[1], G2 = G[2], G3 = G[3], G4 = G[4], G5 = G[5];
    const double n00 = fma(G0, a00, fma(G1, a10, fma(G3, a20, 1.0)));
    const double n01 = fma(G0, a10, fma(G1, a11, G3 * a21));
    const double n02 = fma(G0, a20, fma(G1, a21, G3 * a22));
    const double n10 = fma(G1, a00, fma(G2, a10, G4 * a20));
    const double n11 = fma(G1, a10, fma(G2, a11, fma(G4, a21, 1.0)));
    const double n12 = fma(G1, a20, fma(G2, a21, G4 * a22));
    const double n20 = fma(G3, a00, fma(G4, a10, G5 * a20));
    const double n21 = fma(G3, a10, fma(G4, a11, G5 * a21));
    const double n22 = fma(G3, a20, fma(G4, a21, fma(G5, a22, 1.0)));
    const double c00 = fma(n11, n22, -n12 * n21), c01 = fma(n02, n21, -n01 * n22), c02 = fma(n01, n12, -n02 * n11);
    const double c10 = fma(n12, n20, -n10 * n22), c11 = fma(n00, n22, -n02 * n20), c12 = fma(n02, n10, -n00 * n12);
    const double c20 = fma(n10, n21, -n11 * n20), c21 = fma(n01, n20, -n00 * n21), c22 = fma(n00, n11, -n01 * n10);
    const double idet = fast_rcp(fma(n00, c00, fma(n01, c10, n02 * c20)));
    const double s0 = fma(c00, b[0], fma(c01, b[1], c02 * b[2])) * idet;
    const double s1 = fma(c10, b[0], fma(c11, b[1], c12 * b[2])) * idet;
    const double s2 = fma(c20, b[0], fma(c21, b[1], c22 * b[2])) * idet;
    s[0] = s0; s[1] = s1; s[2] = s2;
    dx[0] = fma(a00, s0, fma(a10, s1, a20 * s2));
    dx[1] = fma(a10, s0, fma(a11, s1, a21 * s2));
    dx[2] = fma(a20, s0, fma(a21, s1, a22 * s2));
    M[0] = fma(c00, G0, fma(c01, G1, c02 * G3)) * idet;
    M[1] = fma(c10, G0, fma(c11, G1, c12 * G3)) * idet;
    M[2] = fma(c10, G1, fma(c11, G2, c12 * G4)) * idet;
    M[3] = fma(c20, G0, fma(c21, G1, c22 * G3)) * idet;
    M[4] = fma(c20, G1, fma(c21, G2, c22 * G4)) * idet;
    M[5] = fma(c20, G3, fma(c21, G4, c22 * G5)) * idet;
    const double w0 = b[0] - fma(G0, dx[0], fma(G1, dx[1], G3 * dx[2]));
    const double w1 = b[1] - fma(G1, dx[0], fma(G2, dx[1], G4 * dx[2]));
    const double w2 = b[2] - fma(G3, dx[0], fma(G4, dx[1], G5 * dx[2]));
    return fma(w0, dx[0], fma(w1, dx[1], w2 * dx[2]));
}

// P^+ = P^- - B M B^T, B = P^-[:, 0:3]  (the reference's (I - K J) P^-), in place on the
// shared-memory column of the packed NS x NS matrix: only B is held in registers.
template <int NS>
KF_DEV void apply_cov_block3(const Col &Pm, const double (&M)[6]) {
    double B[NS][3];
#pragma unroll
    for (int i = 0; i < NS; ++i)
#pragma unroll
        for (int k = 0; k < 3; ++k) B[i][k] = (i >= k) ? Pm[i * (i + 1) / 2 + k] : Pm[k * (k + 1) / 2 + i];
#pragma unroll
    for (int i = 0; i < NS; ++i) {
        const double c0 = fma(B[i][0], M[0], fma(B[i][1], M[1], B[i][2] * M[3]));
        const double c1 = fma(B[i][0], M[1], fma(B[i][1], M[2], B[i][2] * M[4]));
        const double c2 = fma(B[i][0], M[3], fma(B[i][1], M[4], B[i][2] * M[5]));
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            const int k = i * (i + 1) / 2 + j;
            Pm[k] = fma(-c0, B[j][0], fma(-c1, B[j][1], fma(-c2, B[j][2], Pm[k])));
        }
    }
}

// ---- ranging rows of one IEKF gain step as ONE block update of a register-resident (P, dn):
// on entry P = P^- and dn = 0; on exit P = P^- - B M B^T and dn = B s with
//   A = P^-[0:D,0:D], B = P^-[:,0:D], N = I + G A, s = N^-1 b, M = N^-1 G
// (= the sequential rank-1 updates of all m ranging rows; push-through identity, see kfpos_t6.cuh).
// The remaining sensor rows (PX4Flow / IMU / magnetometer) are then applied sequentially to (P, dn).
template <int NS, int D>
KF_DEV void info_block(Sym<NS> &P, double (&dn)[NS], const double (&b)[3], const double (&G)[6]) {
    double s[3] = {0.0, 0.0, 0.0}, M[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    if (D == 2) {
        const double a00 = P.get(0, 0), a10 = P.get(1, 0), a11 = P.get(1, 1);
        const double n00 = fma(G[0], a00, fma(G[1], a10, 1.0)), n01 = fma(G[0], a10, G[1] * a11);
        const double n10 = fma(G[1], a00, G[2] * a10), n11 = fma(G[1], a10, fma(G[2], a11, 1.0));
        const double idet = fast_rcp(fma(n00, n11, -n01 * n10));
        s[0] = fma(n11, b[0], -n01 * b[1]) * idet;
        s[1] = fma(n00, b[1], -n10 * b[0]) * idet;
        M[0] = fma(n11, G[0], -n01 * G[1]) * idet;
        M[1] = fma(n11, G[1], -n01 * G[2]) * idet;
        M[2] = fma(n00, G[2], -n10 * G[1]) * idet;
    } else {
        const double a00 = P.get(0, 0), a10 = P.get(1, 0), a11 = P.get(1, 1), a20 = P.get(2, 0), a21 = P.get(2, 1),
                     a22 = P.get(2, 2);
        const double G0 = G[0], G1 = G[1], G2 = G[2], G3 = G[3], G4 = G[4], G5 = G[5];
        const double n00 = fma(G0, a00, fma(G1, a10, fma(G3, a20, 1.0)));
        const double n01 = fma(G0, a10, fma(G1, a11, G3 * a21));
        const double n02 = fma(G0, a20, fma(G1, a21, G3 * a22));
        const double n10 = fma(G1, a00, fma(G2, a10, G4 * a20));
        const double n11 = fma(G1, a10, fma(G2, a11, fma(G4, a21, 1.0)));
        const double n12 = fma(G1, a20, fma(G2, a21, G4 * a22));
        const double n20 = fma(G3, a00, fma(G4, a10, G5 * a20));
        const double n21 = fma(G3, a10, fma(G4, a11, G5 * a21));
        const double n22 = fma(G3, a20, fma(G4, a21, fma(G5, a22, 1.0)));
        const double c00 = fma(n11, n22, -n12 * n21), c01 = fma(n02, n21, -n01 * n22), c02 = fma(n01, n12, -n02 * n11);
        const double c10 = fma(n12, n20, -n10 * n22), c11 = fma(n00, n22, -n02 * n20), c12 = fma(n02, n10, -n00 * n12);
        const double c20 = fma(n10, n21, -n11 * n20), c21 = fma(n01, n20, -n00 * n21), c22 = fma(n00, n11, -n01 * n10);
        const double idet = fast_rcp(fma(n00, c00, fma(n01, c10, n02 * c20)));
        s[0] = fma(c00, b[0], fma(c01, b[1], c02 * b[2])) * idet;
        s[1] = fma(c10, b[0], fma(c11, b[1], c12 * b[2])) * idet;
        s[2] = fma(c20, b[0], fma(c21, b[1], c22 * b[2])) * idet;
        M[0] = fma(c00, G0, fma(c01, G1, c02 * G3)) * idet;
        M[1] = fma(c10, G0, fma(c11, G1, c12 * G3)) * idet;
        M[2] = fma(c10, G1, fma(c11, G2, c12 * G4)) * idet;
        M[3] = fma(c20, G0, fma(c21, G1, c22 * G3)) * idet;
        M[4] = fma(c20, G1, fma(c21, G2, c22 * G4)) * idet;
        M[5] = fma(c20, G3, fma(c21, G4, c22 * G5)) * idet;
    }
    double B[NS][D];
#pragma unroll
    for (int i = 0; i < NS; ++i)
#pragma unroll
        for (int k = 0; k < D; ++k) B[i][k] = P.get(i, k);
#pragma unroll
    for (int i = 0; i < NS; ++i) {
        double c0, c1, c2 = 0.0;
        if (D == 2) {
            dn[i] = fma(B[i][0], s[0], B[i][1] * s[1]);
            c0 = fma(B[i][0], M[0], B[i][1] * M[1]);
            c1 = fma(B[i][0], M[1], B[i][1] * M[2]);
        } else {
            dn[i] = fma(B[i][0], s[0], fma(B[i][1], s[1], B[i][D - 1] * s[2]));
            c0 = fma(B[i][0], M[0], fma(B[i][1], M[1], B[i][D - 1] * M[3]));
            c1 = fma(B[i][0], M[1], fma(B[i][1], M[2], B[i][D - 1] * M[4]));
            c2 = fma(B[i][0], M[3], fma(B[i][1], M[4], B[i][D - 1] * M[5]));
        }
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            double v = fma(-c0, B[j][0], fma(-c1, B[j][1], P.get(i, j)));
            if (D == 3) v = fma(-c2, B[j][D - 1], v);
            P.at(i, j) = v;
        }
    }
}

// ---- asynchronous epoch loads (LDGSTS / cp.async): the rangings of the NEXT
// epoch stream from HBM straight into a shared-memory landing zone while the current
// epoch is being processed, so no warp ever waits on DRAM and no registers are
// spent on staging.  ranges: SoA with the filter index fastest; `base` = element
// index of slot 0 for this filter, `N` = element stride between slots.
KF_DEV void cp_async_4(void *dst, const void *src) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s), "l"(src) : "memory");
}
KF_DEV void cp_async_8(void *dst, const void *src) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(src) : "memory");
}
KF_DEV void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
KF_DEV void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// Landing zone: 32-bit words for the mm wire formats (half the shared memory of a
// double column), doubles for the f64 format.  Element i of thread t lives at word/double
// index i * stride + t of the region (conflict-free either way).
struct RawCol {
    void *p;
    int stride;
    KF_DEV unsigned *w(int i) const { return reinterpret_cast<unsigned *>(p) + i * stride; }
    KF_DEV double *d(int i) const { return reinterpret_cast<double *>(p) + i * stride; }
};
KF_DEV RawCol make_raw(double *region, int fmt, int tid, int block) {
    RawCol r;
    r.p = fmt == 0 ? static_cast<void *>(region + tid) : static_cast<void *>(reinterpret_cast<unsigned *>(region) + tid);
    r.stride = block;
    return r;
}
// The same landing zone INSIDE a thread's private double column (K8 / T9, where the zone is
// shared with the f64 sensor payloads of other event kinds and warps drift apart in the
// schedule): 32-bit element i is half (i & 1) of the thread's double i / 2.
struct RawColPriv {
    Col c;
    KF_DEV unsigned *w(int i) const { return reinterpret_cast<unsigned *>(&c[i >> 1]) + (i & 1); }
    KF_DEV double *d(int i) const { return &c[i]; }
};
// doubles of shared memory per thread a landing zone of `rows` elements needs
__host__ __device__ inline int raw_rows(int fmt, int rows) { return fmt == 0 ? rows : (rows + 1) / 2; }

template <class RAW>
KF_DEV void prefetch_epoch(const RAW &raw, int m, const void *ranges, int fmt, int64_t base, int64_t N) {
#pragma unroll 4
    for (int i = 0; i < m; ++i) {
        const int64_t idx = base + (int64_t)i * N;
        if (fmt == 0) cp_async_8(raw.d(i), reinterpret_cast<const double *>(ranges) + idx);
        else if (fmt == 1) cp_async_4(raw.w(i), reinterpret_cast<const int32_t *>(ranges) + idx);
        else // uint16: fetch the aligned 32-bit word that holds the element
            cp_async_4(raw.w(i), reinterpret_cast<const void *>(
                                     reinterpret_cast<uintptr_t>(reinterpret_cast<const uint16_t *>(ranges) + idx) & ~(uintptr_t)3));
    }
    cp_async_commit();
}

// landing zone -> metres + valid mask: keep rangings[i] > 0 (TOA.cpp:48-57, ML.cpp:478)
// WIRE_MASK: the mask of the millimetre formats from the integer (mm > 0 exactly when mm / 1000 > 0), an integer compare
// instead of an FP64 one per ranging (the T6 replay)
template <bool PME, int MT, class RAW, bool WIRE_MASK = false>
KF_DEV void convert_epoch(EpochT<PME, MT> &ep, const RAW &raw, const void *ranges, int fmt, const double *err,
                          int64_t base, int64_t N) {
    unsigned valid = 0u;
#pragma unroll(MT > 0 ? MT : 1)
    for (int i = 0; i < ep.m(); ++i) {
        double r;
        bool on;
        if (fmt == 0) {
            r = *raw.d(i);
            on = r > 0;
        } else {
            const unsigned w = *raw.w(i);
            if (fmt == 1) {
                r = mm_to_m((double)(int)w);
                on = (int)w > 0;
            } else {
                const uintptr_t a = reinterpret_cast<uintptr_t>(reinterpret_cast<const uint16_t *>(ranges) + base + (int64_t)i * N);
                const unsigned v = (a & 2) ? (w >> 16) : (w & 0xffffu);
                r = mm_to_m((double)v);
                on = v != 0u;
            }
        }
        if (MT > 0) ep.zr[i] = r;
        else ep.z[i] = r;
        if (WIRE_MASK ? on : r > 0) valid |= 1u << i;
        if (PME) ep.e[i] = __ldg(err + base + (int64_t)i * N);
    }
    ep.valid = valid;
}

} // namespace kfpos
