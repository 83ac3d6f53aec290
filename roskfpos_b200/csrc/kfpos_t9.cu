// kfpos_t9.cu -- KalmanFilterTOAIMU (9-state constant-acceleration iterated EKF on
// rangings + 3-axis accelerometer), persistent event-stream kernel, one thread per
// filter.  Reference: algorithms/KalmanFilterTOAIMU.cpp.  State [p(3), v(3), a(3)].
//
// The ranging path follows the reference exactly (TOAIMU.cpp:242-340).  The IMU rows
// are the RESTATEMENT of SURVEY App. B-5: the reference reserves 9 rows for 3 values,
// writes jacobian(row, 9) on a 9-column matrix (std::logic_error on the first IMU
// sample) and uses diag(a) as dh/da; here: 3 rows, h = a, J = I3 on the acceleration
// block, R = the 3x3 covarianceAcceleration.
#include "kfpos_k8.cuh" // sym_add_row
#include "kfpos_kernels.cuh"

namespace kfpos {

constexpr int T9_BLOCK = 128;
#ifndef T9_LEAN_MINB
#define T9_LEAN_MINB 3
#endif

// shared-memory rows (doubles) per thread: P^- (45), landing zone (rangings or 3 accelerations),
// [metres column when MT == 0], [errorEstimation column]
__host__ __device__ inline int t9_land_rows(int m, int fmt) { return raw_rows(fmt, m) > 3 ? raw_rows(fmt, m) : 3; }
__host__ __device__ inline int t9_smem_rows(int m, int fmt, bool pme, bool in_regs) {
    return 45 + 3 + t9_land_rows(m, fmt) + (in_regs ? 0 : m) + (pme ? m : 0); // + cycle-detector reference point
}

// P^- = F P F^T + Q (TOAIMU.cpp:392-421)
KF_DEV void t9_predict_cov(Sym<9> &P, double t, double jolt) {
    const double h = -0.5 * t * t;
#pragma unroll
    for (int ax = 0; ax < 3; ++ax) {
        sym_add_row<9>(P, 3 + ax, 6 + ax, t);
        sym_add_row<9>(P, ax, 6 + ax, h);
        sym_add_row<9>(P, ax, 3 + ax, t);
    }
    const double t3 = t * t * t / 6, t2 = t * t / 2;
    const double u[3] = {t3, t2, t};
#pragma unroll
    for (int ax = 0; ax < 3; ++ax)
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b <= a; ++b) P.at(ax + 3 * a, ax + 3 * b) += jolt * u[b] * u[a];
}

// 3-row block update on the acceleration block (J = [0 0 I3]), S = P_aa + R packed symmetric
KF_DEV bool accel_block_update(Sym<9> &P, double (&dn)[9], const double (&y)[3], const double (&R)[6]) {
    double S[6], Si[6];
    S[0] = P.get(6, 6) + R[0]; S[1] = P.get(7, 6) + R[1]; S[2] = P.get(7, 7) + R[2];
    S[3] = P.get(8, 6) + R[3]; S[4] = P.get(8, 7) + R[4]; S[5] = P.get(8, 8) + R[5];
    if (!inv_sym3(S, Si)) return false;
    const double n0 = y[0] - dn[6], n1 = y[1] - dn[7], n2 = y[2] - dn[8];
    // g = S^-1 nu
    const double g0 = Si[0] * n0 + Si[1] * n1 + Si[3] * n2;
    const double g1 = Si[1] * n0 + Si[2] * n1 + Si[4] * n2;
    const double g2 = Si[3] * n0 + Si[4] * n1 + Si[5] * n2;
    double pa[9][3];
#pragma unroll
    for (int i = 0; i < 9; ++i) {
        pa[i][0] = P.get(i, 6); pa[i][1] = P.get(i, 7); pa[i][2] = P.get(i, 8);
    }
#pragma unroll
    for (int i = 0; i < 9; ++i) dn[i] = fma(pa[i][0], g0, fma(pa[i][1], g1, fma(pa[i][2], g2, dn[i])));
#pragma unroll
    for (int i = 0; i < 9; ++i) {
        const double k0 = pa[i][0] * Si[0] + pa[i][1] * Si[1] + pa[i][2] * Si[3];
        const double k1 = pa[i][0] * Si[1] + pa[i][1] * Si[2] + pa[i][2] * Si[4];
        const double k2 = pa[i][0] * Si[3] + pa[i][1] * Si[4] + pa[i][2] * Si[5];
#pragma unroll
        for (int j = 0; j <= i; ++j)
            P.at(i, j) = fma(-k0, pa[j][0], fma(-k1, pa[j][1], fma(-k2, pa[j][2], P.at(i, j))));
    }
    return true;
}

// kalmanStep3D (TOAIMU.cpp:242-340).  Pm: P^- (shared-memory column, read only); dx: out = x - x^-.
// Ranging rows: information form (kfpos_solve.cuh).  Without accelerometer rows the result is
// FACTORED like T6's: P = P^- - B M B^T with M returned (Pw untouched, return value 1); with them
// the ranging block is applied to a register copy Pw per gain step, followed by one 3x3 block
// update for the accelerometer rows, and Pw = (I - K J) P^- is returned (return value 0).
template <bool PME, int MT, bool IMU>
KF_DEV int t9_update(const AnchorTable &A, const EpochT<PME, MT> &ep, bool has_r, unsigned used, bool has_imu, const double (&za)[3],
                     const double (&Ra)[6], const double (&xp)[9], const Col &Pm, Sym<9> &Pw, double (&dx)[9],
                     double (&M)[6], StepStats &st, unsigned wmask, const Col &cyc) {
    const unsigned mask = has_r ? used : 0u; // used = ep.valid, or the EKF-side variant's selection
    double sse = -1.0;
    int rc = ML_OK;
    if (has_r) { // TOAIMU.cpp:268-270 (no NaN guard in this class)
        double pml[3] = {xp[0], xp[1], xp[2]};
        rc = ml_solve3<PME, MT>(A, ep, mask, pml, sse, st.ml_iters, nullptr, nullptr, 10000u, nullptr, &cyc);
        if (mask == 0u) sse = -1.0;
        // has_r is a property of the event, common to the batch: every lane of wmask is here
        if (wmask) __syncwarp(wmask);
    }
    if (rc == ML_FEW) st.status |= 2u;
    if (rc == ML_SINGULAR) return ML_SINGULAR;
    const double invR0 = mask ? fast_rcp(fmax(sse, ep.e0)) : 0.0;
    double Rai[6] = {0, 0, 0, 0, 0, 0};
    if (has_imu && !inv_sym3(Ra, Rai)) return ML_SINGULAR; // arma::inv(observationCovariance) would throw

#pragma unroll
    for (int k = 0; k < 9; ++k) dx[k] = 0.0;
#pragma unroll
    for (int k = 0; k < 6; ++k) M[k] = 0.0;
    double cost = 1e20, prior = 0.0;
    bool broke = false;
    if (!IMU || !has_imu) { // ---- ranging rows only: factored form, nothing but 3-vectors and 3x3 matrices in flight
        double a[6], s[3] = {0.0, 0.0, 0.0};
#pragma unroll
        for (int k = 0; k < 6; ++k) a[k] = Pm[k];
        double dxp[3] = {0.0, 0.0, 0.0};
        for (int iter = 0; iter < 20; ++iter) {
            double c = 0.0, b[3] = {0.0, 0.0, 0.0}, G[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
            if (mask) {
                iekf_pass<PME, MT, 3>(A, ep, mask, sse, xp[0] + dxp[0], xp[1] + dxp[1], xp[2] + dxp[2], dxp, c, b, G);
                if (!PME) c *= invR0;
            }
            const double newCost = c + prior;
            st.cost_evals += 1;
            if (rel_change_lt(cost, newCost, 1e-4)) { broke = true; break; }
            cost = newCost;
            st.gain_evals += 1;
            if (!PME) {
#pragma unroll
                for (int k = 0; k < 3; ++k) b[k] *= invR0;
#pragma unroll
                for (int k = 0; k < 6; ++k) G[k] *= invR0;
            }
            prior = info_gain3(a, b, G, dxp, M, s);
        }
        if (!broke) st.status |= 32u;
        // dx = B s over all nine states (velocity is persisted: TOAIMU.cpp:189-191)
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            const double bi0 = Pm[i * (i + 1) / 2 + 0];
            const double bi1 = i >= 1 ? Pm[i * (i + 1) / 2 + 1] : Pm[1];
            const double bi2 = i >= 2 ? Pm[i * (i + 1) / 2 + 2] : Pm[3 + i];
            dx[i] = fma(bi0, s[0], fma(bi1, s[1], bi2 * s[2]));
        }
        return 1;
    }
    if (!IMU) return 1; // (unreachable: the lean kernel never has accelerometer rows)
    for (int iter = 0; iter < 20; ++iter) {
        double c = 0.0, b[3] = {0.0, 0.0, 0.0}, G[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        if (mask) {
            const double dx3[3] = {dx[0], dx[1], dx[2]};
            iekf_pass<PME, MT, 3>(A, ep, mask, sse, xp[0] + dx[0], xp[1] + dx[1], xp[2] + dx[2], dx3, c, b, G);
            if (!PME) c *= invR0;
        }
        double ea[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) ea[k] = za[k] - (xp[6 + k] + dx[6 + k]);
        c += ea[0] * (Rai[0] * ea[0] + Rai[1] * ea[1] + Rai[3] * ea[2]) +
             ea[1] * (Rai[1] * ea[0] + Rai[2] * ea[1] + Rai[4] * ea[2]) +
             ea[2] * (Rai[3] * ea[0] + Rai[4] * ea[1] + Rai[5] * ea[2]);
        const double newCost = c + prior;
        st.cost_evals += 1;
        if (rel_change_lt(cost, newCost, 1e-4)) { broke = true; break; }
        cost = newCost;

        st.gain_evals += 1;
#pragma unroll
        for (int k = 0; k < Sym<9>::SZ; ++k) Pw.a[k] = Pm[k];
        double dn[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        if (mask) {
            if (!PME) {
#pragma unroll
                for (int k = 0; k < 3; ++k) b[k] *= invR0;
#pragma unroll
                for (int k = 0; k < 6; ++k) G[k] *= invR0;
            }
            info_block<9, 3>(Pw, dn, b, G);
        }
        // y_a = eps_a - J delta = eps_a + dx_a
        const double ya[3] = {ea[0] + dx[6], ea[1] + dx[7], ea[2] + dx[8]};
        if (!accel_block_update(Pw, dn, ya, Ra)) return ML_SINGULAR;
        const double w0 = b[0] - (G[0] * dn[0] + G[1] * dn[1] + G[3] * dn[2]);
        const double w1 = b[1] - (G[1] * dn[0] + G[2] * dn[1] + G[4] * dn[2]);
        const double w2 = b[2] - (G[3] * dn[0] + G[4] * dn[1] + G[5] * dn[2]);
        prior = w0 * dn[0] + w1 * dn[1] + w2 * dn[2];
        const double r0 = ya[0] - dn[6], r1 = ya[1] - dn[7], r2 = ya[2] - dn[8];
        prior += dn[6] * (Rai[0] * r0 + Rai[1] * r1 + Rai[3] * r2) +
                 dn[7] * (Rai[1] * r0 + Rai[2] * r1 + Rai[4] * r2) +
                 dn[8] * (Rai[3] * r0 + Rai[4] * r1 + Rai[5] * r2);
#pragma unroll
        for (int k = 0; k < 9; ++k) dx[k] = dn[k];
    }
    if (!broke) st.status |= 32u;
    return 0;
}

// IMU = false: the lean variant for schedules without accelerometer samples (nothing latched, no
// IMU event): no register copy of the 9x9 covariance anywhere, 4 blocks per SM like T6.
// SEL: the EKF-side NLOS variants (see kfpos_t6.cu), 3-D selection from the predicted position.
// ES: per-epoch statistics at every TOA event (see kfpos_t6.cu / kfpos_k8.cu), NEES of the 3x3 position block.
// EH (only with ES): the per-epoch error histogram, binned beside epoch_stats_row (epoch_hist_flush).
template <bool PME, int MT, bool IMU, bool SEL = false, bool ES = false, bool EH = false>
__global__ void __launch_bounds__(T9_BLOCK, IMU ? 2 : T9_LEAN_MINB) t9_replay_kernel(const __grid_constant__ T9Params p) {
    extern __shared__ double smem[];
    const int64_t f = (int64_t)blockIdx.x * T9_BLOCK + threadIdx.x;
    const bool active = f < p.N;
    const unsigned wmask = __ballot_sync(0xffffffffu, active);
    StepStats st = {0u, 0u, 0u, 0u};
    unsigned n_updates = 0, n_bad = 0;
    double errv[4] = {0.0, 0.0, 0.0, 0.0}; // error terms of the final state (fused statistics)
    if (active) {
        const int64_t N = p.N;
        const int m = MT > 0 ? MT : p.rs.m_slots;
        double *col = smem + threadIdx.x;
        int row = 0;
        auto take = [&](int rows) {
            Col c = {col + (size_t)row * T9_BLOCK, T9_BLOCK};
            row += rows;
            return c;
        };
        const Col Pm = take(45);
        const Col cyc = take(3);
        const Col land = take(t9_land_rows(m, p.rs.fmt));
        const RawColPriv raw = {land}; // rangings land in the same private column
        EpochT<PME, MT> ep;
        ep.z = MT > 0 ? Pm : take(m);
        ep.e = PME ? take(m) : Pm;
        ep.e0 = p.rs.err_scalar;
        ep.m_slots = m;
        ep.valid = 0u;

        double pos[3], vel[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            pos[k] = p.x[(int64_t)k * N + f];
            vel[k] = p.x[(int64_t)(3 + k) * N + f];
        }
#pragma unroll
        for (int k = 0; k < Sym<9>::SZ; ++k) Pm[k] = p.P[(int64_t)k * N + f];
        unsigned has = (unsigned)p.has[f];
        unsigned status_or = 0;
        double za[3] = {p.latch[0 * N + f], p.latch[1 * N + f], p.latch[2 * N + f]}; // latched acceleration
        double Ra[6]; // packed symmetric part of the latched 3x3 covariance
        bool asym = false;
        {
            const double *c = p.latch_u;
            Ra[0] = c[0]; Ra[1] = 0.5 * (c[1] + c[3]); Ra[2] = c[4];
            Ra[3] = 0.5 * (c[2] + c[6]); Ra[4] = 0.5 * (c[5] + c[7]); Ra[5] = c[8];
        }
        int n_toa = 0;
        const Col es = {col + (size_t)(ES ? t9_smem_rows(m, p.rs.fmt, PME, MT > 0) : 0) * T9_BLOCK, T9_BLOCK};
        double *const es_out = ES ? p.escratch + (f >> 5) * ES_W : nullptr;
        bool es_pending = false; // the row n_toa - 1 still has to be summed (common to the warp)
        auto prefetch = [&](const EventDesc &ev) {
            if (ev.kind == EV_TOA) {
                prefetch_epoch(raw, m, p.rs.ranges, p.rs.fmt, ev.offset * N + f, N);
            } else {
                for (int i = 0; i < 3; ++i) cp_async_8(&land[i], p.sensors + (ev.offset + i) * N + f);
                cp_async_commit();
            }
        };
        if (p.n_events > 0) prefetch(p.events[0]);
        for (int e = 0; e < p.n_events; ++e) {
            if (ES && es_pending) {
                es_pending = epoch_stats_row(es, wmask, es_out, n_toa - 1, p.n_warps);
                if (EH) epoch_hist_flush(es, wmask, p.ehist + (int64_t)(n_toa - 1) * p.ebins, p.eedges, p.equantity);
            }
            const EventDesc ev = p.events[e];
            double dt = ev.dt;
            if (SEL && p.dt_f) { // ragged replay: every filter has its own time steps
                dt = p.dt_f[(int64_t)e * N + f];
                if (dt < 0.0) { // this filter has no such event
                    cp_async_wait_all();
                    if (e + 1 < p.n_events) prefetch(p.events[e + 1]);
                    if (ev.kind == EV_TOA) { // its trajectory row repeats the current position
                        if (p.traj) {
#pragma unroll
                            for (int k = 0; k < 3; ++k) p.traj[((int64_t)n_toa * 3 + k) * N + f] = pos[k];
                        }
                        if (ES) {
                            epoch_terms_zero(es);
                            es_pending = true;
                        }
                        ++n_toa;
                    }
                    continue;
                }
            }
            if (SEL && p.ml_init && (isnan(pos[0]) || isnan(pos[1]))) {
                // ---- the constructor without initialPosition (TOAIMU.cpp:118-162): the sample is latched, an
                // epoch with rangings initialises the position from the 3-D ML estimate started at (1, 1, 4)
                // and the 2x2 x-y block of the all-zero covariance from its covariance; no predict, no update
                cp_async_wait_all();
                st.status = 256u;
                if (ev.kind == EV_TOA) {
                    convert_epoch<PME, MT>(ep, raw, p.rs.ranges, p.rs.fmt, p.rs.err, ev.offset * N + f, N);
                    if (e + 1 < p.n_events) prefetch(p.events[e + 1]);
                    double p0[3] = {1.0, 1.0, 4.0}, sse0, c0[6] = {0, 0, 0, 0, 0, 0};
                    const int irc = ml_solve3<PME, MT>(p.anchors, ep, ep.valid, p0, sse0, st.ml_iters, c0);
                    if (irc == ML_SINGULAR) {
                        st.status |= 4u; // the solver throws before mPosition is assigned
                    } else {
                        pos[0] = p0[0]; pos[1] = p0[1]; pos[2] = p0[2];
                        if (irc == ML_FEW) st.status |= 2u; // empty covariance matrix: (0,0) throws (:133)
                        else { Pm[0] = c0[0]; Pm[1] = c0[1]; Pm[2] = c0[2]; }
                    }
                    if (p.traj) {
#pragma unroll
                        for (int k = 0; k < 3; ++k) p.traj[((int64_t)n_toa * 3 + k) * N + f] = pos[k];
                    }
                    if (ES) {
                        const double *tr = p.etruth + (int64_t)n_toa * 3 * N + f;
                        epoch_terms<3>(pos[0] - tr[0], pos[1] - tr[N], pos[2] - tr[2 * N], Pm[0], Pm[1], Pm[2], Pm[3], Pm[4], Pm[5],
                                       st.status != 0u, es);
                        es_pending = true;
                    }
                    ++n_toa;
                } else {
                    za[0] = land[0]; za[1] = land[1]; za[2] = land[2];
                    Ra[0] = ev.aux[0]; Ra[1] = 0.5 * (ev.aux[1] + ev.aux[3]); Ra[2] = ev.aux[4];
                    Ra[3] = 0.5 * (ev.aux[2] + ev.aux[6]); Ra[4] = 0.5 * (ev.aux[5] + ev.aux[7]); Ra[5] = ev.aux[8];
                    asym = ev.aux[1] != ev.aux[3] || ev.aux[2] != ev.aux[6] || ev.aux[5] != ev.aux[7];
                    has |= 2u;
                    if (e + 1 < p.n_events) prefetch(p.events[e + 1]);
                }
                if (st.status & ~(32u | 64u | 256u)) n_bad += 1;
                status_or |= st.status;
                continue;
            }
            // ---- predict (TOAIMU.cpp:165-180): a = 0 at the start of every step.  Done before the
            // event's payload is unpacked so that the epoch's ranges are not live across it.
            Sym<9> Pw;
#pragma unroll
            for (int k = 0; k < Sym<9>::SZ; ++k) Pw.a[k] = Pm[k];
            t9_predict_cov(Pw, dt, p.jolt);
#pragma unroll
            for (int k = 0; k < Sym<9>::SZ; ++k) Pm[k] = Pw.a[k];
            cp_async_wait_all();
            st.status = 0u;
            bool has_r = false, has_imu = false;
            if (ev.kind == EV_TOA) { // newTOAMeasurement (TOAIMU.cpp:49-73): rangings + latched IMU
                convert_epoch<PME, MT>(ep, raw, p.rs.ranges, p.rs.fmt, p.rs.err, ev.offset * N + f, N);
                has_r = true;
                has_imu = (has >> 1) & 1u;
            } else { // newIMUMeasurement (TOAIMU.cpp:76-92)
                za[0] = land[0]; za[1] = land[1]; za[2] = land[2];
                Ra[0] = ev.aux[0]; Ra[1] = 0.5 * (ev.aux[1] + ev.aux[3]); Ra[2] = ev.aux[4];
                Ra[3] = 0.5 * (ev.aux[2] + ev.aux[6]); Ra[4] = 0.5 * (ev.aux[5] + ev.aux[7]); Ra[5] = ev.aux[8];
                asym = ev.aux[1] != ev.aux[3] || ev.aux[2] != ev.aux[6] || ev.aux[5] != ev.aux[7];
                has |= 2u;
                has_imu = true;
            }
            if (e + 1 < p.n_events) prefetch(p.events[e + 1]);
            if (has_imu && asym) st.status |= 64u;
            const double xp[9] = {pos[0] + dt * vel[0], pos[1] + dt * vel[1], pos[2] + dt * vel[2],
                                  vel[0], vel[1], vel[2], 0.0, 0.0, 0.0};
            if (has_r && ep.valid == 0u) st.status |= 1u;
            double dx[9], M[6];
            unsigned used = ep.valid;
            if (SEL && has_r) {
                const int n = __popc(ep.valid);
                const double start[3] = {xp[0], xp[1], xp[2]};
                double p0[3] = {xp[0], xp[1], xp[2]}, sse0, cov0[6];
                if (p.variant == 1 && n > 0) {
                    if (ml_solve3<PME, MT>(p.anchors, ep, ep.valid, p0, sse0, st.ml_iters, nullptr) == ML_OK) {
                        const int drop = min(n - 4, p.n_ignore);
                        used = drop_worst<PME, MT>(p.anchors, ep, used, p0, drop < 0 ? 0 : drop);
                    }
                } else if (p.variant == 2 && n >= 4) {
                    int grc;
                    // the all-ranging solve; a failed solve (there or in a subset) selects nothing
                    if (ml_solve3<PME, MT>(p.anchors, ep, ep.valid, p0, sse0, st.ml_iters, cov0) != ML_SINGULAR)
                        best_group<PME, MT>(p.anchors, ep, ep.valid, false, p.best_mode, start, st.ml_iters, p0, cov0, used, grc);
                }
            }
            const int rc = t9_update<PME, MT, IMU>(p.anchors, ep, has_r, used, IMU && has_imu, za, Ra, xp, Pm, Pw, dx, M, st,
                                                   SEL ? 0u : wmask, cyc);
            if (!SEL) __syncwarp(wmask); // the IEKF trip count differs per lane
            if (rc >= 0) {
#pragma unroll
                for (int k = 0; k < 3; ++k) { // velocity and position kept, acceleration dropped (:189-194)
                    pos[k] = xp[k] + dx[k];
                    vel[k] = xp[3 + k] + dx[3 + k];
                }
                if (rc == 1) {
                    apply_cov_block3<9>(Pm, M);
                } else {
#pragma unroll
                    for (int k = 0; k < Sym<9>::SZ; ++k) Pm[k] = Pw.a[k];
                }
                bool fin = true;
#pragma unroll
                for (int k = 0; k < 3; ++k) fin = fin && isfinite(pos[k]) && isfinite(vel[k]);
                if (!fin) st.status |= 8u;
            } else {
                st.status |= 4u;
            }
            n_updates += 1;
            if (st.status & ~(32u | 64u)) n_bad += 1;
            status_or |= st.status;
            if (ev.kind == EV_TOA) {
                if (p.traj) {
#pragma unroll
                    for (int k = 0; k < 3; ++k) p.traj[((int64_t)n_toa * 3 + k) * N + f] = pos[k];
                }
                if (ES) {
                    const double *tr = p.etruth + (int64_t)n_toa * 3 * N + f;
                    epoch_terms<3>(pos[0] - tr[0], pos[1] - tr[N], pos[2] - tr[2 * N], Pm[0], Pm[1], Pm[2], Pm[3], Pm[4], Pm[5],
                                   st.status != 0u, es);
                    es_pending = true;
                }
                ++n_toa;
            }
        }
        if (ES && es_pending) {
            es_pending = epoch_stats_row(es, wmask, es_out, n_toa - 1, p.n_warps);
            if (EH) epoch_hist_flush(es, wmask, p.ehist + (int64_t)(n_toa - 1) * p.ebins, p.eedges, p.equantity);
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            p.x[(int64_t)k * N + f] = pos[k];
            p.x[(int64_t)(3 + k) * N + f] = vel[k];
            p.x[(int64_t)(6 + k) * N + f] = 0.0;
            p.latch[(int64_t)k * N + f] = za[k];
        }
#pragma unroll
        for (int k = 0; k < Sym<9>::SZ; ++k) p.P[(int64_t)k * N + f] = Pm[k];
        p.has[f] = (int32_t)has;
        int32_t st_all = (int32_t)status_or;
        if (p.status) {
            st_all |= p.status[f];
            p.status[f] = st_all;
        }
        if (p.truth) filter_error_terms(pos[0], pos[1], pos[2], p.truth, N, f, st_all != 0, errv);
        if (SEL && p.uninit && (isnan(pos[0]) || isnan(pos[1]))) *p.uninit = 1;
        if (f == 0) {
            // keep the symmetric part as the latched covariance; written to the OUT half (the host copies it over
            // the input after the launch): blocks that start later must still read this launch's input
            double *o = p.latch_u + 16;
            o[0] = Ra[0]; o[1] = Ra[1]; o[2] = Ra[3];
            o[3] = Ra[1]; o[4] = Ra[2]; o[5] = Ra[4];
            o[6] = Ra[3]; o[7] = Ra[4]; o[8] = Ra[5];
        }
    }
    warp_accumulate(p.counters + CNT_UPDATES, n_updates);
    warp_accumulate(p.counters + CNT_ML_ITERS, st.ml_iters);
    warp_accumulate(p.counters + CNT_COST_EVALS, st.cost_evals);
    warp_accumulate(p.counters + CNT_GAIN_EVALS, st.gain_evals);
    warp_accumulate(p.counters + CNT_BAD, n_bad);
    static_assert(T9_BLOCK == STATS_CHUNK, "one statistics partial per replay block");
    if (p.truth) block_stats_partial(errv, smem, p.partials + (int64_t)blockIdx.x * 4);
}

template <bool PME, int MT, bool IMU, bool SEL = false, bool ES = false, bool EH = false>
static cudaError_t launch_k(const T9Params &p, cudaStream_t s) {
    const unsigned grid = (unsigned)((p.N + T9_BLOCK - 1) / T9_BLOCK);
    const size_t smem = (size_t)(t9_smem_rows(p.rs.m_slots, p.rs.fmt, PME, MT > 0) + (ES ? ES_W : 0)) * T9_BLOCK * sizeof(double);
    cudaError_t e = cudaFuncSetAttribute(t9_replay_kernel<PME, MT, IMU, SEL, ES, EH>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess) return e;
    t9_replay_kernel<PME, MT, IMU, SEL, ES, EH><<<grid, T9_BLOCK, smem, s>>>(p);
    return cudaGetLastError();
}

template <bool ES, bool EH>
static cudaError_t launch_replay_es(const T9Params &p, cudaStream_t s) {
    if (p.variant == 1 || p.variant == 2 || p.dt_f != nullptr || p.ml_init) // the general instantiation
        return p.rs.err != nullptr ? launch_k<true, 0, true, true, ES, EH>(p, s) : launch_k<false, 0, true, true, ES, EH>(p, s);
    if (p.no_imu) {
        if (p.rs.err != nullptr) return launch_k<true, 0, false, false, ES, EH>(p, s);
        if (p.rs.m_slots == 8) return launch_k<false, 8, false, false, ES, EH>(p, s);
        return launch_k<false, 0, false, false, ES, EH>(p, s);
    }
    if (p.rs.err != nullptr) return launch_k<true, 0, true, false, ES, EH>(p, s);
    if (p.rs.m_slots == 8) return launch_k<false, 8, true, false, ES, EH>(p, s);
    return launch_k<false, 0, true, false, ES, EH>(p, s);
}

cudaError_t launch_t9_replay(const T9Params &p, cudaStream_t s) {
    if (p.N <= 0 || p.n_events <= 0) return cudaSuccess;
    if (!p.escratch) return launch_replay_es<false, false>(p, s);
    return p.ehist ? launch_replay_es<true, true>(p, s) : launch_replay_es<true, false>(p, s);
}

// getPose (TOAIMU.cpp:476-510): predict-only, state untouched
__global__ void t9_get_pose_kernel(int64_t N, double dt, double jolt, const double *x, const double *P,
                                   double *x_pred, double *P_full) {
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= N) return;
    Sym<9> S;
#pragma unroll
    for (int k = 0; k < Sym<9>::SZ; ++k) S.a[k] = P[(int64_t)k * N + f];
    t9_predict_cov(S, dt, jolt);
    if (x_pred) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const double v = x[(int64_t)(3 + k) * N + f];
            x_pred[(int64_t)k * N + f] = x[(int64_t)k * N + f] + dt * v;
            x_pred[(int64_t)(3 + k) * N + f] = v;
            x_pred[(int64_t)(6 + k) * N + f] = 0.0;
        }
    }
    if (P_full) {
#pragma unroll
        for (int i = 0; i < 9; ++i)
#pragma unroll
            for (int j = 0; j < 9; ++j) P_full[(int64_t)(i * 9 + j) * N + f] = S.get(i, j);
    }
}

cudaError_t launch_t9_get_pose(int64_t N, double dt, double jolt, const double *x, const double *P, double *x_pred,
                               double *P_pred_full, cudaStream_t s) {
    if (N <= 0) return cudaSuccess;
    t9_get_pose_kernel<<<(unsigned)((N + 127) / 128), 128, 0, s>>>(N, dt, jolt, x, P, x_pred, P_pred_full);
    return cudaGetLastError();
}

} // namespace kfpos
