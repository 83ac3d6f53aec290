// kfpos_k8.cu -- persistent event-stream replay kernel for KalmanFilter (K8) batches:
// one thread per filter, the 8-state filter stays on chip while a schedule of
// sensor events (TOA / PX4Flow / IMU / magnetometer / compass, KF.cpp:64-221) is
// streamed through it.  The schedule (kind, dt) is common to the batch, the
// payload is per filter (SoA rows, filter index fastest).
#include "kfpos_k8.cuh"
#include "kfpos_kernels.cuh"

namespace kfpos {

#ifndef K8_BLOCK_SZ
#define K8_BLOCK_SZ 128
#endif
constexpr int K8_BLOCK = K8_BLOCK_SZ;
#ifndef K8_MINB
#define K8_MINB 2 // 255 registers: the register copy of P (72) + increments + Jacobian entries
#endif

// shared-memory rows (doubles) per thread: P^- (36), latched sensor samples (8), the landing
// zone of the event prefetch (rangings or <= 5 sensor values), [metres column when MT == 0],
// [errorEstimation column]
__host__ __device__ inline int k8_land_rows(int m, int fmt) { return raw_rows(fmt, m) > 5 ? raw_rows(fmt, m) : 5; }
__host__ __device__ inline int k8_smem_rows(int m, int fmt, bool pme, bool in_regs) {
    return 36 + 8 + k8_land_rows(m, fmt) + (in_regs ? 0 : m) + (pme ? m : 0);
}

// (the raw-magnetometer event's atan2, ~140 instructions, kept out of the replay loop's code)
static __device__ __noinline__ double atan2_out_of_line(double y, double x) { return atan2(y, x); }

KF_DEV int event_rows(int kind) {
    switch (kind) {
    case EV_PX4: return 5;
    case EV_IMU: return 3;
    case EV_MAG: return 2;
    default: return 1;
    }
}

KF_DEV void prefetch_event(const RawColPriv &raw, const Col &land, const EventDesc &ev, int m, const RangeStream &rs,
                           const double *sensors, int64_t N, int64_t f) {
    if (ev.kind == EV_TOA) {
        prefetch_epoch(raw, m, rs.ranges, rs.fmt, ev.offset * N + f, N);
    } else {
        const int rows = event_rows(ev.kind);
        for (int i = 0; i < rows; ++i) cp_async_8(&land[i], sensors + (ev.offset + i) * N + f);
        cp_async_commit();
    }
}

// SEL: EKF-side NLOS variants (config_pos.xml variant / numIgnoredRangings / bestMode, see kfpos_t6.cu):
// at a TOA event the 2-D ML estimator, started at the predicted position, selects the rangings --
// variant 1 drops the N with the largest residual, variant 2 keeps the best THREE anchors -- and the
// update runs on the survivors.
// MLI: the ML-initialisation branch and the per-filter tag height (kfpos_config.ml_initial_position) are compiled in.
// ES: per-epoch statistics at every TOA event (see kfpos_t6.cu): the terms go to a private shared-memory column, and
// the warp sums them at the top of the next event or after the last one, behind a __syncwarp -- lanes of a ragged
// replay (SEL && dt_f) reach that point on different paths.  The NEES is that of the x-y block, z = the tag height.
// EH (only with ES): the per-epoch error histogram, binned beside epoch_stats_row (epoch_hist_flush).
template <bool PME, int MT, bool SEL = false, bool MLI = SEL, bool ES = false, bool EH = false>
__global__ void __launch_bounds__(K8_BLOCK, K8_MINB) k8_replay_kernel(const __grid_constant__ K8Params p) {
    extern __shared__ double smem[];
    const int64_t f = (int64_t)blockIdx.x * K8_BLOCK + threadIdx.x;
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
            Col c = {col + (size_t)row * K8_BLOCK, K8_BLOCK};
            row += rows;
            return c;
        };
        const Col Pm = take(36);
        // latched samples: px4 vx,vy,gz,cv | imu ax,ay,wz | mag angle   (KF.h:92-130)
        const Col latch = take(8);
        const Col land = take(k8_land_rows(m, p.rs.fmt));
        const RawColPriv raw = {land}; // rangings land in the same private column
        EpochT<PME, MT> ep;
        ep.z = MT > 0 ? Pm : take(m);
        ep.e = PME ? take(m) : Pm;
        ep.e0 = p.rs.err_scalar;
        ep.m_slots = m;
        ep.valid = 0u;

        // persistent members: position, velocity, angle, angular speed (acceleration is never
        // written back: KF.cpp:287-291,315-318)
        double px = p.x[0 * N + f], py = p.x[1 * N + f], vx = p.x[2 * N + f], vy = p.x[3 * N + f];
        double th = p.x[6 * N + f], om = p.x[7 * N + f];
        // the covariance lives in REGISTERS from event to event (Pr); Pm only backs P^- up inside an event that
        // fuses several sensors
        Sym<8> Pr;
#pragma unroll
        for (int k = 0; k < Sym<8>::SZ; ++k) Pr.a[k] = p.P[(int64_t)k * N + f];
#pragma unroll
        for (int k = 0; k < 8; ++k) latch[k] = p.latch[(int64_t)k * N + f];
        unsigned has = (unsigned)p.has[f]; // bit0 px4, bit1 imu, bit2 mag latched
        unsigned status_or = 0;
        // time of the events this filter skipped (a PX4 frame of quality 0 returns before the
        // reference reads its clock, KF.cpp:111-113); persists across launches in latch row 8
        double carry = p.latch[8 * N + f];
        double ic00 = p.latch_u[0], ic01 = p.latch_u[1], ic11 = p.latch_u[2], icw = p.latch_u[3];
        int n_toa = 0;
        // the tag height is per filter only after a 3-D ML initialisation (KF.cpp:256-257)
        const bool z_per_filter = MLI && p.cfg.ml_init && !p.cfg.use_fixed_height;
        double tag_z = z_per_filter ? p.latch[9 * N + f] : p.cfg.tag_z;
        const Col es = {col + (size_t)(ES ? k8_smem_rows(m, p.rs.fmt, PME, MT > 0) : 0) * K8_BLOCK, K8_BLOCK};
        double *const es_out = ES ? p.escratch + (f >> 5) * ES_W : nullptr;
        bool es_pending = false; // the row n_toa - 1 still has to be summed (common to the warp)

        if (p.n_events > 0) prefetch_event(raw, land, p.events[0], m, p.rs, p.sensors, N, f);
        for (int e = 0; e < p.n_events; ++e) {
            if (ES && es_pending) {
                es_pending = epoch_stats_row(es, wmask, es_out, n_toa - 1, p.n_warps);
                if (EH) epoch_hist_flush(es, wmask, p.ehist + (int64_t)(n_toa - 1) * p.ebins, p.eedges, p.equantity);
            }
            const EventDesc ev = p.events[e];
            cp_async_wait_all();
            double dt_ev = ev.dt;
            if (SEL && p.dt_f) { // ragged replay: every filter has its own time steps
                dt_ev = p.dt_f[(int64_t)e * N + f];
                if (dt_ev < 0.0) { // this filter has no such event
                    if (e + 1 < p.n_events) prefetch_event(raw, land, p.events[e + 1], m, p.rs, p.sensors, N, f);
                    if (ev.kind == EV_TOA) { // its trajectory row repeats the current state
                        if (p.traj) {
                            p.traj[((int64_t)n_toa * 3 + 0) * N + f] = px;
                            p.traj[((int64_t)n_toa * 3 + 1) * N + f] = py;
                            p.traj[((int64_t)n_toa * 3 + 2) * N + f] = th;
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
            st.status = 0u;
            K8Meas ms;
            ms.has_px4 = ms.has_imu = ms.has_mag = false;
            ms.latch = latch;
            ms.px4_cg = p.cfg.px4_cov_gyro;
            ms.mag_c = p.cfg.mag_cov;
            bool has_r = false, skip = false;
            switch (ev.kind) {
            case EV_TOA: { // newTOAMeasurement (KF.cpp:64-97): rangings + latched px4 / imu / mag
                convert_epoch<PME, MT>(ep, raw, p.rs.ranges, p.rs.fmt, p.rs.err, ev.offset * N + f, N);
                has_r = true;
                ms.has_px4 = has & 1u; ms.has_imu = (has >> 1) & 1u; ms.has_mag = (has >> 2) & 1u;
                break;
            }
            case EV_PX4: { // newPX4FlowMeasurement (KF.cpp:100-133)
                const double ix = land[0], iy = land[1], irz = land[2], itus = land[3];
                const int quality = (int)land[4];
                if (quality == 0) { skip = true; break; }
                const double it = itus / 1000000.0;
                const double pvy = iy / it * p.cfg.px4_height, pvx = ix / it * p.cfg.px4_height;
                const double cv = itus > 0 ? p.cfg.px4_cov_vel / it * p.cfg.px4_height / quality
                                           : p.cfg.px4_cov_vel * quality;
                latch[0] = pvx; latch[1] = pvy; latch[2] = irz / it; latch[3] = cv;
                has |= 1u;
                ms.has_px4 = true;
                break;
            }
            case EV_IMU: { // newIMUMeasurement (KF.cpp:137-176); aux = cov_acc[0],[1],[3],[4], cov_av[8]
                ic00 = p.cfg.imu_fix_acc ? p.cfg.imu_cov_acc : ev.aux[0];
                ic01 = ev.aux[1];
                ic11 = p.cfg.imu_fix_acc ? p.cfg.imu_cov_acc : ev.aux[3];
                icw = p.cfg.imu_fix_gyro ? p.cfg.imu_cov_gyro : ev.aux[4];
                if (ev.aux[1] != ev.aux[2]) st.status |= 64u; // asymmetric block: symmetric part used
                const double wz = land[0], lax = land[1], lay = land[2];
                latch[6] = wz; latch[4] = lax; latch[5] = lay;
                has |= 2u;
                ms.has_imu = true;
                break;
            }
            case EV_MAG: { // newMAGMeasurement (KF.cpp:179-193): mag only, angle not normalised
                latch[7] = atan2_out_of_line(land[1], land[0]) - p.cfg.mag_offset;
                has |= 4u;
                ms.has_mag = true;
                break;
            }
            default: { // newCompassMeasurement (KF.cpp:195-221): mag + latched px4 + latched imu
                latch[7] = wrap_angle(land[0]);
                has |= 4u;
                ms.has_mag = true;
                ms.has_px4 = has & 1u; ms.has_imu = (has >> 1) & 1u;
                break;
            }
            }
            if (e + 1 < p.n_events) prefetch_event(raw, land, p.events[e + 1], m, p.rs, p.sensors, N, f);
            // lanes that re-converge after the inner Newton loop of a ranging event: every lane of the warp, except
            // the filters that are still uninitialised (ML initialisation) -- and nobody in a ragged replay
            unsigned umask = (SEL && p.dt_f) ? 0u : wmask;
            if (MLI && umask && p.cfg.ml_init && ev.kind == EV_TOA) umask = __ballot_sync(wmask, !(isnan(px) || isnan(py)));
            if (skip) {
                carry += dt_ev;
            } else if (MLI && p.cfg.ml_init && (isnan(px) || isnan(py))) {
                // ---- the constructor without initialPosition (KF.cpp:244-285): the clock is read, the sample is
                // latched (above), and an epoch with rangings initialises position and the 2x2 position block
                // of the all-zero covariance from MLLocation; no predict, no update
                carry = 0.0;
                st.status |= 256u;
                if (has_r) {
                    const bool fh = p.cfg.use_fixed_height != 0;
                    double p0[3] = {1.0, 1.0, fh ? tag_z : 4.0}, sse0, c0[6] = {0, 0, 0, 0, 0, 0};
                    int irc;
                    if (fh) irc = ml_solve2<PME, MT>(p.anchors, ep, ep.valid, p0, sse0, st.ml_iters, c0, nullptr, p.cfg.zero_tz != 0);
                    else irc = ml_solve3<PME, MT>(p.anchors, ep, ep.valid, p0, sse0, st.ml_iters, c0);
                    if (irc == ML_SINGULAR) {
                        st.status |= 4u; // the solver throws before mPosition is assigned
                    } else {
                        px = p0[0]; py = p0[1];
                        if (!fh) tag_z = p0[2];
                        // too few rangings: the start point comes back with an EMPTY covariance matrix, whose
                        // (0,0) throws after position (and tag height) have been assigned (KF.cpp:267)
                        if (irc == ML_FEW) st.status |= 2u;
                        else { Pr.a[0] = c0[0]; Pr.a[1] = c0[1]; Pr.a[2] = c0[2]; } // xx, yx, yy (both packings agree)
                    }
                }
                if (st.status & ~(32u | 64u | 256u)) n_bad += 1;
                status_or |= st.status;
                if (ev.kind == EV_TOA) {
                    if (p.traj) {
                        p.traj[((int64_t)n_toa * 3 + 0) * N + f] = px;
                        p.traj[((int64_t)n_toa * 3 + 1) * N + f] = py;
                        p.traj[((int64_t)n_toa * 3 + 2) * N + f] = th;
                    }
                    if (ES) {
                        const double *tr = p.etruth + (int64_t)n_toa * 3 * N + f;
                        epoch_terms<2>(px - tr[0], py - tr[N], tag_z - tr[2 * N], Pr.a[0], Pr.a[1], Pr.a[2], 0.0, 0.0, 0.0,
                                       st.status != 0u, es);
                        es_pending = true;
                    }
                    ++n_toa;
                }
            } else {
                const double dt = dt_ev + carry;
                carry = 0.0;

                // ---- predict (KF.cpp:287-305): a = 0 at the start of every step
                Sym<8> &Pw = Pr;
                k8_predict_cov(Pw, dt, p.cfg.accel_noise, p.cfg.jolt);
                // one sensor and no rangings: the deferred update on the register copy (k8_update_light)
                bool light = ev.kind == EV_IMU || ev.kind == EV_PX4 || ev.kind == EV_MAG;
                if (!light || ev.kind == EV_IMU) { // (the IMU event's straight-line form keeps P^- there as its backup)
#pragma unroll
                    for (int k = 0; k < Sym<8>::SZ; ++k) Pm[k] = Pw.a[k];
                }
                const double xp[8] = {px + dt * vx, py + dt * vy, vx, vy, 0.0, 0.0, wrap_angle(th + dt * om), om};

                if (ms.has_imu) {
                    ms.imu_c00 = ic00; ms.imu_c01 = ic01; ms.imu_c11 = ic11; ms.imu_cw = icw;
                }

                if (has_r && ep.valid == 0u) st.status |= 1u;
                double dx[8];
                unsigned used = ep.valid;
                if (SEL && has_r) {
                    const int n = __popc(ep.valid);
                    const double start[3] = {xp[0], xp[1], tag_z};
                    double p0[3] = {start[0], start[1], start[2]}, sse0, cov0[6];
                    if (p.cfg.variant == 1 && n > 0) {
                        if (ml_solve2<PME, MT>(p.anchors, ep, ep.valid, p0, sse0, st.ml_iters, nullptr, nullptr,
                                               p.cfg.zero_tz != 0) == ML_OK) {
                            const int drop = min(n - 3, p.cfg.n_ignore);
                            used = drop_worst<PME, MT>(p.anchors, ep, used, p0, drop < 0 ? 0 : drop);
                        }
                    } else if (p.cfg.variant == 2 && n >= 3) {
                        int grc;
                        double c2[3];
                        // the all-ranging solve; a failed solve (there or in a subset) selects nothing
                        if (ml_solve2<PME, MT>(p.anchors, ep, ep.valid, p0, sse0, st.ml_iters, c2, nullptr,
                                               p.cfg.zero_tz != 0) != ML_SINGULAR)
                            best_group<PME, MT>(p.anchors, ep, ep.valid, true, p.cfg.best_mode, start, st.ml_iters, p0,
                                                cov0, used, grc, p.cfg.zero_tz != 0);
                    }
                }
                int rc = 0;
                if (ev.kind == EV_IMU) {
                    // speculation failed (the break tests did not come out as continue, continue, stop): the general
                    // form below repeats the event from the backed-up P^-
                    if (!k8_update_imu_fast(ms, xp, Pw, dx, st)) light = false;
                }
                if (light) {
                    if (ev.kind == EV_IMU) { /* done above */ }
                    else if (ev.kind == EV_PX4) k8_update_light<EV_PX4>(p.cfg, ms, dt, xp, Pw, dx, st);
                    else k8_update_light<EV_MAG>(p.cfg, ms, dt, xp, Pw, dx, st);
                } else {
                    rc = k8_update<PME, MT>(p.anchors, p.cfg, tag_z, ep, has_r, used, ms, dt, xp, Pm, Pw, dx, st, umask);
                    if (rc != 0) { // update skipped: P^- is what remains
#pragma unroll
                        for (int k = 0; k < Sym<8>::SZ; ++k) Pw.a[k] = Pm[k];
                    }
                }
                if (rc == 0) {
                    px = xp[0] + dx[0]; py = xp[1] + dx[1];
                    vx = xp[2] + dx[2]; vy = xp[3] + dx[3];
                    th = xp[6] + dx[6]; om = xp[7] + dx[7]; // written back un-wrapped (KF.cpp:317)
                    if (!(isfinite(px) && isfinite(py) && isfinite(vx) && isfinite(vy) && isfinite(th) && isfinite(om)))
                        st.status |= 8u;
                } else {
                    st.status |= 4u; // the reference would abort on this uncaught exception; the update is skipped
                }
                n_updates += 1;
                if (st.status & ~(32u | 64u)) n_bad += 1;
                status_or |= st.status;
                if (ev.kind == EV_TOA) {
                    if (p.traj) {
                        p.traj[((int64_t)n_toa * 3 + 0) * N + f] = px;
                        p.traj[((int64_t)n_toa * 3 + 1) * N + f] = py;
                        p.traj[((int64_t)n_toa * 3 + 2) * N + f] = th;
                    }
                    if (ES) {
                        const double *tr = p.etruth + (int64_t)n_toa * 3 * N + f;
                        epoch_terms<2>(px - tr[0], py - tr[N], tag_z - tr[2 * N], Pr.a[0], Pr.a[1], Pr.a[2], 0.0, 0.0, 0.0,
                                       st.status != 0u, es);
                        es_pending = true;
                    }
                    ++n_toa;
                }

            }
            if (!(SEL && p.dt_f)) __syncwarp(wmask); // the IEKF trip count differs per lane
        }
        if (ES && es_pending) {
            es_pending = epoch_stats_row(es, wmask, es_out, n_toa - 1, p.n_warps);
            if (EH) epoch_hist_flush(es, wmask, p.ehist + (int64_t)(n_toa - 1) * p.ebins, p.eedges, p.equantity);
        }
        p.x[0 * N + f] = px; p.x[1 * N + f] = py; p.x[2 * N + f] = vx; p.x[3 * N + f] = vy;
        p.x[4 * N + f] = 0.0; p.x[5 * N + f] = 0.0; p.x[6 * N + f] = th; p.x[7 * N + f] = om;
#pragma unroll
        for (int k = 0; k < Sym<8>::SZ; ++k) p.P[(int64_t)k * N + f] = Pr.a[k];
#pragma unroll
        for (int k = 0; k < 8; ++k) p.latch[(int64_t)k * N + f] = latch[k];
        p.has[f] = (int32_t)has;
        p.latch[8 * N + f] = carry;
        if (z_per_filter) p.latch[9 * N + f] = tag_z;
        if (MLI && p.uninit && (isnan(px) || isnan(py))) *p.uninit = 1;
        int32_t st_all = (int32_t)status_or;
        if (p.status) {
            st_all |= p.status[f];
            p.status[f] = st_all;
        }
        // planar filter: z is the configured tag height (KF.cpp:328-332)
        if (p.truth) filter_error_terms(px, py, tag_z, p.truth, N, f, st_all != 0, errv);
        if (f == 0) {
            // written to the OUT half: blocks of this launch that start later must still read the launch's input
            p.latch_u[16] = ic00; p.latch_u[17] = ic01; p.latch_u[18] = ic11; p.latch_u[19] = icw;
        }
    }
    warp_accumulate(p.counters + CNT_UPDATES, n_updates);
    warp_accumulate(p.counters + CNT_ML_ITERS, st.ml_iters);
    warp_accumulate(p.counters + CNT_COST_EVALS, st.cost_evals);
    warp_accumulate(p.counters + CNT_GAIN_EVALS, st.gain_evals);
    warp_accumulate(p.counters + CNT_BAD, n_bad);
    static_assert(K8_BLOCK == STATS_CHUNK, "one statistics partial per replay block");
    if (p.truth) block_stats_partial(errv, smem, p.partials + (int64_t)blockIdx.x * 4);
}

template <bool PME, int MT, bool SEL, bool MLI, bool ES, bool EH>
static cudaError_t launch_k(const K8Params &p, cudaStream_t s) {
    const unsigned grid = (unsigned)((p.N + K8_BLOCK - 1) / K8_BLOCK);
    const size_t smem = (size_t)(k8_smem_rows(p.rs.m_slots, p.rs.fmt, PME, MT > 0) + (ES ? ES_W : 0)) * K8_BLOCK * sizeof(double);
    cudaError_t e = cudaFuncSetAttribute(k8_replay_kernel<PME, MT, SEL, MLI, ES, EH>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k8_replay_kernel<PME, MT, SEL, MLI, ES, EH><<<grid, K8_BLOCK, smem, s>>>(p);
    return cudaGetLastError();
}

template <bool PME, int MT, bool ES, bool EH>
static cudaError_t launch_tuned(const K8Params &p, cudaStream_t s) {
    return p.cfg.ml_init ? launch_k<PME, MT, false, true, ES, EH>(p, s) : launch_k<PME, MT, false, false, ES, EH>(p, s);
}

template <bool ES, bool EH>
static cudaError_t launch_replay_es(const K8Params &p, cudaStream_t s) {
    if (p.cfg.variant == 1 || p.cfg.variant == 2 || p.dt_f != nullptr) // the general instantiation
        return p.rs.err != nullptr ? launch_k<true, 0, true, true, ES, EH>(p, s) : launch_k<false, 0, true, true, ES, EH>(p, s);
    if (p.rs.err != nullptr) return launch_tuned<true, 0, ES, EH>(p, s);
    if (p.rs.m_slots == 8 && !p.cfg.zero_tz) return launch_tuned<false, 8, ES, EH>(p, s);
    return launch_tuned<false, 0, ES, EH>(p, s);
}

cudaError_t launch_k8_replay(const K8Params &p, cudaStream_t s) {
    if (p.N <= 0 || p.n_events <= 0) return cudaSuccess;
    if (!p.escratch) return launch_replay_es<false, false>(p, s);
    return p.ehist ? launch_replay_es<true, true>(p, s) : launch_replay_es<true, false>(p, s);
}

// getPose (KF.cpp:709-747): predict-only, state untouched
__global__ void k8_get_pose_kernel(int64_t N, double dt, double accel_noise, double jolt, const double *x,
                                   const double *P, double *x_pred, double *P_full) {
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= N) return;
    Sym<8> S;
#pragma unroll
    for (int k = 0; k < Sym<8>::SZ; ++k) S.a[k] = P[(int64_t)k * N + f];
    k8_predict_cov(S, dt, accel_noise, jolt);
    if (x_pred) {
        const double px = x[f], py = x[N + f], vx = x[2 * N + f], vy = x[3 * N + f], th = x[6 * N + f], om = x[7 * N + f];
        x_pred[0 * N + f] = px + dt * vx; x_pred[1 * N + f] = py + dt * vy;
        x_pred[2 * N + f] = vx; x_pred[3 * N + f] = vy;
        x_pred[4 * N + f] = 0.0; x_pred[5 * N + f] = 0.0;
        x_pred[6 * N + f] = wrap_angle(th + dt * om); x_pred[7 * N + f] = om;
    }
    if (P_full) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) P_full[(int64_t)(i * 8 + j) * N + f] = S.get(i, j);
    }
}

cudaError_t launch_k8_get_pose(int64_t N, double dt, double accel_noise, double jolt, const double *x,
                               const double *P, double *x_pred, double *P_pred_full, cudaStream_t s) {
    if (N <= 0) return cudaSuccess;
    k8_get_pose_kernel<<<(unsigned)((N + 127) / 128), 128, 0, s>>>(N, dt, accel_noise, jolt, x, P, x_pred, P_pred_full);
    return cudaGetLastError();
}

} // namespace kfpos
