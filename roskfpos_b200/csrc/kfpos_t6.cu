// kfpos_t6.cu -- persistent replay kernel for KalmanFilterTOA batches (G1+G2+G3+G5
// of SURVEY.md §2).  One thread per filter; across all T steps the filter's position
// (and, for a compile-time anchor count, the epoch's ranges) stay in registers and its
// packed covariance in a private shared-memory column; the update is computed in
// factored form (kfpos_t6.cuh), so the covariance is touched twice per step (predict,
// apply).  Per step the only global traffic is the coalesced read of the filter's M
// rangings (SoA, filter index fastest), prefetched one epoch ahead with cp.async, and
// the optional trajectory / selection stores.
#include "kfpos_kernels.cuh"
#include "kfpos_t6.cuh"

namespace kfpos {

constexpr int T6_BLOCK = 128;
#ifndef T6_MINB
#define T6_MINB 4 // 128 registers; more resident warps do not help a dispatch-bound kernel (profiles/README.md)
#endif

// shared-memory rows (doubles) per thread: [metres column when MT == 0], [errorEstimation
// column], P^-, the reference point of the Newton cycle detector, landing zone of the prefetch
__host__ __device__ inline int t6_smem_rows(int m, int fmt, bool pme, bool in_regs) {
    return (in_regs ? 0 : m) + (pme ? m : 0) + 21 + 3 + raw_rows(fmt, m);
}

// MT > 0: compile-time anchor count (unrolled anchor loops, ranges in registers); MT == 0: run-time.
// SEL: EKF-side NLOS variants (README.md:85-108, config_pos.xml:5-28; the reference documents them
// but only implements them in MLLocation): before the update the ML estimator, started at the
// predicted position, selects the rangings -- variant 1 drops the numIgnoredRangings with the
// largest residual at its solution (ML.cpp:307-347), variant 2 keeps the 4-anchor group with the
// smallest covariance criterion (ML.cpp:351-414, bestMode) -- and the iterated update runs on the
// survivors.  The mask of the slots used goes to `sel`.
// FMT: the wire format as a compile-time constant (the tuned instantiation: the per-epoch prefetch / conversion code of
// the other two formats -- a third of the replay loop's 2300 instructions, against a 32 KB instruction cache -- is
// not generated); -1 = read from the parameters.
// ES: per-epoch statistics (kfpos_batch_set_truth_traj): after every epoch the filter's error terms go to a private
// shared-memory column (6 rows behind the others), and at the top of the next epoch -- the one point every lane of
// the warp passes, stepping or not -- the warp sums them (epoch_stats_flush).  The ES = false code is unchanged.
// EH (only with ES): the per-epoch error histogram, binned at the same two points as the sums (epoch_hist_flush).
template <bool PME, bool LOO, int MT, bool SEL = false, int FMT = -1, bool ES = false, bool EH = false>
__global__ void __launch_bounds__(T6_BLOCK, T6_MINB) t6_replay_kernel(const __grid_constant__ T6Params p) {
    extern __shared__ double smem[];
    const int fmt = FMT >= 0 ? FMT : p.rs.fmt;
    // per-filter time steps (assembled logs of different length) only in the FMT = -1 instantiations: the launcher routes them there
    const double *dt_f = FMT >= 0 ? nullptr : p.dt_f;
    const int64_t f = (int64_t)blockIdx.x * T6_BLOCK + threadIdx.x;
    const bool active = f < p.N;
    const unsigned wmask = __ballot_sync(0xffffffffu, active);
    StepStats st = {0u, 0u, 0u, 0u};
    unsigned n_updates = 0, n_bad = 0, n_ignored = 0;
    double errv[4] = {0.0, 0.0, 0.0, 0.0}; // error terms of the final state (fused statistics)

    if (active) {
        const int64_t N = p.N;
        const int m = MT > 0 ? MT : p.rs.m_slots;
        // carve this thread's columns
        double *col = smem + threadIdx.x;
        int row = 0;
        auto take = [&](int rows) {
            Col c = {col + (size_t)row * T6_BLOCK, T6_BLOCK};
            row += rows;
            return c;
        };
        EpochT<PME, MT> ep;
        const Col Pm = take(21);
        const Col cyc = take(3);
        ep.z = MT > 0 ? Pm : take(m);
        ep.e = PME ? take(m) : Pm;
        ep.e0 = p.rs.err_scalar;
        ep.m_slots = m;
        // landing zone of the cp.async prefetch of the next epoch
        const RawCol raw = make_raw(smem + (size_t)row * T6_BLOCK, fmt, threadIdx.x, T6_BLOCK);
        const Col es = {col + (size_t)(ES ? t6_smem_rows(m, fmt, PME, MT > 0) : 0) * T6_BLOCK, T6_BLOCK};
        double *const es_out = ES ? p.escratch + (f >> 5) * ES_W : nullptr;

        double pos[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) pos[k] = p.x[(int64_t)k * N + f];
#pragma unroll
        for (int k = 0; k < Sym<6>::SZ; ++k) Pm[k] = p.P[(int64_t)k * N + f];
        unsigned status_or = 0;

        prefetch_epoch(raw, m, p.rs.ranges, fmt, f, N);
        double dt_next = dt_f ? __ldg(dt_f + f) : 0.0;
        for (int t = 0; t < p.T; ++t) {
            if (ES && t > 0) epoch_stats_flush(es, wmask, es_out + (int64_t)(t - 1) * p.n_warps * ES_W);
            if (EH && t > 0) epoch_hist_flush(es, wmask, p.ehist + (int64_t)(t - 1) * p.ebins, p.eedges, p.equantity);
            // per-filter time steps (assembled logs): a negative dt = this filter has no epoch t.
            // The lanes that do step are the ones that re-converge below.
            const double dt = dt_f ? dt_next : __ldg(p.dt + t);
            if (dt_f && t + 1 < p.T) dt_next = __ldg(dt_f + (int64_t)(t + 1) * N + f);
            const bool stepping = !dt_f || !(dt < 0.0);
            const unsigned emask = dt_f ? __ballot_sync(wmask, stepping) : wmask;
            if (!stepping) { // keep the landing zone protocol going, touch nothing else
                cp_async_wait_all();
                if (t + 1 < p.T) prefetch_epoch(raw, m, p.rs.ranges, fmt, (int64_t)(t + 1) * m * N + f, N);
                if (p.traj) {
#pragma unroll
                    for (int k = 0; k < 3; ++k) p.traj[((int64_t)t * 3 + k) * N + f] = pos[k];
                }
                if (p.sel) p.sel[(int64_t)t * N + f] = -1;
                if (ES) epoch_terms_zero(es);
                continue;
            }

            // ---- predict (TOA.cpp:115-123): x^- = F x with v = 0, P^- = F P F^T + Q.
            // The member covariance is overwritten before the try block, so P^-
            // is what survives a failed update.
            {
                Sym<6> Pw;
#pragma unroll
                for (int k = 0; k < Sym<6>::SZ; ++k) Pw.a[k] = Pm[k];
                t6_predict_cov(Pw, dt, p.accel_noise);
#pragma unroll
                for (int k = 0; k < Sym<6>::SZ; ++k) Pm[k] = Pw.a[k];
            }
            // ---- this epoch's rangings (landed during the previous epoch); start the next fetch
            cp_async_wait_all();
            convert_epoch<PME, MT, RawCol, true>(ep, raw, p.rs.ranges, fmt, p.rs.err, (int64_t)t * m * N + f, N);
            if (t + 1 < p.T) prefetch_epoch(raw, m, p.rs.ranges, fmt, (int64_t)(t + 1) * m * N + f, N);

            st.status = 0u;
            if (ep.valid == 0u) st.status |= 1u;
            T6Result res;
            int rc, ignored = -1;
            if (SEL) {
                unsigned used = ep.valid;
                const int n = __popc(ep.valid);
                double p0[3] = {pos[0], pos[1], pos[2]}, sse0, cov0[6];
                if (p.variant == 1 && n > 0) {
                    if (ml_solve3<PME, MT>(p.anchors, ep, ep.valid, p0, sse0, st.ml_iters, nullptr) == ML_OK) {
                        int drop = min(n - 4, p.n_ignore);
                        used = drop_worst<PME, MT>(p.anchors, ep, used, p0, drop < 0 ? 0 : drop);
                    }
                } else if (p.variant == 2 && n >= 4) {
                    int grc;
                    // the all-ranging solve of :353; a failed solve (there or in a subset) selects nothing
                    if (ml_solve3<PME, MT>(p.anchors, ep, ep.valid, p0, sse0, st.ml_iters, cov0) != ML_SINGULAR)
                        best_group<PME, MT>(p.anchors, ep, ep.valid, false, p.best_mode, pos, st.ml_iters, p0, cov0, used, grc);
                }
                rc = t6_update<PME, MT>(p.anchors, ep, used, pos, Pm, res, st, 0u, &cyc);
                ignored = (int)used;
            } else if (!LOO) {
                rc = t6_update<PME, MT, !LOO>(p.anchors, ep, ep.valid, pos, Pm, res, st, emask, &cyc, p.counters);
                __syncwarp(emask);
            } else {
                // kalmanStep3DCanIgnoreAnAnchor (TOA.cpp:185-238): the all-anchor solve (i = -1),
                // then -- only with > 4 rangings -- one solve per left-out anchor, all from the same P^-
                T6Result best;
                double maxDist = 0.0;
                int idx = -1;
                bool first = true;
                const int n_try = __popc(ep.valid) > 4 ? m : 0;
                rc = 0;
                for (int i = -1; i < n_try && rc == 0; ++i) {
                    if (i >= 0 && !((ep.valid >> i) & 1u)) continue;
                    T6Result ri;
                    rc = t6_update<PME, MT>(p.anchors, ep, i < 0 ? ep.valid : (ep.valid & ~(1u << i)), pos, Pm, ri, st, 0u, &cyc);
                    if (rc != 0) break;
                    if (i < 0) {
                        res = ri;
                        continue;
                    }
                    const double ex = p.anchors.x[i] - (pos[0] + ri.dx[0]);
                    const double ey = p.anchors.y[i] - (pos[1] + ri.dx[1]);
                    const double ez = p.anchors.z[i] - (pos[2] + ri.dx[2]);
                    const double diff = ep.z_at(i) - sqrt(ex * ex + ey * ey + ez * ez);
                    if (first || diff > maxDist) { // strict >, first seeds (TOA.cpp:209)
                        maxDist = diff;
                        best = ri;
                        idx = i;
                        first = false;
                    }
                }
                if (rc == 0 && idx >= 0 && maxDist > 0 && (res.cost - best.cost) > p.ignore_thr) {
                    res = best;
                    ignored = idx;
                    n_ignored += 1;
                }
            }
            if (rc == 0) {
                // stateToPose (TOA.cpp:159-183): position kept, velocity dropped
                pos[0] += res.dx[0]; pos[1] += res.dx[1]; pos[2] += res.dx[2];
                apply_cov_block3<6>(Pm, res.M);
                if (!(isfinite(pos[0]) && isfinite(pos[1]) && isfinite(pos[2]))) st.status |= 8u;
            } else {
                st.status |= 4u; // catch (std::runtime_error): update skipped (TOA.cpp:151)
            }
            n_updates += 1;
            if (st.status & ~32u) n_bad += 1;
            status_or |= st.status;
            if (p.traj) {
#pragma unroll
                for (int k = 0; k < 3; ++k) p.traj[((int64_t)t * 3 + k) * N + f] = pos[k];
            }
            if (p.sel) p.sel[(int64_t)t * N + f] = ignored;
            if (ES) {
                const double *tr = p.etruth + (int64_t)t * 3 * N + f;
                epoch_terms<3>(pos[0] - tr[0], pos[1] - tr[N], pos[2] - tr[2 * N], Pm[0], Pm[1], Pm[2], Pm[3], Pm[4], Pm[5],
                               st.status != 0u, es);
            }
        }
        if (ES) epoch_stats_flush(es, wmask, es_out + (int64_t)(p.T - 1) * p.n_warps * ES_W);
        if (EH) epoch_hist_flush(es, wmask, p.ehist + (int64_t)(p.T - 1) * p.ebins, p.eedges, p.equantity);

#pragma unroll
        for (int k = 0; k < 3; ++k) p.x[(int64_t)k * N + f] = pos[k];
#pragma unroll
        for (int k = 0; k < Sym<6>::SZ; ++k) p.P[(int64_t)k * N + f] = Pm[k];
        int32_t st_all = (int32_t)status_or;
        if (p.status) {
            st_all |= p.status[f];
            p.status[f] = st_all;
        }
        if (p.truth) filter_error_terms(pos[0], pos[1], pos[2], p.truth, N, f, st_all != 0, errv);
    }
    warp_accumulate(p.counters + CNT_UPDATES, n_updates);
    warp_accumulate(p.counters + CNT_ML_ITERS, st.ml_iters);
    warp_accumulate(p.counters + CNT_COST_EVALS, st.cost_evals);
    warp_accumulate(p.counters + CNT_GAIN_EVALS, st.gain_evals);
    warp_accumulate(p.counters + CNT_BAD, n_bad);
    warp_accumulate(p.counters + CNT_IGNORED, n_ignored);
    // the block-level reduction of the error statistics, fused into the last step of the replay
    static_assert(T6_BLOCK == STATS_CHUNK, "one statistics partial per replay block");
    if (p.truth) block_stats_partial(errv, smem, p.partials + (int64_t)blockIdx.x * 4);
}

template <bool PME, bool LOO, int MT, bool SEL = false, int FMT = -1, bool ES = false, bool EH = false>
static cudaError_t launch_k(const T6Params &p, cudaStream_t s) {
    const unsigned grid = (unsigned)((p.N + T6_BLOCK - 1) / T6_BLOCK);
    const size_t smem = (size_t)(t6_smem_rows(p.rs.m_slots, p.rs.fmt, PME, MT > 0) + (ES ? ES_W : 0)) * T6_BLOCK * sizeof(double);
    cudaError_t e = cudaFuncSetAttribute(t6_replay_kernel<PME, LOO, MT, SEL, FMT, ES, EH>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    t6_replay_kernel<PME, LOO, MT, SEL, FMT, ES, EH><<<grid, T6_BLOCK, smem, s>>>(p);
    return cudaGetLastError();
}
// the plain replay with a compile-time anchor count: one instantiation per wire format
template <int MT, bool ES, bool EH>
static cudaError_t launch_tuned(const T6Params &p, cudaStream_t s) {
    if (p.dt_f != nullptr) return launch_k<false, false, MT, false, -1, ES, EH>(p, s); // per-filter time steps
    switch (p.rs.fmt) {
    case 1: return launch_k<false, false, MT, false, 1, ES, EH>(p, s);
    case 2: return launch_k<false, false, MT, false, 2, ES, EH>(p, s);
    default: return launch_k<false, false, MT, false, 0, ES, EH>(p, s);
    }
}

template <bool ES, bool EH>
static cudaError_t launch_replay_es(const T6Params &p, cudaStream_t s) {
    const bool pme = p.rs.err != nullptr;
    const int m = p.rs.m_slots;
    if (p.variant == 1 || p.variant == 2) {
        if (p.ignore_worst) return cudaErrorInvalidValue; // the two heuristics are alternatives
        return pme ? launch_k<true, false, 0, true, -1, ES, EH>(p, s) : launch_k<false, false, 0, true, -1, ES, EH>(p, s);
    }
    if (p.ignore_worst) {
        if (pme) return launch_k<true, true, 0, false, -1, ES, EH>(p, s);
        if (m == 8) return launch_k<false, true, 8, false, -1, ES, EH>(p, s);
        if (m == 16) return launch_k<false, true, 16, false, -1, ES, EH>(p, s);
        return launch_k<false, true, 0, false, -1, ES, EH>(p, s);
    }
    if (pme) return launch_k<true, false, 0, false, -1, ES, EH>(p, s);
    if (m == 4) return launch_k<false, false, 4, false, -1, ES, EH>(p, s);
    if (m == 8) return launch_tuned<8, ES, EH>(p, s);
    if (m == 16) return launch_tuned<16, ES, EH>(p, s);
    return launch_k<false, false, 0, false, -1, ES, EH>(p, s);
}

cudaError_t launch_t6_replay(const T6Params &p, cudaStream_t s) {
    if (p.N <= 0 || p.T <= 0) return cudaSuccess;
    if (!p.escratch) return launch_replay_es<false, false>(p, s);
    return p.ehist ? launch_replay_es<true, true>(p, s) : launch_replay_es<true, false>(p, s);
}

// getPose (TOA.cpp:438-473): predict-only, state untouched
__global__ void t6_get_pose_kernel(int64_t N, double dt, double accel_noise, const double *x,
                                   const double *P, double *x_pred, double *P_full) {
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= N) return;
    Sym<6> S;
#pragma unroll
    for (int k = 0; k < Sym<6>::SZ; ++k) S.a[k] = P[(int64_t)k * N + f];
    t6_predict_cov(S, dt, accel_noise);
    if (x_pred) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            // velocity is always 0 at the start of a step, so F x = x
            x_pred[(int64_t)k * N + f] = x[(int64_t)k * N + f];
            x_pred[(int64_t)(3 + k) * N + f] = 0.0;
        }
    }
    if (P_full) {
#pragma unroll
        for (int i = 0; i < 6; ++i)
#pragma unroll
            for (int j = 0; j < 6; ++j) P_full[(int64_t)(i * 6 + j) * N + f] = S.get(i, j);
    }
}

cudaError_t launch_t6_get_pose(int64_t N, double dt, double accel_noise, const double *x,
                               const double *P, double *x_pred, double *P_pred_full, cudaStream_t s) {
    if (N <= 0) return cudaSuccess;
    t6_get_pose_kernel<<<(unsigned)((N + 127) / 128), 128, 0, s>>>(N, dt, accel_noise, x, P, x_pred,
                                                                  P_pred_full);
    return cudaGetLastError();
}

} // namespace kfpos
