// kfpos_kernels.cuh -- kernel parameter blocks and launch entry points shared
// between the kernels (*.cu) and the C-ABI layer (kfpos_api.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "kfpos_math.cuh"

namespace kfpos {


// Range stream of a replay: SoA [T][M][N] in `fmt`, optional per-ranging
// errorEstimation of the same shape.
struct RangeStream {
    const void *ranges;
    const double *err; // null -> err_scalar
    double err_scalar;
    int fmt;
    int m_slots;
};

// ---- error statistics with a summation order that depends on nothing but the filter index:
// partial c covers filters [128c, 128c + 128) -- one replay block -- summed by a fixed 128-leaf binary
// tree in shared memory; the partials are then folded by a pairwise tree over the partial index
// (launch_error_stats_tree).  Every replay kernel can leave the partials of its final state behind
// (params.truth / params.partials): the reduction is fused into the last step of the replay, and a
// shard that starts at a multiple of its power-of-two size is a complete subtree of the global tree, so
// the reduced result is BIT-IDENTICAL for 1, 2, 4 or 8 GPUs (kfpos_stats_allreduce).
constexpr int STATS_CHUNK = 128;
// v = {|e|^2, |e_xy|^2, 1, bad} of this thread's filter (zeros for a thread without one); `sh` = at least
// 4 * 128 doubles of shared memory nobody else is using any more; every thread of the block calls it
KF_DEV void block_stats_partial(const double (&v)[4], double *sh, double *partial_out) {
    const int t = threadIdx.x;
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 4; ++q) sh[q * STATS_CHUNK + t] = v[q];
    __syncthreads();
    for (int s = STATS_CHUNK / 2; s > 0; s >>= 1) {
        if (t < s) {
#pragma unroll
            for (int q = 0; q < 4; ++q) sh[q * STATS_CHUNK + t] += sh[q * STATS_CHUNK + t + s];
        }
        __syncthreads();
    }
    if (t < 4) partial_out[t] = sh[t * STATS_CHUNK];
}
KF_DEV void filter_error_terms(double px, double py, double pz, const double *truth, int64_t N, int64_t f, bool bad,
                               double (&v)[4]) {
    const double ex = px - truth[f], ey = py - truth[N + f], ez = pz - truth[2 * N + f];
    const double e2 = ex * ex + ey * ey + ez * ez;
    v[0] = v[1] = v[2] = 0.0;
    if (isfinite(e2)) {
        v[0] = e2;
        v[1] = ex * ex + ey * ey;
        v[2] = 1.0;
    }
    v[3] = bad ? 1.0 : 0.0;
}

// ---- per-epoch statistics (kfpos_batch_set_truth_traj): at every output row a replay kernel compiled with
// ES = true leaves, per 32-filter warp, the 6 values of kfpos_batch_epoch_stats summed by a fixed 32-leaf tree
// (level s = 16, 8, 4, 2, 1: lane i += lane i + s; lanes without a filter count as zeros) at
// escratch[(row * n_warps + f / 32) * 6].  The folds over the warp index and over ranks are stats_tree's.
constexpr int ES_W = 6;
// The 6 terms of one filter: e = position - truth (3 components; K8: z = tag height); S = the packed position
// block of the covariance the filter holds now (s00, s10, s11, s20, s21, s22; nd = 2: the x-y block, s2x unused).
// NEES = e^T S^-1 e by LDL^T in a fixed order; a non-positive or non-finite pivot excludes the filter from [4], [5].
template <int nd>
KF_DEV void epoch_terms(double ex, double ey, double ez, double s00, double s10, double s11, double s20, double s21,
                        double s22, bool bad, const Col &out) {
    // (no contraction into FMAs: a host can reproduce [0] and [1] bit for bit from the trajectory)
    const double exy = __dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey));
    const double e2 = __dadd_rn(exy, __dmul_rn(ez, ez));
    const bool fin = isfinite(e2);
    out[0] = fin ? e2 : 0.0;
    out[1] = fin ? exy : 0.0;
    out[2] = fin ? 1.0 : 0.0;
    out[3] = bad ? 1.0 : 0.0;
    const double d0 = s00;
    const double l10 = s10 / d0;
    const double d1 = s11 - l10 * s10;
    const double y1 = ey - l10 * ex;
    double nees = ex * ex / d0 + y1 * y1 / d1;
    bool pd = d0 > 0.0 && d0 < INFINITY && d1 > 0.0 && d1 < INFINITY;
    if (nd == 3) {
        const double l20 = s20 / d0;
        const double c = s21 - l20 * s10;
        const double l21 = c / d1;
        const double d2 = s22 - l20 * s20 - l21 * c;
        const double y2 = ez - l20 * ex - l21 * y1;
        nees += y2 * y2 / d2;
        pd = pd && d2 > 0.0 && d2 < INFINITY;
    }
    const bool ok = pd && isfinite(nees);
    out[4] = ok ? nees : 0.0;
    out[5] = ok ? 1.0 : 0.0;
}
KF_DEV void epoch_terms_zero(const Col &out) {
#pragma unroll
    for (int q = 0; q < ES_W; ++q) out[q] = 0.0;
}
// the warp's sum of the W terms in `v` (every lane of wmask calls it; wmask = the lanes with a filter, a prefix);
// W = 4: the Cramer-Rao terms of kfpos_crlb.cu
template <int W = ES_W>
KF_DEV void epoch_stats_flush(const Col &v, unsigned wmask, double *out) {
    const int lane = threadIdx.x & 31;
    double a[W];
#pragma unroll
    for (int q = 0; q < W; ++q) a[q] = v[q];
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        const bool has = lane + s < 32 && ((wmask >> (lane + s)) & 1u);
#pragma unroll
        for (int q = 0; q < W; ++q) {
            const double o = __shfl_down_sync(wmask, a[q], s);
            a[q] += has ? o : 0.0;
        }
    }
    if (lane == 0) {
#pragma unroll
        for (int q = 0; q < W; ++q) out[q] = a[q];
    }
}

// row `row` of the event kernels: the lanes of a warp may arrive on different paths -- reconverge, then sum
KF_DEV bool epoch_stats_row(const Col &v, unsigned wmask, double *es_out, int64_t row, int64_t n_warps) {
    __syncwarp(wmask);
    epoch_stats_flush(v, wmask, es_out + row * n_warps * ES_W);
    return false;
}

// ---- per-epoch error histograms (kfpos_batch_set_error_hist): a replay kernel compiled with EH = true (always
// with ES = true) bins one of the terms already in the column wherever it flushes a row of the statistics.
// Quantity (KFPOS_HIST_*): 0 = e^2 (v[0]), 1 = e_xy^2 (v[1]), counted when v[2] == 1; 2 = NEES (v[4]), counted
// when v[5] == 1 -- so a row's counts add up to its [2] (or [5]) of kfpos_batch_epoch_stats.  Bin k = the number
// of table entries <= the value (0 .. n_bins - 1); the table holds the squared edges for the error quantities, so
// no square root is taken.  The device table always has EH_MAX_BINS - 1 entries, padded with +inf (> every counted
// value).  Counts are integers: any order of the atomics gives the same result.
constexpr int EH_MAX_BINS = 256;
KF_DEV void epoch_hist_flush(const Col &v, unsigned wmask, unsigned long long *counts, const double *edges,
                             int quantity) {
    const int lane = threadIdx.x & 31;
    const bool nees = quantity == 2;
    const double x = nees ? v[4] : (quantity == 1 ? v[1] : v[0]);
    const bool ok = (nees ? v[5] : v[2]) == 1.0;
    // binary search with a trip count common to the warp: the lanes load from the read-only cache side by side
    int k = 0;
#pragma unroll
    for (int s = EH_MAX_BINS / 2; s > 0; s >>= 1)
        if (__ldg(edges + k + s - 1) <= x) k += s;
    // one atomic per distinct bin of the warp; the lanes that count nothing form the key -1 and add nothing
    const int key = ok ? k : -1;
    const unsigned peers = __match_any_sync(wmask, key);
    if (ok && lane == __ffs(peers) - 1) atomicAdd(counts + k, (unsigned long long)__popc(peers));
}

struct T6Params {
    AnchorTable anchors;
    RangeStream rs;
    int64_t N;
    int T;
    int ignore_worst;
    int variant, n_ignore, best_mode; // EKF-side NLOS variants (config_pos.xml; 0 = normal)
    double ignore_thr;
    double accel_noise;
    const double *dt;   // device [T], common to the batch
    const double *dt_f; // or null: per-filter SoA [T][N]; a value < 0 = this filter has no epoch t
    double *x;        // SoA [6][N]  (rows 3..5 stay 0)
    double *P;        // SoA [21][N] packed lower triangle
    int32_t *status;  // [N], OR-ed
    double *traj;     // SoA [T][3][N] or null
    int32_t *sel;     // SoA [T][N] or null
    unsigned long long *counters;
    const double *truth; // SoA [3][N] or null: leave the error partials of the final state in `partials`
    double *partials;    // [ceil(N / 128)][4]
    // per-epoch statistics (launchers pick the ES = true kernels when non-null): truth rows SoA [rows][3][N] and
    // the per-warp sums [rows][n_warps][6] of this launch's first output row
    const double *etruth;
    double *escratch;
    int64_t n_warps;
    // per-epoch error histogram (the launchers pick the EH = true twins of the ES kernels when non-null): counts
    // [rows][ebins] of this launch's first output row, the device edge table [EH_MAX_BINS - 1] (squared for the
    // error quantities, +inf behind the last edge) and the quantity (KFPOS_HIST_*).  Last in the struct: the offsets of the fields above stay.
    unsigned long long *ehist;
    const double *eedges;
    int equantity;
    int ebins;
};

struct MlParams {
    AnchorTable anchors;
    RangeStream rs;
    int64_t N;
    int use2d, variant, n_ignore, best_mode;
    int zero_tz, _pad; // ml2d_zero_tentative_z
    double start[3];
    double min_z, max_z; // output gate (config_pos.xml minZ / maxZ), active when max_z > min_z
    double *pos;     // SoA [3][N] or null
    double *cov;     // SoA [9][N] or null
    int32_t *iters;  // [N] or null
    int32_t *sel;    // SoA [2][N] or null
    int32_t *status; // [N] or null
    unsigned long long *counters;
    // straggler queues (kfpos_mlk.cu): two buffers of queue_cap 64-byte records + their counters;
    // launch_ml_solve points q_in / q_out at them launch by launch
    void *queue[2];
    int *queue_count; // device int[2]
    int queue_cap;
    const void *q_in;      // records this launch resumes / advances (RESUME and cooperative kernels)
    const int *q_in_count;
    void *q_out;           // where this launch parks; null = finish in place
    int *q_out_count;
    unsigned first_cap;    // Newton iterations a solve gets in this launch before it is parked
    int coop_min, coop_max; // queue lengths [min, max) for which a cooperative launch does its work
    // exact-order solver (kfpos_exact.cu): kfpos_config.ml_exact_order, and the queue of epoch indices
    // whose residual order the fast solver found too close to a tie to decide (variant 1)
    int exact_mode;
    int xq_cap;
    int32_t *xq;
    int *xq_count;
    // scratch of the warp-per-epoch BestGroup kernels (parked 3-D subset solves), see ml_exact_scratch_bytes
    void *xw_scratch;
    size_t xw_scratch_bytes;
    int *stream_counter; // device int: the epoch counter of ml_stream3_kernel
};
constexpr int KFPOS_MAX_ANCHORS_DEV = 32;
// relative margin below which the fast solver does not trust its own order of two squared residuals
// (its positions agree with the reference's to ~1e-11: four orders of magnitude of room)
constexpr double ML_TIE_MARGIN = 1e-6;

// ---- sensor event streams (K8, T9).  The schedule (kind, dt) is common to the batch;
// `offset` is the first ROW (units of N elements) of the event's payload: rows of the
// range tensor for EV_TOA, rows of the f64 `sensors` tensor otherwise:
//   EV_PX4: integration_x, integration_y, integration_rot_z, integration_time_us, quality
//   EV_IMU: K8: ang_vel_z, lin_acc_x, lin_acc_y   T9: lin_acc_x, lin_acc_y, lin_acc_z
//   EV_MAG: mag_x, mag_y      EV_COMPASS: compass (rad)
// aux: EV_IMU covariances, common to the batch: K8: cov_acc[0],[1],[3],[4], cov_ang_vel[8];
// T9: cov_acc[0..8].  Mirrors kfpos_event of include/kfpos_b200.h.
enum { EV_TOA = 0, EV_PX4 = 1, EV_IMU = 2, EV_MAG = 3, EV_COMPASS = 4 };
struct EventDesc {
    int32_t kind;
    int32_t _pad;
    double dt;
    int64_t offset;
    double aux[9];
};

// constants of the five XML files + launch parameters (KF.cpp:766-844, node_pos.cpp:48-113)
struct K8Cfg {
    double accel_noise, jolt;
    double tag_z;                  // mUWBtagZ
    double px4_height, arm1, arm2; // mPX4flowHeight, mPX4FlowArmP1/P2
    double px4_cov_vel, px4_cov_gyro;
    double imu_cov_acc, imu_cov_gyro;
    double mag_offset, mag_cov;
    int imu_fix_acc, imu_fix_gyro;
    int variant, n_ignore, best_mode; // EKF-side NLOS variants (config_pos.xml; 0 = normal)
    int zero_tz;                      // ml2d_zero_tentative_z (App. B-1 as a zero-initialising build computes it)
    // the constructor without initialPosition (kfpos_config.ml_initial_position, KF.cpp:244-285): a filter whose
    // position is NaN initialises itself from its first epoch with rangings -- 2-D ML from (1, 1, tag height)
    // when use_fixed_height, else 3-D ML from (1, 1, 4), whose z becomes THIS filter's tag height (latch row 9)
    int ml_init, use_fixed_height;
};

struct K8Params {
    AnchorTable anchors;
    K8Cfg cfg;
    RangeStream rs;
    const double *sensors;   // SoA rows [R][N] f64
    const EventDesc *events; // device [n_events]
    int n_events;
    int64_t N;
    double *x;       // SoA [8][N]
    double *P;       // SoA [36][N] packed
    int32_t *status; // [N]
    double *latch;   // SoA [16][N]: px4 vx,vy,gz,cv | imu ax,ay,wz | mag angle | [8] dt carry | [9] tag height
    int32_t *has;    // [N] bit0 px4, bit1 imu, bit2 mag latched
    int *uninit;     // null, or a flag set by every filter that is still uninitialised when the launch ends
    double *latch_u; // batch-wide latched IMU covariances c00,c01,c11,cw: read from [0..3], written to [16..19]
    const double *dt_f; // null, or per-filter time steps SoA [n_events][N] (see T9Params)
    double *traj;    // SoA [n_toa][3][N] (px, py, theta) after each TOA event, or null
    unsigned long long *counters;
    const double *truth; // see T6Params
    double *partials;
    const double *etruth; // see T6Params (output rows = TOA events)
    double *escratch;
    int64_t n_warps;
    unsigned long long *ehist; // see T6Params
    const double *eedges;
    int equantity;
    int ebins;
};

cudaError_t launch_t6_replay(const T6Params &p, cudaStream_t s);
cudaError_t launch_k8_replay(const K8Params &p, cudaStream_t s);
cudaError_t launch_k8_get_pose(int64_t N, double dt, double accel_noise, double jolt, const double *x,
                               const double *P, double *x_pred, double *P_pred_full, cudaStream_t s);
cudaError_t launch_ml_solve(const MlParams &p, cudaStream_t s);
cudaError_t launch_ml_exact(const MlParams &p, bool queued, cudaStream_t s); // kfpos_exact.cu
size_t ml_exact_scratch_bytes(int64_t epochs);
int64_t ml_exact_scratch_epochs(int64_t N);
cudaError_t launch_selftest_ieee(int64_t n, const double *a, const double *b, double *div_fast, double *div_ieee,
                                 double *sqrt_fast, double *sqrt_ieee, int32_t *flags, cudaStream_t s);

struct T9Params {
    AnchorTable anchors;
    double accel_noise, jolt;
    RangeStream rs;
    const double *sensors;
    const EventDesc *events;
    int n_events;
    int64_t N;
    double *x;       // SoA [9][N]
    double *P;       // SoA [45][N] packed
    int32_t *status; // [N]
    double *latch;   // SoA rows 0..2: latched acceleration
    int32_t *has;    // [N] bit1: imu latched
    double *latch_u; // batch-wide latched 3x3 acceleration covariance: read from [0..8], written to [16..24]
    const double *dt_f; // null, or per-filter time steps SoA [n_events][N] replacing EventDesc::dt (< 0: the
                        // filter has no such event) -- the ragged epochs of kfpos_batch_replay_epochs
    int no_imu;      // host knowledge: no IMU sample latched and none in this schedule -> lean kernel
    int variant, n_ignore, best_mode; // EKF-side NLOS variants (config_pos.xml; 0 = normal)
    int ml_init;     // the constructor without initialPosition (TOAIMU.cpp:118-162), see K8Cfg::ml_init
    int *uninit;     // see K8Params
    double *traj;    // SoA [n_toa][3][N] or null
    unsigned long long *counters;
    const double *truth; // see T6Params
    double *partials;
    const double *etruth; // see T6Params (output rows = TOA events)
    double *escratch;
    int64_t n_warps;
    unsigned long long *ehist; // see T6Params
    const double *eedges;
    int equantity;
    int ebins;
};
cudaError_t launch_t9_replay(const T9Params &p, cudaStream_t s);
cudaError_t launch_t9_get_pose(int64_t N, double dt, double jolt, const double *x, const double *P, double *x_pred,
                               double *P_pred_full, cudaStream_t s);
cudaError_t launch_i32_to_f64(int64_t N, const int32_t *in, double *out, cudaStream_t s);

// full row-major SoA [n*n][N]  <->  packed lower-triangle SoA [n(n+1)/2][N]
cudaError_t launch_pack_cov(int n, int64_t N, const double *full, double *packed, cudaStream_t s);
cudaError_t launch_unpack_cov(int n, int64_t N, const double *packed, double *full, cudaStream_t s);

// predict-only pose poll (getPose)
cudaError_t launch_t6_get_pose(int64_t N, double dt, double accel_noise, const double *x,
                               const double *P, double *x_pred, double *P_pred_full, cudaStream_t s);

// error statistics (see block_stats_partial): partial[c][4] over the 128-filter chunks -- skipped when
// `truth` is null, i.e. when a replay kernel has already left them -- then the pairwise tree -> out[4]
// (position = rows 0,1 and row `zrow`, or the constant `zconst` when zrow < 0)
cudaError_t launch_error_stats(int64_t N, const double *x, int zrow, double zconst, const int32_t *status,
                               const double *truth, double *partials, double *out4, cudaStream_t s);
// pairwise tree over n vectors of 4 doubles (IN PLACE on `part`): level by level part[i] += part[i + stride]
cudaError_t launch_error_stats_tree(int64_t n, double *part, double *out4, cudaStream_t s);
// the same tree over n vectors of `width` (4 or 6) doubles, for `rows` rows at once: vector i of row r is at
// [r * row_stride + i * elem_stride]; the first level reads `src` and writes `part` (src == part: in place), the
// others work in `part`; out[r * width + q]
cudaError_t launch_stats_tree(int width, int64_t rows, int64_t n, const double *src, double *part, int64_t row_stride,
                              int64_t elem_stride, double *out, cudaStream_t s);

// getPose report in the publisher's layout (kfpos_misc.cu); model 1 = T6, 2 = K8, 3 = T9
// tagz: null, or the per-filter tag height replacing tag_z (K8 after a 3-D ML initialisation)
cudaError_t launch_pose_msg(int model, int64_t N, double tag_z, const double *tagz, const double *x_pred,
                            const double *P_pred_full, double *pose13, double *cov36, cudaStream_t s);
cudaError_t launch_fill(double *p, int64_t n, double v, cudaStream_t s);
// out[i] = sum of src[r * n + i] over r < n_ranks (the rank fold of the error histograms)
cudaError_t launch_sum_ranks_u64(int n_ranks, int64_t n, const unsigned long long *src, unsigned long long *out,
                                 cudaStream_t s);

// epoch assembler (kfpos_assemble.cu): N logs of L messages, SoA [L][N]
struct AssembleParams {
    int64_t N, L, max_epochs;
    int M, fix_b12;
    double first_dt;
    const uint8_t *anchor, *seq;
    const int32_t *range_mm;
    const double *err, *t;
    int32_t *tbl_r; // [rows][M][N], rows = 256 (as written) or 1 (fix_b12), pre-set to -1
    double *tbl_e;  // same shape, pre-set to 0
    int32_t *ranges_out;
    double *err_out, *dt_out;
    int32_t *n_epochs;
    double *t_out; // [max_epochs][N] or null: the time of every report (-1 = no such epoch)
};
cudaError_t launch_assemble(const AssembleParams &p, cudaStream_t s);

// stream merger (kfpos_assemble.cu): stream 0 = ranging reports, 1..4 = PX4 / IMU / MAG / COMPASS samples
struct MergeParams {
    int64_t N;
    int M, n_slots;
    int64_t L[5];
    const double *t_src[5];   // [L_k][N] arrival times; negative / NaN ends the stream
    const int32_t *ranges;    // [L_0][M][N]
    const double *err_src;    // [L_0][M][N] or null
    const double *src[5];     // k > 0: [L_k][rows_k][N]
    const int32_t *slot_kind; // device [n_slots]
    const int64_t *slot_row;  // device [n_slots]: first output row of the slot
    double first_dt;
    double *dt_f;             // [n_slots][N]
    int32_t *ranges_out;      // [range rows][N]
    double *err_out;          // [range rows][N] or null
    double *sensors_out;      // [sensor rows][N]
    int32_t *n_dropped;       // [N] or null
};
cudaError_t launch_merge(const MergeParams &p, cudaStream_t s);

cudaError_t launch_selftest_math(int64_t n, const double *x, double *rcp, double *rsq, double *sn, double *cs,
                                 cudaStream_t s);

// Monte Carlo input generator for K8 batches (kfpos_synth.cu)
struct SynthEvent {
    int32_t kind;
    int32_t global_index; // index of the event in the whole run (RNG counter)
    double t;             // time of the event, s
    int64_t offset;       // first output row (rows of `ranges` for EV_TOA, of `sensors` otherwise)
};
struct SynthK8Params {
    AnchorTable anchors;
    int64_t N, filter0;
    uint64_t seed;
    int M, n_events;
    double tag_z, sigma_r, t_end;
    const SynthEvent *events; // device [n_events]
    int32_t *ranges;          // SoA [rows][N] int32 mm
    double *sensors;          // SoA [rows][N]
    double *x0;               // SoA [8][N] or null
    double *truth_end;        // SoA [3][N] or null: (x, y, tag z) at t_end
};
cudaError_t launch_synth_k8(const SynthK8Params &p, cudaStream_t s);
// truth of the same workload at host times t[0..n_times): SoA [n_times][3][N] = (x, y, tag_z)
struct SynthTruthParams {
    int64_t N, filter0;
    uint64_t seed;
    int n_times;
    double tag_z;
    const double *t; // device [n_times]
    double *truth;
};
cudaError_t launch_synth_k8_truth(const SynthTruthParams &p, cudaStream_t s);
// ranging epochs of the same truth for [T][M][N] range logs (kfpos_synth_toa_ranges); a launch covers at most
// SYNTH_TOA_T epochs, whose times travel in the parameter block (8 KB of the 32 KB it may hold)
constexpr int SYNTH_TOA_T = 1024;
constexpr int SYNTH_TOA_OBSTACLES = 32; // KFPOS_MAX_OBSTACLES
struct SynthObstacle {                  // kfpos_obstacle
    double lo[3], hi[3], excess_per_m, spread, p_loss;
};
struct SynthToaParams {
    AnchorTable anchors;
    int64_t N, filter0;
    uint64_t seed;
    int M, n_epochs;
    uint32_t epoch0; // global index of epoch 0 of this launch (RNG counter)
    double tag_z, sigma_r, p_missing, p_nlos, nlos_mean;
    void *ranges; // SoA [n_epochs][M][N], int32 or uint16 mm
    double t[SYNTH_TOA_T];
    uint32_t *nlos; // SoA [n_epochs][N] NLOS bit masks, or null (last: the offsets of the fields above stay)
    int n_obstacles; // boxes of kfpos_synth_toa_ranges_geo, 0: none (after the fields above, which keep their offsets)
    SynthObstacle obstacles[SYNTH_TOA_OBSTACLES];
};
cudaError_t launch_synth_toa(const SynthToaParams &p, bool u16, cudaStream_t s); // u16: uint16 mm, else int32 mm

// selection scores against the NLOS truth (kfpos_score.cu, kfpos_batch_score_selection): counts [n_rows][8],
// zeroed by the caller.  How `sel` [n_rows][N] is read: SCORE_NONE not at all (nothing dropped), SCORE_LOO the
// ignored slot or -1, SCORE_MASK the bit mask of the slots used.
constexpr int SCORE_COLS = 8;
enum { SCORE_NONE = 0, SCORE_LOO = 1, SCORE_MASK = 2 };
struct ScoreParams {
    const void *ranges;   // SoA [n_rows][M][N] in fmt
    const int32_t *sel;   // SoA [n_rows][N], or null with SCORE_NONE
    const uint32_t *nlos; // SoA [n_rows][N], or null: no ranging is NLOS
    unsigned long long *counts;
    int64_t N, n_rows;
    int M, fmt, mode;
};
cudaError_t launch_score_selection(const ScoreParams &p, cudaStream_t s);

// The rangings of filter f in one epoch of a SoA log: bit a set when ranging a is present, the replay's rule of
// convert_epoch (value > 0; NaN is not).  base = the index of (row, anchor 0, f), m anchors of stride N.
template <int FMT>
KF_DEV unsigned present_mask(const void *ranges, int64_t base, int m, int64_t N) {
    unsigned present = 0u;
#pragma unroll 8
    for (int a = 0; a < m; ++a) {
        const int64_t i = base + (int64_t)a * N;
        bool on;
        if (FMT == 0) on = __ldg(reinterpret_cast<const double *>(ranges) + i) > 0.0; // false for NaN
        else if (FMT == 1) on = __ldg(reinterpret_cast<const int32_t *>(ranges) + i) > 0;
        else on = __ldg(reinterpret_cast<const uint16_t *>(ranges) + i) != 0;
        present |= (unsigned)on << a;
    }
    return present;
}
// The rangings filter f kept in row r, decoded from `sel` (SoA [rows][N]) as the batch's configuration wrote it
// (mode SCORE_*): the one place that reads a selection, for the scorer and the Cramer-Rao bound alike.  May name
// absent slots (SCORE_MASK).
KF_DEV unsigned used_mask(unsigned present, const int32_t *sel, int64_t r, int64_t N, int64_t f, int mode) {
    unsigned used = present;
    if (mode == SCORE_LOO) {
        const int s = __ldg(sel + r * N + f);
        if (s >= 0 && s < 32) used &= ~(1u << s);
    } else if (mode == SCORE_MASK) {
        used = (unsigned)__ldg(sel + r * N + f);
    }
    return used;
}

// Cramer-Rao bound of the position per epoch (kfpos_crlb.cu, kfpos_batch_crlb): for each (filter, row) the four
// terms {tr J^-1, (J^-1)_xx + (J^-1)_yy, 1, 0} (or {0, 0, 0, 1} without a bound) of the Fisher information J of
// the set `set` (KFPOS_CRLB_*), summed per 32-filter warp by epoch_stats_flush<4> into
// partials[(row * n_warps + f / 32) * 4]; the caller folds them over the warp index with launch_stats_tree(4, ...).
constexpr int CRLB_W = 4;
enum { CRLB_PRESENT = 0, CRLB_LOS = 1, CRLB_USED = 2 };
struct CrlbParams {
    AnchorTable anchors;
    const double *truth;  // SoA [n_rows][3][N]
    const void *ranges;   // SoA [n_rows][M][N] in fmt
    const double *var;    // SoA [n_rows][M][N] true ranging variances, or null: 1 / w_scalar for all
    const int32_t *sel;   // SoA [n_rows][N] read with sel_mode (KFPOS_CRLB_USED), else null
    const uint32_t *nlos; // SoA [n_rows][N] (KFPOS_CRLB_LOS), else null
    double *partials;     // [n_rows][n_warps][4]
    double w_scalar;      // 1 / var_scalar
    int64_t N, n_rows, n_warps;
    int M, fmt, set, sel_mode, dim; // dim: 3, or 2 (K8, ML use2d: x-y information, known height)
};
cudaError_t launch_crlb(const CrlbParams &p, cudaStream_t s);

// DFMA-only microbenchmark on the current device (the FP64 roofline denominator)
cudaError_t measure_fp64_peak(double *flops_per_s);

} // namespace kfpos
