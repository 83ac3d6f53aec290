/*
 * kfpos_b200.h -- C ABI of libkfpos_b200.so: batched, B200-native (sm_100a)
 * replacement for the numeric filter core of GTEC-UDC/roskfpos.
 *
 * One opaque handle = a BATCH of N independent filters of one model and one
 * configuration on one GPU.  Each entry point cites the reference interface it
 * replaces (paths relative to /root/reference/src/kfpos/):
 *
 *   PositionEstimationAlgorithm      algorithms/PositionEstimationAlgorithm.h:8-37
 *   MLLocation                       algorithms/MLLocation.h:25-76
 *   KalmanFilterTOA (T6)             algorithms/KalmanFilterTOA.h:18-55
 *   KalmanFilter (K8)                algorithms/KalmanFilter.h:28-134
 *   KalmanFilterTOAIMU (T9)          algorithms/KalmanFilterTOAIMU.h:15-79
 *   sole caller                      publishers/Posgenerator.cpp:99-141,476-496,510-548
 *
 * Conventions
 *  - every function returns 0 (KFPOS_OK) or a negative kfpos_status code and
 *    never throws; per-filter numerical events (singular solve, NaN, too few
 *    rangings) are reported in the per-filter `status` words, not the return code;
 *  - "SoA [k][N]" = k rows of N contiguous values, filter index fastest;
 *  - data pointers may be HOST or DEVICE pointers (the library asks the CUDA
 *    runtime which); device pointers must belong to the batch's device;
 *  - `stream` is a cudaStream_t passed as void* (NULL = the legacy default
 *    stream); work is enqueued on it, calls taking host pointers synchronise it
 *    before returning;
 *    the small arrays declared as HOST arrays (dt, event schedules, ...) do not count;
 *  - calls on one handle must be serialised by the caller (the reference is
 *    single-threaded: publishers/node_pos.cpp:176-181); handles are independent;
 *  - there is NO CPU fallback: without a usable CUDA device every call fails
 *    with KFPOS_ERR_CUDA.
 */
#ifndef KFPOS_B200_H
#define KFPOS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KFPOS_ABI_VERSION 1
#define KFPOS_MAX_ANCHORS 32 /* anchor slots per epoch (reference MAX_NUM_ANCS = 64; PG.h:102) */

typedef struct kfpos_batch kfpos_batch;

/* return codes */
enum kfpos_status_code {
    KFPOS_OK = 0,
    KFPOS_ERR_INVALID = -1,     /* bad argument / wrong model for this call   */
    KFPOS_ERR_CUDA = -2,        /* CUDA runtime error or no device            */
    KFPOS_ERR_NOMEM = -3,       /* allocation failed                          */
    KFPOS_ERR_NOT_READY = -4,   /* anchors / state not set yet                */
    KFPOS_ERR_UNSUPPORTED = -5, /* configuration outside the kernels' domain  */
    KFPOS_ERR_PARSE = -6        /* malformed XML configuration string         */
};

/* models = the factory ids of PosGenerator::setAlgorithm (PG.cpp:510-538) */
enum kfpos_model {
    KFPOS_MODEL_ML = 0, /* MLLocation                                  */
    KFPOS_MODEL_T6 = 1, /* KalmanFilterTOA: 6-state, rangings only     */
    KFPOS_MODEL_K8 = 2, /* KalmanFilter: 8-state, UWB+PX4Flow+IMU+mag  */
    KFPOS_MODEL_T9 = 3  /* KalmanFilterTOAIMU: 9-state, rangings+accel */
};

/* range tensor element formats; a value <= 0 means "no ranging" (TOA.cpp:50) */
enum kfpos_range_fmt {
    KFPOS_FMT_F64_M = 0,  /* double, metres (what newTOAMeasurement receives)              */
    KFPOS_FMT_I32_MM = 1, /* int32 millimetres, the PosGenerator table format (PG.cpp:213) */
    KFPOS_FMT_U16_MM = 2  /* uint16 millimetres (ranges < 65.5 m)                          */
};

/* per-filter status bits (OR-ed over the steps since the last set_state) */
#define KFPOS_ST_OK 0
#define KFPOS_ST_NO_MEAS 1   /* a TOA update had no valid ranging                           */
#define KFPOS_ST_ML_FEW 2    /* inner ML had < 3/4 rangings and returned its start point     */
#define KFPOS_ST_SINGULAR 4  /* a solve hit a singular matrix: update skipped (TOA.cpp:151)  */
#define KFPOS_ST_NAN 8       /* non-finite state after an update                             */
#define KFPOS_ST_ML_NAN 16   /* T6 NaN guard fired (TOA.cpp:270-272)                         */
#define KFPOS_ST_MAXITER 32  /* IEKF used all iterations without meeting the break test      */
#define KFPOS_ST_ASYM_R 64   /* K8 IMU covariance block not symmetric (cov[1] != cov[3])     */
#define KFPOS_ST_Z_GATE 128  /* ML: estimated z outside [min_z, max_z] (config_pos.xml:22-25) */
#define KFPOS_ST_UNINIT 256  /* K8 / T9 with ml_initial_position: an event met the filter while its position
                                was still NaN and ended in the ML-initialisation branch (KF.cpp:244-285,
                                TOAIMU.cpp:118-162): no predict, no update                        */

/* ML variants (MLLocation.h:5-7) and best-group criteria (MLLocation.h:10-11) */
#define KFPOS_ML_VARIANT_NORMAL 0
#define KFPOS_ML_VARIANT_IGNORE_N 1
#define KFPOS_ML_VARIANT_BEST 2
#define KFPOS_BEST_MODE_XYZ 0
#define KFPOS_BEST_MODE_Z 1

/*
 * Flat configuration: the constructor arguments of the four classes plus the
 * attributes of the five XML files KalmanFilter::loadConfigurationFiles reads
 * (KF.cpp:749-893).  Field comments give the reference name.
 */
typedef struct kfpos_config {
    /* constructor / launch parameters (node_pos.cpp:48-113) */
    double accel_noise;           /* accelerationNoise (all KFs)                    */
    double jolt;                  /* jolt (K8, T9)                                  */
    double initial_angle;         /* initialAngle (K8)                              */
    int32_t ignore_worst_anchor;  /* ignoreWorstAnchorMode (T6)                     */
    int32_t ml2d_zero_tentative_z; /* 0 (default): the 2-D ML solver's tentative cost uses z = start z
                                      (SURVEY App. B-1, the evident intent of ML.cpp:64,102-106);
                                      1: z = 0, what a build of the reference that zero-initialises
                                      the uninitialised `tentativePos` computes (K8, 2-D ML)        */
    double ignore_cost_threshold; /* ignoreCostThreshold (T6)                       */
    /* MLLocation ctor (ML.h:30) + config_pos.xml <algorithm .../>.  For T6, K8 and T9 batches variant /
     * num_ignored_rangings / best_mode select the EKF-side NLOS variants that README.md:85-108
     * documents (the reference implements them only in MLLocation): the ML estimator, started at
     * the predicted position, picks the rangings (variant 1: drop the N with the largest residual,
     * ML.cpp:307-347; variant 2: keep the best group, ML.cpp:351-414 -- 4 anchors for the 3-D
     * solves of T6 / T9, the "best 3 anchors" of the documentation for K8's 2-D solve) and the iterated update
     * runs on the survivors; for T6 `sel` of kfpos_batch_replay_toa holds the slot mask used.     */
    int32_t use2d;                /* use2d                                          */
    int32_t variant;              /* variant                                        */
    int32_t num_ignored_rangings; /* numIgnoredRangings                             */
    int32_t best_mode;            /* bestMode                                       */
    double min_z, max_z;          /* minZ, maxZ: ML output gate, active when max_z >
                                     min_z: estimates outside get KFPOS_ST_Z_GATE    */
    double ml_start[3];           /* previousEstimation: (1,1,4) by default         */
    /* config_uwb.xml <uwb .../>  (KF.cpp:793-800) */
    int32_t use_fixed_height;     /* useFixedHeight                                 */
    int32_t tag_id;               /* tagId (loaded, never read)                     */
    double fixed_height;          /* fixedHeight -> mUWBtagZ                        */
    /* config_px4flow.xml <px4flow .../>  (KF.cpp:766-779) */
    int32_t px4_use_fixed_sensor_height; /* useFixedSensorHeight (never read)       */
    int32_t ml_exact_order;       /* ML batches: 0 (default) BestGroup epochs are solved in the reference's
                                     exact operation order (IEEE division / square root, no fused
                                     multiply-adds: selection indices, iteration counts and values are bit-
                                     identical to a CPU build of MLLocation.cpp's arithmetic), IgnoreN
                                     epochs whose residual order is within 1e-6 of a tie are re-decided
                                     the same way; 1: every epoch of every variant in exact order;
                                     -1: fast formulation only (selection may flip on rounding-level ties) */
    double px4_sensor_height;     /* sensorHeight -> mPX4flowHeight                 */
    double px4_arm_p0;            /* armP0 -> mPX4FlowArmP1                         */
    double px4_arm_p1;            /* armP1 -> mPX4FlowArmP2                         */
    double px4_sensor_init_angle; /* sensorInitAngle (never read)                   */
    double px4_cov_velocity;      /* covarianceVelocity                             */
    double px4_cov_gyro_z;        /* covarianceGyroZ                                */
    /* config_imu.xml <imu .../>  (KF.cpp:815-824) */
    int32_t imu_use_fixed_cov_acc;    /* useFixedCovarianceAcceleration             */
    int32_t imu_use_fixed_cov_gyro_z; /* useFixedCovarianceAngularVelocityZ         */
    double imu_cov_acc;               /* covarianceAcceleration                     */
    double imu_cov_gyro_z;            /* covarianceAngularVelocityZ                 */
    /* config_mag.xml <mag .../>  (KF.cpp:839-844) */
    double mag_angle_offset;      /* angleOffset                                    */
    double mag_cov;               /* covarianceMag                                  */
    /* The constructors WITHOUT initialPosition (KF.cpp:6-32, TOAIMU.cpp:6-24; what PosGenerator builds
     * when the launch file leaves useStartPosition at 0, PG.cpp:519-528).  0 (default): fixed initial
     * position, x0 of kfpos_batch_set_state is the state.  1 (K8, T9): a filter whose x0 position is
     * NaN is UNINITIALISED -- every event updates the sensor latches and the filter's clock only,
     * until an epoch with rangings arrives: its position then comes from MLLocation (K8: 2-D from
     * (1, 1, fixedHeight) when use_fixed_height, else 3-D from (1, 1, 4) and the estimated z becomes
     * THIS filter's tag height; T9: 3-D from (1, 1, 4)) and the 2x2 x-y block of the all-zero
     * covariance from the ML covariance (KF.cpp:244-285, TOAIMU.cpp:118-162); the epoch performs no
     * update.  As written: fewer than 3 / 4 rangings initialise the filter AT the start point with
     * P = 0 (KFPOS_ST_ML_FEW; the reference then throws on the empty covariance matrix); a failed
     * solve leaves the filter uninitialised (KFPOS_ST_SINGULAR).  T6's branch (TOA.cpp:90-108) is not
     * offered: it leaves a NON-symmetric covariance behind (SURVEY App. B-6).                      */
    int32_t ml_initial_position;
    int32_t _reserved0;
} kfpos_config;

/* Fills the defaults the reference uses when an attribute/param is absent (all 0;
 * ml_start = (1,1,4), PG.cpp:531). */
void kfpos_config_default(kfpos_config *cfg);

/* Parses ONE of the reference's XML configuration strings (the content of
 * config_uwb / config_px4flow / config_imu / config_mag / config_pos .xml) and
 * overwrites the matching fields; unknown elements are ignored, missing
 * attributes get the reference default 0.  Replaces KF.cpp:749-893.           */
int kfpos_config_load_xml(kfpos_config *cfg, const char *xml);

const char *kfpos_strerror(int code);
int kfpos_abi_version(void);

/* ------------------------------------------------------------------ lifetime
 * Replaces the constructors + init() (TOA.cpp:5-40, KF.cpp:6-62,
 * TOAIMU.cpp:6-46, ML.cpp:3-22).  State is zero, covariance zero, no latched
 * sensor samples -- the fixed-initial-position constructors (SURVEY App. B-7). */
int kfpos_batch_create(kfpos_batch **out, int device, int model, int64_t n_filters,
                       const kfpos_config *cfg);
void kfpos_batch_destroy(kfpos_batch *b);
int64_t kfpos_batch_size(const kfpos_batch *b);
int kfpos_batch_state_dim(const kfpos_batch *b); /* 3 (ML), 6, 8, 9 */

/* Anchor table shared by the batch: the `beacons` argument of newTOAMeasurement
 * (PEA.h:16; built by PG.cpp:476-496 from the anchor index order).  xyz [n][3]. */
int kfpos_batch_set_anchors(kfpos_batch *b, int n_anchors, const double *xyz);

/* State and covariance.  x: SoA [n][N]; P: SoA [n*n][N]
 * row-major full matrix, or NULL for the reference's initial P0 = 0.
 * set_state RE-INITIALISES the filters (it is the constructor's initial position): latched sensor
 * samples, their flags and the status words are cleared.  A checkpoint of a running K8 / T9 batch is
 * get_state + kfpos_batch_get_latches, restored by set_state followed by kfpos_batch_set_latches.
 * (T6 ignores rows 3..5 of x -- the velocity is zero at the start of every step, TOA.cpp:110-112 --
 * and get_state returns them as zeros.)
 * State layouts: T6 [px,py,pz,vx,vy,vz]  (v is always 0: TOA.cpp:110-112)
 *                K8 [px,py,vx,vy,ax,ay,theta,omega]  (a always 0: KF.cpp:287-291)
 *                T9 [px,py,pz,vx,vy,vz,ax,ay,az]     (a always 0: TOAIMU.cpp:165-168)
 * Also clears the per-filter status, selection and latched-sensor flags.      */
int kfpos_batch_set_state(kfpos_batch *b, const double *x, const double *P, void *stream);
int kfpos_batch_get_state(kfpos_batch *b, double *x, double *P, int32_t *status, void *stream);

/* The rest of a running K8 / T9 filter: the members the sensor callbacks latch (KF.h:92-130,
 * KalmanFilterTOAIMU.h:60-70).  latch: SoA [16][N] -- K8 rows 0..3 lastPX4FlowMeasurement (vx, vy,
 * gyroZ, covarianceVelocity), 4..6 lastImuMeasurement (ax, ay, angularVelocityZ), 7 lastMagMeasurement
 * angle, 8 time carried over from PX4 frames of quality 0 (KF.cpp:111-113), 9 this filter's tag height
 * (mUWBtagZ, see ml_initial_position); T9 rows 0..2 latched acceleration.  has: [N] bit0 PX4, bit1 IMU,
 * bit2 magnetometer sample latched.  latch_u: 16 doubles common to the batch (the IMU covariances of
 * the last sample: K8 c00, c01, c11, cw; T9 the 3x3 matrix row-major).  Any pointer may be NULL.
 * Host or device pointers.                                                                        */
int kfpos_batch_get_latches(kfpos_batch *b, double *latch, int32_t *has, double *latch_u, void *stream);
int kfpos_batch_set_latches(kfpos_batch *b, const double *latch, const int32_t *has, const double *latch_u,
                            void *stream);

/* ---------------------------------------------------------------- EKF steps
 * One newTOAMeasurement per filter (PEA.h:16; TOA.cpp:43-61, KF.cpp:64-97,
 * TOAIMU.cpp:49-73): predict with `dt` (the reference measures it with
 * steady_clock, SURVEY App. B-8), inner ML solve, iterated update.
 * ranges: SoA [n_anchors][N] in `fmt`; err_var: per-ranging errorEstimation SoA
 * [n_anchors][N] or NULL to use the scalar `err_scalar` for every ranging.     */
int kfpos_batch_step_toa(kfpos_batch *b, double dt, const void *ranges, int fmt,
                         double err_scalar, const double *err_var, void *stream);

/* T steps in ONE persistent kernel with state and covariance held on chip.
 * dt: HOST array [T]; ranges: SoA [T][n_anchors][N]; err_var NULL or same shape.
 * Optional outputs (NULL to skip): traj SoA [T][3][N] position after each step;
 * sel SoA [T][N] int32 anchor slot ignored by T6's leave-one-out, -1 if none.   */
int kfpos_batch_replay_toa(kfpos_batch *b, int n_steps, const double *dt, const void *ranges,
                           int fmt, double err_scalar, const double *err_var, double *traj,
                           int32_t *sel, void *stream);

/* The same persistent replay with PER-FILTER time steps, for logs assembled by
 * kfpos_assemble_epochs (every tag has its own report times).  dt_per_filter: SoA [T][N];
 * a value < 0 means "filter f has no epoch t": neither predict nor update, its trajectory row
 * repeats the current position.  T6, and K8 / T9 as ranging-only schedules (their general
 * kernel instantiation; latched sensor samples of earlier event calls take part as usual);
 * traj rows as in kfpos_batch_replay_toa / kfpos_batch_replay_events.                  */
int kfpos_batch_replay_epochs(kfpos_batch *b, int n_steps, const double *dt_per_filter, const void *ranges,
                              int fmt, double err_scalar, const double *err_var, double *traj, void *stream);

/* newPX4FlowMeasurement (PEA.h:15; KF.cpp:100-133).  K8 only.  SoA [N] each.
 * Filters whose quality is 0 skip the event; its dt is carried to their next one
 * (the reference returns before reading its clock, KF.cpp:111-113).              */
int kfpos_batch_step_px4(kfpos_batch *b, double dt, const double *integration_x,
                         const double *integration_y, const double *integration_rot_z,
                         const double *integration_time_us, const int32_t *quality, void *stream);
/* newIMUMeasurement (PEA.h:17; KF.cpp:137-176, TOAIMU.cpp:76-92).  K8 and T9.
 * ang_vel, lin_acc: SoA [3][N]; cov_ang_vel, cov_acc: HOST arrays of 9 doubles
 * (row-major 3x3) applying to the whole batch, or NULL (= 0).  T9's IMU rows are
 * the restatement of SURVEY App. B-5 (the reference throws on its first IMU sample). */
int kfpos_batch_step_imu(kfpos_batch *b, double dt, const double *ang_vel,
                         const double *cov_ang_vel, const double *lin_acc, const double *cov_acc,
                         void *stream);
/* newMAGMeasurement (PEA.h:18; KF.cpp:179-193).  K8 only.  mag: SoA [3][N].     */
int kfpos_batch_step_mag(kfpos_batch *b, double dt, const double *mag, void *stream);
/* newCompassMeasurement (PEA.h:19; KF.cpp:195-221).  K8 only.  compass: [N] rad. */
int kfpos_batch_step_compass(kfpos_batch *b, double dt, const double *compass, void *stream);

/* A whole sensor-event schedule in ONE persistent kernel (K8, T9): the batched form
 * of the reference's callback sequence.  The schedule (kind, dt) is common to the
 * batch, the payload is per filter.  `offset` = first ROW (units of N elements) of
 * the event's payload: rows of `ranges` for KFPOS_EV_TOA (row = step * n_anchors),
 * rows of the f64 tensor `sensors` (SoA [R][N]) otherwise:
 *   KFPOS_EV_PX4     integration_x, integration_y, integration_rot_z, integration_time_us, quality
 *   KFPOS_EV_IMU     K8: ang_vel_z, lin_acc_x, lin_acc_y     T9: lin_acc_x, lin_acc_y, lin_acc_z
 *   KFPOS_EV_MAG     mag_x, mag_y            KFPOS_EV_COMPASS  compass (rad)
 * aux (KFPOS_EV_IMU, batch-wide covariances): K8: cov_acc[0], cov_acc[1], cov_acc[3],
 * cov_acc[4], cov_ang_vel[8];  T9: cov_acc[0..8].
 * events: HOST array.  traj (optional): SoA [n_toa][3][N] = (px, py, theta) for K8,
 * (px, py, pz) for T9, after each TOA event.                                       */
enum kfpos_event_kind {
    KFPOS_EV_TOA = 0,
    KFPOS_EV_PX4 = 1,
    KFPOS_EV_IMU = 2,
    KFPOS_EV_MAG = 3,
    KFPOS_EV_COMPASS = 4
};
typedef struct kfpos_event {
    int32_t kind;
    int32_t _pad;
    double dt;
    int64_t offset;
    double aux[9];
} kfpos_event;
int kfpos_batch_replay_events(kfpos_batch *b, int n_events, const kfpos_event *events, const void *ranges,
                              int fmt, double err_scalar, const double *err_var, const double *sensors,
                              int64_t sensor_rows, double *traj, void *stream);

/* The same with PER-FILTER time steps: dt_per_filter SoA [n_events][N] replaces kfpos_event::dt; a
 * value < 0 means "filter f has no such event" (nothing is latched, predicted or updated; a TOA slot's
 * trajectory row repeats the current state).  This is how N tags whose sensor messages arrive in
 * different orders and numbers share one launch: kfpos_merge_streams lays their streams onto a common
 * schedule (K8 / T9, general kernel instantiation).                                              */
int kfpos_batch_replay_events_ragged(kfpos_batch *b, int n_events, const kfpos_event *events,
                                     const double *dt_per_filter, const void *ranges, int fmt, double err_scalar,
                                     const double *err_var, const double *sensors, int64_t sensor_rows,
                                     double *traj, void *stream);

/* getPose (PEA.h:14; TOA.cpp:438-473, KF.cpp:709-747, TOAIMU.cpp:476-510):
 * predict-only to `dt` after the last update, state untouched.  x_pred SoA
 * [n][N], P_pred SoA [n*n][N] (either may be NULL).                              */
int kfpos_batch_get_pose(kfpos_batch *b, double dt, double *x_pred, double *P_pred, void *stream);

/* getPose as the publisher consumes it (PosGenerator::publishPositionReport, Posgenerator.cpp:
 * 385-470, after stateToPose TOA.cpp:159-183 / KF.cpp:324-363 / TOAIMU.cpp:198-241): the batched
 * output formatter for downstream consumers.  pose13 SoA [13][N]: position x,y,z (K8: z = the
 * configured tag height), orientation quaternion x,y,z,w (K8: rotation by theta about z; T6/T9:
 * all 0 as the reference leaves it), linear speed x,y,z, angular speed x,y,z (T9 reports its
 * ACCELERATION there, TOAIMU.cpp:213-215).  cov36 SoA [36][N]: the 36 values copied into
 * geometry_msgs/PoseWithCovariance.covariance, cov36[i] = covarianceMatrix(i) in Armadillo's
 * column-major linear order (T9's matrix is 9x9: its first four columns).  Either output may be
 * NULL.  Returns KFPOS_ERR_NOT_READY until a measurement has been processed after
 * set_state(x, NULL) (getPose returns false, KF.cpp:713-717).                           */
int kfpos_batch_get_pose_msg(kfpos_batch *b, double dt, double *pose13, double *cov36, void *stream);

/* ----------------------------------------------------------------------- ML
 * newTOAMeasurement + getPose of MLLocation (ML.cpp:421-486) for N independent
 * epochs; variant / use2d / num_ignored_rangings / best_mode / ml_start from the
 * batch config.  ranges SoA [n_anchors][N].  Outputs (NULL to skip):
 * pos SoA [3][N]; cov SoA [9][N] (3x3 row-major, the 2x2 block top-left when
 * use2d); iters [N] total Newton iterations; sel SoA [2][N]: row 0 = bit mask of
 * the anchor slots used by the final solve, row 1 = #dropped (variant 1) or the
 * subset index in prev_permutation order (variant 2); status [N].
 * Variant 2 runs in the exact-order solver (ml_exact_order >= 0) with one warp per epoch; the 3-D
 * scan parks its long subset solves in device scratch that the batch allocates on first use
 * (~190 MB, independent of N: epochs go through in chunks of 131072).             */
int kfpos_batch_ml_solve(kfpos_batch *b, const void *ranges, int fmt, double err_scalar,
                         const double *err_var, double *pos, double *cov, int32_t *iters,
                         int32_t *sel, int32_t *status, void *stream);

/* --------------------------------------------------------- epoch assembler
 * The ranging aggregation of PosGenerator (publishers/Posgenerator.cpp:143-281,476-507) for N
 * independent, time-sorted ranging logs (one tag each; the tagId filter of :203 is the caller's):
 * rangings are grouped by `seq` into epochs; an epoch is emitted when the next sequence number
 * starts and when the one-shot 50 ms timer (Posgenerator.h:77) expires after the last ranging
 * of a sequence (the row stays open: late rangings of the same seq are added and the row is
 * emitted again, as the reference does).
 *   inputs, SoA [L][N]: anchor (index into the anchor table, i.e. _anchorIndexById[anchorId] of
 *     :226 -- which yields index 0 for an id it does not know; 0xFF or >= n_anchors = padding of
 *     a ragged log), seq (0..255), range_mm (gtec_msgs/Ranging.range), err (errorEstimation,
 *     NULL = none; only values > 0 overwrite within a sequence, :94,236), t (arrival time, s);
 *   outputs: ranges_out int32 SoA [max_epochs][n_anchors][N] (-1 = no ranging, the table's
 *     initial value :505), err_out f64 same shape or NULL, dt_out f64 SoA [max_epochs][N] = time
 *     between consecutive reports (first report: first_dt; epochs a log does not have: -1),
 *     n_epochs [N] or NULL = reports each log produced (may exceed max_epochs: truncated).
 * flags: 0 = as written, the 256-row table whose new row gets only slot 0 cleared (:251-255,
 * SURVEY App. B-12: slots written 256 sequence numbers earlier survive);
 * KFPOS_ASM_FIX_ROW_CLEAR = clear the whole row.  The outputs feed kfpos_batch_replay_epochs
 * (KFPOS_FMT_I32_MM).  With device pointers the call is asynchronous on `stream`; its table
 * scratch is per device and reused by the next call, so concurrent calls on one device must use
 * one stream.  Host pointers are staged and the stream is synchronised before returning.   */
#define KFPOS_ASM_FIX_ROW_CLEAR 1
int kfpos_assemble_epochs(int device, int64_t n_logs, int64_t n_msgs, int n_anchors, const uint8_t *anchor,
                          const uint8_t *seq, const int32_t *range_mm, const double *err, const double *t,
                          int64_t max_epochs, int flags, double first_dt, int32_t *ranges_out, double *err_out,
                          double *dt_out, int32_t *n_epochs, void *stream);

/* The assembler with the REPORT TIMES as well: t_out SoA [max_epochs][N] = the time at which each
 * report reaches newTOAMeasurement (the arrival time of the ranging that started the next sequence
 * number, or last ranging + 0.05 s when the timer sent it); -1 for epochs a log does not have.  NULL
 * = kfpos_assemble_epochs.                                                                       */
int kfpos_assemble_epochs_t(int device, int64_t n_logs, int64_t n_msgs, int n_anchors, const uint8_t *anchor,
                            const uint8_t *seq, const int32_t *range_mm, const double *err, const double *t,
                            int64_t max_epochs, int flags, double first_dt, int32_t *ranges_out, double *err_out,
                            double *dt_out, int32_t *n_epochs, double *t_out, void *stream);

/* ------------------------------------------------------------ stream merger
 * PosGenerator runs every callback of a tag on one thread (Posgenerator.cpp:92-140): ranging reports
 * (from the aggregation above) and PX4Flow / IMU / magnetometer / compass samples reach the filter in
 * ARRIVAL ORDER, and the filter takes the time since its previous callback as dt (0.1 s for the first
 * one, KF.cpp:232-243).  This call does that interleaving for N tags at once and lays the N sequences
 * onto ONE schedule of n_slots events for kfpos_batch_replay_events_ragged: slot s has kind
 * slot_kind[s] (KFPOS_EV_*, host array, any pattern -- e.g. the tags' nominal message pattern
 * repeated); a tag's next event takes the next slot of its kind; slots it passes over get dt = -1
 * ("this filter has no such event").  Equal time stamps: sensor samples in KFPOS_EV_* order, then
 * the ranging report.
 *   t_epoch SoA [n_epochs][N], ranges int32 SoA [n_epochs][n_anchors][N], err f64 same shape or NULL:
 *       outputs of kfpos_assemble_epochs_t;
 *   sensor streams q = 0..3 (PX4, IMU, MAG, COMPASS): n_samples[q], t_sensor[q] SoA [n_samples][N]
 *       arrival times (a negative or NaN value ends the tag's stream), payload[q] SoA
 *       [n_samples][rows][N] with the rows of kfpos_event (5 / 3 / 2 / 1); NULL / 0 = no such stream;
 *   imu_aux: the 9 aux doubles every IMU slot gets (covariances, common to the batch), or NULL;
 *   outputs: events_out HOST [n_slots] (kind, offset; dt unused); dt_out SoA [n_slots][N];
 *       ranges_out int32 SoA [n_anchors * #TOA slots][N] (-1 where no event); err_out same shape or
 *       NULL; sensors_out f64 SoA [sum of the sensor slots' rows][N]; n_dropped [N] or NULL = events of
 *       a tag that found no slot left (raise n_slots).
 * Host or device pointers for the tensors; the call synchronises `stream` before returning.       */
int kfpos_merge_streams(int device, int64_t n_logs, int n_anchors, int64_t n_epochs, const double *t_epoch,
                        const int32_t *ranges, const double *err, const int64_t n_samples[4],
                        const double *const t_sensor[4], const double *const payload[4], int n_slots,
                        const int32_t *slot_kind, double first_dt, const double *imu_aux,
                        kfpos_event *events_out, double *dt_out, int32_t *ranges_out, double *err_out,
                        double *sensors_out, int32_t *n_dropped, void *stream);

/* ------------------------------------------------------------- diagnostics
 * Work counters accumulated on the device since the last reset, as doubles:
 * [0] updates, [1] inner-ML Newton iterations, [2] IEKF cost evaluations,
 * [3] IEKF gain computations, [4] updates with status != OK, [5] anchors
 * ignored by leave-one-out, [6] T6 inner-ML solves that ended at the reference's
 * 10000-iteration cap (ML.cpp:165), [7] of those, the ones whose tail the exact cycle
 * detection skipped (both counted by the tuned T6 replay only).                  */
int kfpos_batch_get_counters(kfpos_batch *b, double out[8], int reset, void *stream);

/* Error statistics against a truth position SoA [3][N] (host or device):
 * out[0] = sum |p - truth|^2, out[1] = same over x,y only, out[2] = filters
 * counted (finite), out[3] = filters with status != OK.  Summation order: a fixed
 * 128-leaf tree per 128-filter chunk (one replay block), then a pairwise tree over
 * the chunk index -- it depends on the filter index only, not on launch geometry.
 *   truth == NULL : the ground truth registered with kfpos_batch_set_truth is used;
 *                   if a replay has run since, only the final tree is launched
 *                   (the chunk partials were left behind by the replay kernel).
 *   out == NULL   : enqueue only; the result stays on the device for
 *                   kfpos_stats_allreduce (no host synchronisation).              */
int kfpos_batch_error_stats(kfpos_batch *b, const double *truth, double out[4], void *stream);

/* Registers the ground truth (SoA [3][N]; a device pointer is borrowed, a host array
 * is copied) for the Monte Carlo statistics: from now on every replay launch ends with
 * the block-level reduction of |p - truth|^2 of its final state (SURVEY.md G5: the
 * reduction is fused into the last replay step).  NULL unregisters.                */
int kfpos_batch_set_truth(kfpos_batch *b, const double *truth, void *stream);

/* The one collective of a sharded run (SURVEY.md 8e; no reference equivalent -- the
 * reference runs one filter): reduces the error statistics of the batches of all ranks
 * of `comm` (an NCCL communicator with one rank per GPU; NULL = this batch alone).
 *   out[0..3] as kfpos_batch_error_stats, summed over all ranks;
 *   out[4] = RMSE = sqrt(out[0] / out[2]);  out[5] = RMSE over x,y.
 * One ncclAllGather of 4 doubles per rank, then the pairwise tree over the rank index on
 * every rank: with shards that are aligned powers of two (N_total / n_ranks filters, a
 * multiple of 128) the result is BIT-IDENTICAL to the single-GPU result.  truth as above
 * (NULL with nothing registered: reduces what the last kfpos_batch_error_stats left on
 * the device).  NCCL is bound with dlopen("libnccl.so.2") at the first call:
 * KFPOS_ERR_UNSUPPORTED when it cannot be found.  Synchronises `stream`.            */
struct ncclComm;
int kfpos_stats_allreduce(kfpos_batch *b, struct ncclComm *comm, const double *truth, double out[6], void *stream);

/* Time-resolved Monte Carlo statistics (no reference equivalent; SURVEY.md G5 extended to every epoch).
 * Registers a truth trajectory SoA [n_rows][3][N] (x, y, z per output row; K8: z = the tag height, as for
 * kfpos_batch_set_truth).  A device pointer is borrowed; a host array is copied.  NULL unregisters.
 * Registering, and every kfpos_batch_set_state, sets the row cursor to 0.  While a trajectory is
 * registered, every replay launch (replay_toa / step_toa, replay_epochs, replay_events, _ragged) leaves,
 * for each of its output rows (the rows of its `traj`: a T6 epoch, a K8 / T9 TOA event), the partial
 * sums of row `cursor + r`, and advances the cursor.  A launch that would pass n_rows fails with
 * KFPOS_ERR_INVALID and runs nothing.  ML batches: KFPOS_ERR_INVALID.  Device scratch: 48 B per 32
 * filters per row, allocated here (KFPOS_ERR_NOMEM when it cannot be).                                  */
int kfpos_batch_set_truth_traj(kfpos_batch *b, int64_t n_rows, const double *truth, void *stream);

/* out [n_rows][6] (host or device; n_rows must equal the registered count), per row:
 *   [0] sum |p - truth|^2   [1] same over x, y   [2] filters counted (finite error)
 *   [3] filters whose status word of THIS epoch is != 0
 *   [4] sum NEES = e^T S^-1 e over the position block S of the covariance after the epoch
 *       (T6 / T9: 3x3, K8: the x-y 2x2 block, e = the x-y error)   [5] filters in [4] (finite NEES, S positive
 *       definite by its LDL^T pivots)
 * A filter without an epoch in that row (per-filter dt < 0) adds nothing.  Rows the cursor has not
 * reached are zero.  Summation order: a fixed 32-leaf tree per 32-filter chunk, then a pairwise tree
 * over the chunk index.  It depends on the filter index only.  Device `out`: asynchronous on `stream`.
 * Nothing registered: KFPOS_ERR_NOT_READY.                                                             */
int kfpos_batch_epoch_stats(kfpos_batch *b, int64_t n_rows, double *out, void *stream);

/* The same summed over the ranks of `comm`: one ncclAllGather of n_rows * 6 doubles per rank, then the
 * pairwise rank tree on every rank.  With aligned power-of-two shards (a multiple of 32 filters) the
 * result is bit-identical to the single-GPU result.  NCCL is bound as for kfpos_stats_allreduce
 * (comm == NULL: this batch alone).                                                                    */
int kfpos_epoch_stats_allreduce(kfpos_batch *b, struct ncclComm *comm, int64_t n_rows, double *out, void *stream);

/* Per-epoch error histograms for Monte Carlo runs (no reference equivalent; the distributions behind the
 * means of kfpos_batch_epoch_stats: error percentiles such as CEP50 / CEP95 over time, and the fraction of
 * NEES values inside chi-square bounds).  Registers a histogram of one quantity per output row:
 *   KFPOS_HIST_ERR     |p - truth| in m           (the value behind epoch_stats column [0])
 *   KFPOS_HIST_ERR_XY  x-y error in m             (column [1])
 *   KFPOS_HIST_NEES    NEES, dimensionless        (column [4])
 * `edges` is a HOST array of 1..255 finite, strictly increasing values (m and >= 0 for the two error
 * quantities).  Bin k of a value v holds the values with exactly k edges <= v: bin 0 is below edges[0], bin
 * n_edges is at or above the last edge.  The error quantities are binned as e^2 against the squared edges
 * (each squared once here, an IEEE multiply), so a host reproduces every bin exactly from the trajectory,
 * e.g. numpy.searchsorted(edges * edges, e2, side="right").  A filter counts where it counts in epoch_stats
 * ([2] for the errors, [5] for NEES), so each row's total equals that column.  n_edges == 0 or edges == NULL
 * unregisters.  The histogram is a batch attribute: it stays registered across kfpos_batch_set_truth_traj,
 * and it is filled only while a truth trajectory is registered.  Storage [rows][n_edges + 1] uint64 on the
 * device is (re)allocated and zeroed by whichever of the two registrations comes last, and by every later
 * truth registration.  Each replay launch overwrites the rows it fills (a re-run after set_state replaces
 * them).  KFPOS_ERR_INVALID: ML batch, bad quantity, bad edge table.  KFPOS_ERR_NOMEM: no storage.       */
#define KFPOS_HIST_ERR 0    /* |p - truth|   (the value of epoch_stats column [0]) */
#define KFPOS_HIST_ERR_XY 1 /* x-y error     (column [1])                          */
#define KFPOS_HIST_NEES 2   /* NEES          (column [4])                          */
int kfpos_batch_set_error_hist(kfpos_batch *b, int quantity, int n_edges, const double *edges);

/* counts [n_rows][n_edges + 1] uint64 (host or device; n_rows must equal the registered truth rows), the
 * number of filters per bin at each output row.  Rows the cursor has not reached are zero.  Device `counts`:
 * asynchronous on `stream`.  KFPOS_ERR_NOT_READY: no histogram or no truth trajectory registered.          */
int kfpos_batch_error_hist(kfpos_batch *b, int64_t n_rows, uint64_t *counts, void *stream);

/* The same summed over the ranks of `comm`: one ncclAllGather of n_rows * (n_edges + 1) uint64 per rank,
 * then an integer sum over the ranks.  Counts are integers, so the result is EXACTLY the single-GPU result
 * for any shard sizes.  NCCL is bound as for kfpos_stats_allreduce (comm == NULL: this batch alone).      */
int kfpos_error_hist_allreduce(kfpos_batch *b, struct ncclComm *comm, int64_t n_rows, uint64_t *counts,
                               void *stream);

/* Roofline denominator for this FP64 CUDA-core path (no reference equivalent):
 * times a DFMA-only kernel on `device` and returns the sustained FLOP/s.        */
int kfpos_measure_fp64_peak(int device, double *flops_per_s);

/* Monte Carlo inputs for K8 batches, generated on the device (no reference equivalent; BASELINE
 * configs 3 and 5 run millions of filters for 1000 steps: their sensor streams do not fit in memory
 * and are synthesised chunk by chunk into the tensors kfpos_batch_replay_events streams).  Each
 * value is a pure function of (seed, first_filter + f, event global_index, sample) through the
 * counter-based Philox4x32-10 generator: independent of sharding and chunking.  Truth: planar
 * Lissajous x = 5 + 3 sin(0.20 t + a), y = 5 + 3 sin(0.31 t + b), heading th0 + 0.05 t with a, b, th0
 * per filter.  Payload rows written at `offset` (rows of N values): KFPOS_EV_TOA n_anchors int32 mm
 * ranges (noise sigma_r m) into `ranges`; KFPOS_EV_IMU gyro z, body accel x, y (variances 0.089,
 * 0.003); KFPOS_EV_PX4 the five PX4Flow fields (33.333 ms, height 5 m, quality 200);
 * KFPOS_EV_COMPASS heading + N(0, 0.01^2) -- the payload layouts of kfpos_batch_replay_events.
 * events: HOST array; x0 (SoA [8][N], state at t = 0) and truth_end (SoA [3][N], position at
 * t_end) optional.  Asynchronous on `stream` when every output is a device pointer (so that the next
 * chunk can be generated on one stream while the current one is replayed on another), else it
 * synchronises `stream` before returning.                                    */
typedef struct kfpos_synth_event {
    int32_t kind;         /* kfpos_event_kind                                   */
    int32_t global_index; /* index of the event in the whole run (RNG counter)  */
    double t;             /* time of the event, s                               */
    int64_t offset;       /* first output row                                   */
} kfpos_synth_event;
int kfpos_synth_k8(int device, int64_t n_filters, int64_t first_filter, uint64_t seed, int n_anchors,
                   const double *anchors_xyz, double tag_z, double sigma_r, int n_events,
                   const kfpos_synth_event *events, double t_end, int64_t range_rows, int64_t sensor_rows,
                   int32_t *ranges, double *sensors, double *x0, double *truth_end, void *stream);

/* Truth of the kfpos_synth_k8 AND kfpos_synth_toa_ranges workloads at host times t[0..n_times): SoA
 * [n_times][3][N] = (x, y, tag_z).  Both generators draw the same per-filter Philox constants and use the
 * same kinematics, so that a chunked run can register the truth of each chunk's TOA events / epochs.
 * Asynchronous on `stream` when `t` and `truth` are device pointers, else it synchronises `stream`
 * before returning.                                                                                  */
int kfpos_synth_k8_truth(int device, int64_t n_filters, int64_t first_filter, uint64_t seed, int n_times,
                         const double *t, double tag_z, double *truth, void *stream);

/* Monte Carlo ranging epochs, generated on the device (no reference equivalent): the [T][M][N] millimetre
 * range log every ranging consumer takes (kfpos_batch_replay_toa, the K8 / T9 ranging replays,
 * kfpos_batch_ml_solve), with optional missing rangings and NLOS biases.  For filter gf = first_filter + f,
 * epoch g = first_epoch + k at time t[k] and anchor a (Philox4x32-10 counter (gf lo, gf hi, event, sample),
 * key (seed lo, seed hi), as kfpos_synth_k8):
 *   truth     (x, y, z) = the Lissajous of kfpos_synth_k8 (kfpos_synth_k8_truth gives it), z = tag_z;
 *   distance  d_a = |(x, y, z) - anchor_a|;
 *   noise     n_a = Box-Muller normal number a & 1 of the counter (gf, g, a >> 1);
 *   impaired  only when p_missing > 0 or p_nlos > 0: (u, v) = two uniforms of the counter
 *             (gf, g, 0x80000000 | a); missing when u < p_missing; NLOS bias b = -nlos_mean log(v / p_nlos)
 *             when v < p_nlos (an exponential of mean nlos_mean), else 0;
 *   output    mm = floor((d_a + sigma_r n_a + b) * 1000); 0 ("no ranging") when missing or mm <= 0;
 *             KFPOS_FMT_U16_MM clamps to 65535.
 * Each value is a pure function of (seed, gf, g, a): a run gives the same numbers however it is sharded
 * (first_filter) or cut into chunks (first_epoch).  Epoch index 0xFFFFFFFF is reserved for the per-filter
 * constants: first_epoch + n_epochs must not exceed it.                                                 */
typedef struct kfpos_synth_toa {
    uint64_t seed;
    int64_t first_filter;  /* global index of output filter 0 (sharding)                 */
    int64_t first_epoch;   /* global index of epoch 0 of this call (chunking)            */
    double tag_z;          /* m                                                          */
    double sigma_r;        /* ranging noise sd, m (>= 0)                                 */
    double p_missing;      /* probability that a ranging is absent, [0, 1]               */
    double p_nlos;         /* probability of a positive NLOS bias, [0, 1]                */
    double nlos_mean;      /* mean of the exponential bias, m (> 0 when p_nlos > 0)      */
} kfpos_synth_toa;

/* t: HOST array [n_epochs] of epoch times, s.  ranges: SoA [n_epochs][n_anchors][N] in fmt
 * (KFPOS_FMT_I32_MM or KFPOS_FMT_U16_MM).  A device `ranges` makes the call asynchronous on `stream`; a
 * host one is staged and `stream` is synchronised before returning.  KFPOS_ERR_INVALID: a bad count,
 * n_anchors outside [1, KFPOS_MAX_ANCHORS], a probability outside [0, 1], sigma_r < 0, nlos_mean <= 0 with
 * p_nlos > 0, first_filter < 0, an epoch range that reaches the reserved index, another fmt.
 * KFPOS_ERR_CUDA without a device (there is no CPU path).                                              */
int kfpos_synth_toa_ranges(int device, int64_t n_filters, int n_anchors, const double *anchors_xyz,
                           int n_epochs, const double *t, const kfpos_synth_toa *gen, int fmt,
                           void *ranges, void *stream);

/* The same log with its NLOS ground truth: nlos SoA [n_epochs][N] uint32 (host or device), bit a set when ranging
 * a drew a bias (v < p_nlos above) AND is present in the log (value > 0 after the missing test and the floor).
 * All zero without impairments.  `ranges` is byte for byte what kfpos_synth_toa_ranges writes for the same
 * arguments.  Arguments, errors and the sync rule are those of kfpos_synth_toa_ranges (the call is asynchronous
 * when `ranges` and `nlos` are both device pointers); a NULL nlos is KFPOS_ERR_INVALID.                     */
int kfpos_synth_toa_ranges_nlos(int device, int64_t n_filters, int n_anchors, const double *anchors_xyz,
                                int n_epochs, const double *t, const kfpos_synth_toa *gen, int fmt,
                                void *ranges, uint32_t *nlos, void *stream);

/* Obstacle-based NLOS (DESIGN §4.5f): the log of kfpos_synth_toa_ranges in a room with axis-aligned boxes that
 * bias or remove the rangings whose direct path crosses them.  For the ranging of filter gf, epoch g and anchor
 * a, with truth T = (x, y, tag_z), anchor A and Dv = A - T, the segment T + s Dv, s in [0, 1], meets box o when
 * the slab test gives enter < exit: enter = 0, exit = 1, and per axis i with Dv_i != 0 (inv_i = 1 / Dv_i)
 *   s1 = (lo_i - T_i) inv_i, s2 = (hi_i - T_i) inv_i, enter = max(enter, min(s1, s2)), exit = min(exit, max(s1, s2));
 * an axis with Dv_i == 0 lets the box block only when lo_i < T_i < hi_i.  Boxes are open: a segment that only
 * touches a face is not blocked.  Every step is one IEEE operation, so a host reproduces the decision exactly
 * from the truth of kfpos_synth_k8_truth.  L_o = (exit - enter) d_a is the length of the path inside box o.
 * When at least one box blocks the ranging, after the noise and the i.i.d. bias of kfpos_synth_toa_ranges:
 *   r += sum_o excess_per_m_o L_o over the blocking boxes, in box order;
 *   (u, v) = two uniforms of the counter (gf, g, 0x40000000 | a);
 *   the ranging is absent when u < 1 - prod_o (1 - p_loss_o) (blocking boxes, in box order);
 *   r += -S log(v) when S = sum_o spread_o > 0 (an exponential of mean S).
 * Then mm = floor(r * 1000) as before; the ranging is absent when missing, lost or mm <= 0.  nlos (or NULL):
 * bit a set when ranging a drew an i.i.d. bias OR was blocked, and is present -- a blocked ranging with no
 * bias is NLOS too, its direct path is obstructed.  n_obstacles == 0, or boxes that block nothing, give the
 * log and mask of kfpos_synth_toa_ranges / _nlos byte for byte.  obstacles: HOST array, copied before the call
 * returns.  Errors and the sync rule are kfpos_synth_toa_ranges's; KFPOS_ERR_INVALID also for n_obstacles
 * outside [0, KFPOS_MAX_OBSTACLES], NULL obstacles with n_obstacles > 0, a non-finite corner, !(lo < hi) on an
 * axis, excess_per_m or spread negative or not finite, p_loss outside [0, 1].                                 */
typedef struct kfpos_obstacle {
    double lo[3], hi[3];  /* box corners, m; lo < hi on every axis                                     */
    double excess_per_m;  /* range excess per metre of direct path inside the box, >= 0 (a dielectric
                             slab of permittivity eps_r delays by (sqrt(eps_r) - 1) per metre)          */
    double spread;        /* mean of an exponential bias added when the box blocks the ranging, m, >= 0 */
    double p_loss;        /* probability that a ranging this box blocks is absent, [0, 1]               */
} kfpos_obstacle;
#define KFPOS_MAX_OBSTACLES 32
int kfpos_synth_toa_ranges_geo(int device, int64_t n_filters, int n_anchors, const double *anchors_xyz,
                               int n_epochs, const double *t, const kfpos_synth_toa *gen,
                               int n_obstacles, const kfpos_obstacle *obstacles, int fmt,
                               void *ranges, uint32_t *nlos, void *stream);

/* Ranging epochs along a caller's trajectory (DESIGN §4.5g): kfpos_synth_toa_ranges_geo with the truth of epoch
 * g = first_epoch + k read from row k of `truth`, SoA [n_epochs][3][N] (x, y, z per epoch; the layout of
 * kfpos_batch_set_truth_traj and kfpos_batch_crlb), HOST or device, in place of the Lissajous; gen->tag_z is
 * ignored (z comes from the array, the slab test uses it too).  Everything else is kfpos_synth_toa_ranges_geo's:
 * the Philox counters, noise, i.i.d. impairments, boxes, mask, formats and clamp -- so the truth of
 * kfpos_synth_k8_truth at the same times gives the same bytes as kfpos_synth_toa_ranges / _nlos / _geo.  A NaN
 * truth value gives absent rangings (0: mm > 0 fails); an infinite one gives the format's largest value (the
 * clamp).  obstacles may be NULL with n_obstacles == 0,
 * nlos may be NULL.  A host truth, ranges or nlos is staged and `stream` synchronised before returning; with device
 * pointers only the call is asynchronous on `stream`.  Errors are kfpos_synth_toa_ranges_geo's; a NULL truth with
 * n_epochs > 0 is KFPOS_ERR_INVALID.                                                                            */
int kfpos_synth_toa_ranges_truth(int device, int64_t n_filters, int n_anchors, const double *anchors_xyz,
                                 int n_epochs, const double *truth, const kfpos_synth_toa *gen,
                                 int n_obstacles, const kfpos_obstacle *obstacles, int fmt,
                                 void *ranges, uint32_t *nlos, void *stream);

/* A random walk of the tag inside a caller's box (DESIGN §4.5g), the truth kfpos_synth_toa_ranges_truth takes:
 * discrete white-noise acceleration, the F and Q of the T6 prediction, per axis i, kept inside [lo_i, hi_i].
 * For filter gf = first_filter + f (Philox4x32-10 counter (gf lo, gf hi, event, sample), key (seed lo, seed hi)):
 *   initial   (init 1) velocity 0; position lo_i + (hi_i - lo_i) u_i with (u_x, u_y) the uniforms of counter
 *             (gf, 0xFFFFFFFF, 2) and u_z the first of (gf, 0xFFFFFFFF, 3); an axis with accel_sd_i == 0 starts at
 *             (lo_i + hi_i) / 2 and stays there (a fixed tag height);
 *   epoch g   (n_x, n_y) = the Box-Muller pair of counter (gf, g, 0x20000000); n_z the first normal of
 *             (gf, g, 0x20000001), drawn only when accel_sd_z > 0 (else a_z = 0); per axis, with dt = period and
 *             h = dt dt / 2:  a = accel_sd_i n_i,  p' = (p + v dt) + a h,  v' = v + a dt;
 *             if p' > hi: p' = (hi + hi) - p', v' = -v'; else if p' < lo: p' = (lo + lo) - p', v' = -v';
 *             then p' = min(max(p', lo), hi), v' = min(max(v', -v_max), v_max).
 * Every step is one IEEE operation (no contraction), so a host reproduces a trajectory from its normals, and
 * each value is a pure function of (seed, gf, g) and the initial state: a run gives the same trajectory however
 * it is sharded (first_filter) or cut into chunks (first_epoch, with `state` carried).  The walk's samples
 * (0x20000000, 0x20000001) are not among the ranging generator's (0..15, 0x80000000 | a, 0x40000000 | a), so
 * the walk and the rangings may share one seed without sharing a draw.
 * state: SoA [6][N] x, y, z, vx, vy, vz (the T6 state layout): the state at first_epoch on entry (read with
 * init 0), the state after the last epoch on return.  truth: SoA [n_epochs][3][N], row k the position at time
 * (first_epoch + k + 1) period (x0 is the state at t = 0).  init 1 with n_epochs == 0 writes the initial state
 * and returns.  Host or device arrays; a host one is staged and `stream` synchronised before returning, with
 * device pointers only the call is asynchronous on `stream`.  KFPOS_ERR_INVALID: a bad count, first_filter or
 * first_epoch < 0, an epoch range that reaches the reserved index, period <= 0 or not finite, accel_sd negative
 * or not finite, v_max <= 0 or NaN, a non-finite corner or !(lo < hi) on an axis, init not 0 or 1, a NULL state,
 * a NULL truth with n_epochs > 0.  KFPOS_ERR_CUDA without a device (there is no CPU path).                       */
struct kfpos_synth_walk { /* a struct tag only, beside the function of the same name (as struct stat / stat()) */
    uint64_t seed;
    int64_t first_filter;  /* global index of output filter 0 (sharding)                 */
    int64_t first_epoch;   /* global index of epoch 0 of this call (chunking)            */
    double period;         /* s, > 0                                                     */
    double accel_sd[3];    /* m/s^2 per axis, >= 0, finite                               */
    double v_max[3];       /* m/s per axis, > 0 (INFINITY: no cap)                       */
    double lo[3], hi[3];   /* region, m, finite, lo < hi                                 */
    int32_t init;          /* 1: draw the initial state; 0: continue from `state`        */
    int32_t reserved;
};
int kfpos_synth_walk(int device, int64_t n_filters, int n_epochs, const struct kfpos_synth_walk *walk,
                     double *state, double *truth, void *stream);

/* NLOS detection scores of a ranging selection (no reference equivalent; DESIGN §4.5d): how the selection of
 * rows [0, n_rows) of a log this batch has just replayed (T6, kfpos_batch_replay_toa) or solved (ML,
 * kfpos_batch_ml_solve) compares with the NLOS truth.  ranges: the log, SoA [n_rows][n_anchors][N] in any fmt; a
 * ranging is present when its value is > 0 (mm > 0, metres > 0; NaN is not), the replay's rule.  nlos: SoA
 * [n_rows][N] uint32 masks (kfpos_synth_toa_ranges_nlos), or NULL: no ranging is NLOS (drop rates of real logs).
 * `sel` is read as the batch's configuration wrote it:
 *   T6, variant 1 or 2:         sel [n_rows][N] = the bit mask of the slots used, read as uint32 (with 32 anchors a
 *                               full mask is -1);
 *   T6, ignore_worst_anchor:    sel [n_rows][N] = the slot left out, or -1 for none;
 *   T6 otherwise:               nothing is dropped; sel is not read and may be NULL;
 *   ML, variant 1 or 2:         n_rows == 1 and sel = the [2][N] output of kfpos_batch_ml_solve; row 0, the mask of
 *                               the final solve, is read.  Epochs with too few rangings (KFPOS_ST_ML_FEW) hold the
 *                               present set there, so they drop nothing.  So do epochs whose all-ranging solve
 *                               failed (KFPOS_ST_SINGULAR), and variant-2 epochs in which a subset solve failed
 *                               (the reference selects nothing then).  A variant-1 epoch whose re-solve after the
 *                               drop failed keeps the reduced set: its drop counts;
 *   ML, variant 0:              nothing is dropped; sel is not read (n_rows == 1 still).
 * used = that set, dropped = present & ~used.  counts [n_rows][KFPOS_SCORE_COLS] uint64 (host or device),
 * overwritten, per row summed over the filters:
 *   [0] rangings present          [1] rangings dropped
 *   [2] NLOS rangings (present, mask bit set)                  [3] NLOS rangings dropped
 *   [4] filters with at least one NLOS ranging                 [5] of [4], filters whose used set has no NLOS ranging
 *   [6] filters that dropped at least one ranging              [7] of [6], filters without any NLOS ranging
 * Detection rate [3]/[2], false-drop rate ([1]-[3])/([0]-[2]), clean-filter rate [5]/[4], filter false-alarm rate
 * [7]/(N-[4]).  Counts are integers: a sharded run sums them exactly with any integer all-reduce.
 * KFPOS_ERR_UNSUPPORTED: K8 and T9 batches.  KFPOS_ERR_INVALID: n_rows <= 0, a bad fmt, NULL ranges or counts, a
 * NULL sel where it is read, n_rows != 1 for ML.  KFPOS_ERR_NOT_READY: no anchors.                           */
#define KFPOS_SCORE_COLS 8
int kfpos_batch_score_selection(kfpos_batch *b, int n_rows, const void *ranges, int fmt, const int32_t *sel,
                                const uint32_t *nlos, uint64_t *counts, void *stream);

/* Cramer-Rao lower bound of the position per epoch (no reference equivalent; DESIGN §4.5e): the position-error
 * floor of the rangings of rows [0, n_rows) of a log, for the set `set` of each filter:
 *   KFPOS_CRLB_PRESENT: the rangings present in the log (value > 0, NaN is not: the scorer's rule);
 *   KFPOS_CRLB_LOS:     present and not set in the `nlos` mask -- the set a perfect NLOS detector keeps;
 *   KFPOS_CRLB_USED:    present and kept by the batch's selection, `sel` read exactly as
 *                       kfpos_batch_score_selection reads it (nothing dropped: plain T6, ML variant 0).
 * With the true position p (truth, SoA [n_rows][3][N]; ML: [3][N]) and the batch's anchors b_a, the Fisher
 * information of the epoch is J = sum_{a in S} g_a g_a^T / v_a, g_a = (p - b_a) / |p - b_a|.  D = 3 for T6, T9
 * and 3-D ML batches; D = 2 for K8 and ML batches with use2d, whose height is known: g_a is then the x-y part of
 * the same 3-D unit vector.  v_a = var[r][a][f] (SoA [n_rows][n_anchors][N], or NULL: var_scalar) is the TRUE
 * variance of the ranging noise, not the filters' errorEstimation.  A filter's terms are
 *   [0] tr J^-1   [1] (J^-1)_xx + (J^-1)_yy   [2] 1   [3] 0
 * or 0, 0, 0, 1 when it has no bound: |S| < D, a non-finite truth, a v_a (a in S) that is not finite and > 0, a
 * non-positive or non-finite pivot of the LDL^T of J, or a non-finite trace.  out [n_rows][KFPOS_CRLB_COLS]
 * doubles (host or device), overwritten: per row the terms summed over the filters in a fixed order -- each 32
 * filters by the 32-leaf tree of kfpos_batch_epoch_stats, then pairwise over the 32-filter groups -- which
 * depends on the filter index only: chunks of rows change nothing, and the rows of aligned power-of-two shards
 * (multiples of 32 filters) added pairwise in rank order equal the whole batch's bit for bit.  sqrt([0] / [2])
 * is the RMS floor of the epoch.  Reads nothing and changes nothing of the batch's state.  Scratch: 32 B per 32
 * filters per row, at most 256 MB, kept by the batch.
 * KFPOS_ERR_INVALID: a bad set, n_rows <= 0, a bad fmt, NULL truth, ranges or out, var NULL with var_scalar not
 * finite and > 0, KFPOS_CRLB_LOS with a NULL nlos, KFPOS_CRLB_USED with a NULL sel where it is read, n_rows != 1
 * for ML.  KFPOS_ERR_UNSUPPORTED: KFPOS_CRLB_USED on K8 and T9 batches (they keep no selection).
 * KFPOS_ERR_NOT_READY: no anchors.                                                                              */
#define KFPOS_CRLB_PRESENT 0
#define KFPOS_CRLB_LOS 1
#define KFPOS_CRLB_USED 2
#define KFPOS_CRLB_COLS 4
int kfpos_batch_crlb(kfpos_batch *b, int set, int n_rows, const double *truth, const void *ranges, int fmt,
                     double var_scalar, const double *var, const int32_t *sel, const uint32_t *nlos, double *out,
                     void *stream);

/* Accuracy self-test of the kernels' elementary functions (no reference equivalent): evaluates the
 * MUFU-seeded reciprocal and reciprocal square root and the reduced-range sincos on x[0..n) so that
 * a test can compare them with IEEE division / sqrt / libm.  Outputs may be NULL.               */
int kfpos_selftest_math(int device, int64_t n, const double *x, double *rcp, double *rsqrt, double *sn,
                        double *cs);

/* Self-test of the exact-order solver's branch-free IEEE division and square root (kfpos_exact.cu: the
 * compiler's own fast-path sequences with the operand-range test accumulated into a flag): a[i] / b[i] and
 * sqrt(a[i]) through them (plain operator when the flag says so) next to the plain operators, so that a test
 * can compare the two BIT FOR BIT; flags bit 0 / 1 = the fast path was taken.  Outputs may be NULL.        */
int kfpos_selftest_ieee(int device, int64_t n, const double *a, const double *b, double *div_fast,
                        double *div_ieee, double *sqrt_fast, double *sqrt_ieee, int32_t *flags);

#ifdef __cplusplus
}
#endif
#endif /* KFPOS_B200_H */
