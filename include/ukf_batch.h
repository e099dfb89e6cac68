/*
 * ukf_batch.h -- C ABI of the B200-native batched unscented Kalman filter engine.
 *
 * Drop-in boundary for the predict/update hot path of rock-slam/slam-pose_estimation.
 * One handle owns B independent filters of one kind (PoseUKF or OrientationUKF), on ONE
 * CUDA device (ukfb_create) or split by filter index over several devices of one box
 * (ukfb_create_sharded); filter b of the batch behaves exactly like one instance of the
 * reference class.  Every entry point below names the reference interface it
 * replaces (file:line relative to the reference tree).  The reference is a C++
 * class API with no FFI of its own; the headers under include/pose_estimation_b200/ re-create
 * those classes (same names, arguments and exceptions) on top of this ABI, and
 * INTEGRATION.md shows the binding a maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; all arrays are caller-owned, dense, row-major,
 *     IEEE double unless stated; nothing is retained after a call returns.
 *   - functions without a suffix take HOST pointers and copy inside the call;
 *     the `_dev` variants take DEVICE pointers (same layout) and only enqueue work
 *     on the handle's stream.
 *   - mu layout (quaternion stored x,y,z,w as Eigen does):
 *       POSE        13: p[0:3] q[3:7] v[7:10] w[10:13]   (PoseWithVelocity.hpp:18-23)
 *       ORIENTATION 14: q[0:4] v[4:7] bg[7:10] ba[10:13] g[13]  (OrientationState.hpp:20-26)
 *     covariance: n x n with n = 12 / 13, tangent order as in ukfb_constants.h.
 *     The engine stores the lower triangle (the covariance is symmetric up to
 *     rounding in the reference; Cholesky 'L' reads only that triangle anyway).
 *   - return value: 0 = ok, < 0 = UKFB_ERR_*; ukfb_last_error() gives text.
 *   - the reference throws std::runtime_error for a negative / too large time
 *     delta (UnscentedKalmanFilter.hpp:110-122) and for a non-finite measurement
 *     (:142-147).  A batch cannot throw per filter: the operation is skipped for
 *     that filter exactly as the throw would have skipped it, and a sticky
 *     per-filter status bit UKFB_STATUS_* is set.  The C++ shim re-throws.
 *   - a handle is single-caller (the reference is not thread-safe either,
 *     UnscentedKalmanFilter.hpp:16); different handles are independent and may be
 *     driven from different host threads (a sharded handle does exactly that inside).
 *   - there is no CPU fallback: every entry point fails with UKFB_ERR_CUDA when no
 *     sm_100-class device is usable.
 */
#ifndef UKF_BATCH_H
#define UKF_BATCH_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ukfb_handle ukfb_handle;

/* filter kinds */
#define UKFB_POSE 0        /* pose_estimation::PoseUKF         (PoseUKF.hpp:17-93)        */
#define UKFB_ORIENTATION 1 /* pose_estimation::OrientationUKF  (OrientationUKF.hpp:20-59) */

/* measurement kinds: one per integrateMeasurement overload that calls ukf->update */
#define UKFB_MEAS_NONE (-1)
#define UKFB_MEAS_POSE_POSITION 0         /* PositionMeasurement        m=3  PoseUKF.cpp:112-117 */
#define UKFB_MEAS_POSE_XY 1               /* XYMeasurement              m=2  PoseUKF.cpp:119-124 */
#define UKFB_MEAS_POSE_Z 2                /* ZMeasurement               m=1  PoseUKF.cpp:126-131 */
#define UKFB_MEAS_POSE_ORIENTATION 3      /* OrientationMeasurement     SO3  PoseUKF.cpp:133-138 */
#define UKFB_MEAS_POSE_VELOCITY 4         /* VelocityMeasurement        m=3  PoseUKF.cpp:140-145 */
#define UKFB_MEAS_POSE_XY_VELOCITY 5      /* XYVelocityMeasurement      m=2  PoseUKF.cpp:147-152 */
#define UKFB_MEAS_POSE_Z_VELOCITY 6       /* ZVelocityMeasurement       m=1  PoseUKF.cpp:154-159 */
#define UKFB_MEAS_POSE_XVEL_YAWVEL 7      /* XVelYawVelMeasurement      m=2  PoseUKF.cpp:161-166 */
#define UKFB_MEAS_POSE_ANGULAR_VELOCITY 8 /* AngularVelocityMeasurement m=3  PoseUKF.cpp:168-173 */
#define UKFB_MEAS_ORI_VELOCITY 9          /* OrientationUKF::VelocityMeasurement m=3  OrientationUKF.cpp:65-72 */
#define UKFB_MEAS_KIND_COUNT 10

/* event kinds of an event stream (ukfb_run_events): every measurement kind above, plus the integrateMeasurement
 * overloads that only store their sample for the next predict, plus "no sample in this slot" */
#define UKFB_EVENT_IDLE (-2)
#define UKFB_EVENT_POSE_ACCELERATION 10 /* PoseUKF::integrateMeasurement(AccelerationMeasurement)   PoseUKF.cpp:175-178 */
#define UKFB_EVENT_ORI_ROTATION_RATE 11 /* OrientationUKF::integrateMeasurement(RotationRate)       OrientationUKF.cpp:53-57 */
#define UKFB_EVENT_ORI_ACCELERATION 12  /* OrientationUKF::integrateMeasurement(Acceleration)       OrientationUKF.cpp:59-63 */
#define UKFB_EVENT_KIND_COUNT 13

/* sticky per-filter status bits */
#define UKFB_STATUS_NEG_DT 1u            /* "Delta time is negative!"                          :110-113 */
#define UKFB_STATUS_DT_TOO_LARGE 2u      /* "Delta time is greater then the allowed maximum!"  :119-122 */
#define UKFB_STATUS_NONFINITE_MEAS 4u    /* "Measurement or covariance contains non-finite values!" :142-147 */
#define UKFB_STATUS_NOT_SPD 8u           /* ukfom: Cholesky of sigma failed (MTK asserts)               */
#define UKFB_STATUS_MEAN_NO_CONVERGE 16u /* ukfom: sigma_points_mean hit max_it (MTK asserts)           */
#define UKFB_STATUS_MEAS_REJECTED 64u     /* not an error: a measurement failed the Mahalanobis gate and was not integrated */
#define UKFB_STATUS_BAD_EVENT 32u        /* an event stream held a kind this filter class has no overload for (ignored) */

/* error codes */
#define UKFB_OK 0
#define UKFB_ERR_INVALID (-1)         /* bad argument / wrong filter kind for this call */
#define UKFB_ERR_NOT_INITIALIZED (-2) /* getCurrentState() == false, UnscentedKalmanFilter.hpp:51-60 */
#define UKFB_ERR_CUDA (-3)            /* CUDA runtime error or no usable device */
#define UKFB_ERR_NOMEM (-4)

/* Text of the last error on the calling thread. */
const char* ukfb_last_error(void);

/* ---- lifecycle ---------------------------------------------------------- */

/* Constructors PoseUKF::PoseUKF (PoseUKF.cpp:99-110) / OrientationUKF::OrientationUKF
 * (OrientationUKF.cpp:41-51) minus their initializeFilter call (see ukfb_initialize):
 * base defaults Q = 0, t_last = 0, min_dt = 1e-9, max_dt = DBL_MAX
 * (UnscentedKalmanFilter.hpp:27-33); POSE: default diagonal Q and acceleration = NaN;
 * ORIENTATION: tau = +inf, latitude = 0 until ukfb_set_orientation_params. */
int ukfb_create(int filter_kind, int64_t batch, int device, ukfb_handle** out);
int ukfb_destroy(ukfb_handle* h);

/* The same B filters split by filter index over n_devices CUDA devices of one box.  Reference objects share nothing
 * (each owns its mu, sigma, Q and timestamp: UnscentedKalmanFilter.hpp:150-154), so shard i holds the contiguous
 * index range [first_i, first_i + count_i) with counts batch / n (+1 for the first batch % n shards), on devices[i],
 * with its own CUDA streams and its own host worker thread; there is no inter-device traffic.
 * EVERY host-pointer entry point of this header (blocking and _async) accepts the handle: the call fans out, each worker
 * serves its range of the caller's arrays, and the call returns when all shards have (ukfb_get_state[_async] therefore
 * lands all shards in the caller's single host buffer: the final gather).  Scalars and broadcast arguments
 * (per_filter = 0) go to every shard.  Results per filter are bit-for-bit those of a one-device handle.
 * `_dev` entry points take pointers of ONE device: on a sharded handle they return UKFB_ERR_INVALID; use them on the
 * per-device handles ukfb_shard() hands out.  devices = NULL: devices 0 .. n_devices - 1.  A device may appear twice. */
int ukfb_create_sharded(int filter_kind, int64_t batch, const int* devices, int n_devices, ukfb_handle** out);
/* number of shards (1 for a ukfb_create handle) */
int ukfb_shard_count(const ukfb_handle* h);
/* shard i of a sharded handle: its one-device handle (owned by the parent: do not destroy), first filter and count.
 * On a one-device handle, i = 0 returns the handle itself. */
int ukfb_shard(ukfb_handle* h, int i, ukfb_handle** shard, int64_t* first, int64_t* count);

/* Page-locked host memory visible to every device (cudaHostAllocPortable), for callers without the CUDA headers: the
 * _async entry points only overlap copies with kernels when their host arrays are pinned. */
int ukfb_host_alloc(void** ptr, uint64_t bytes);
int ukfb_host_free(void* ptr);

int64_t ukfb_batch(const ukfb_handle* h);
int ukfb_dof(const ukfb_handle* h);     /* getStateSize(), UnscentedKalmanFilter.hpp:127 */
int ukfb_mu_size(const ukfb_handle* h); /* 13 / 14 */
int ukfb_device(const ukfb_handle* h);

/* initializeFilter(initial_state, state_cov) for every filter
 * (UnscentedKalmanFilter.hpp:40-44): state replaced, t_last reset to 0.
 * mu: B x MU, sigma: B x n x n.  The first call on an ORIENTATION handle also does
 * what the constructor does after it: rotation_rate = 0, acceleration = (0,0,g0)
 * (OrientationUKF.cpp:49-50). */
int ukfb_initialize(ukfb_handle* h, const double* mu, const double* sigma);
/* isInitialized(), :128 */
int ukfb_is_initialized(const ukfb_handle* h);

/* getCurrentState(state, cov) / getCurrentState(state) (:51-75).  sigma may be NULL.
 * Returns UKFB_ERR_NOT_INITIALIZED where the reference returns false. */
int ukfb_get_state(ukfb_handle* h, double* mu, double* sigma);
int ukfb_get_state_dev(ukfb_handle* h, double* d_mu, double* d_sigma);

/* A contiguous range [mu_first, mu_first + mu_count) of the state vector only, out: B x mu_count.  What a consumer of
 * toRigidBodyState's pose needs (BodyStateMeasurement.hpp:30-31: position and orientation = entries 0..6 of a POSE
 * state) is 56 of the 104 bytes per filter of the full mean; on a link-bound host that is the difference. */
int ukfb_get_mu_range(ukfb_handle* h, int mu_first, int mu_count, double* out);
int ukfb_get_mu_range_dev(ukfb_handle* h, int mu_first, int mu_count, double* d_out);
int ukfb_get_mu_range_async(ukfb_handle* h, int mu_first, int mu_count, double* out); /* rules of ukfb_get_state_async */

/* BodyStateMeasurement (pose_with_velocity/BodyStateMeasurement.hpp:12-41), the format the reference's callers
 * exchange PoseUKF states in, for every filter of a POSE handle.  One base::samples::RigidBodyState is passed as
 * UKFB_RBS_DOUBLES doubles:
 *     position[3] orientation[4: x,y,z,w] velocity[3] angular_velocity[3]
 *     cov_position[9] cov_orientation[9] cov_velocity[9] cov_angular_velocity[9]        (3 x 3 blocks)
 * ukfb_initialize_from_body_states = fromRigidBodyState (:14-26) + initializeFilter: the four vectors are taken as
 * they are (the velocity is NOT rotated into the body frame, as in the reference), the covariance is the four
 * blocks on the diagonal and zero elsewhere.
 * ukfb_get_body_states = getCurrentState + toRigidBodyState (:28-39): velocity = orientation * body velocity (rotated
 * into the navigation frame), all else copied; the covariance blocks are NOT rotated. */
#define UKFB_RBS_DOUBLES 49
int ukfb_initialize_from_body_states(ukfb_handle* h, const double* rbs);
int ukfb_initialize_from_body_states_dev(ukfb_handle* h, const double* d_rbs);
int ukfb_get_body_states(ukfb_handle* h, double* rbs);
int ukfb_get_body_states_dev(ukfb_handle* h, double* d_rbs);

/* set/getProcessNoiseCovariance (:129-130).  per_filter = 0: Q is n x n and is
 * broadcast; 1: B x n x n.  The lower triangle is used. */
int ukfb_set_process_noise(ukfb_handle* h, const double* Q, int per_filter);
int ukfb_get_process_noise(ukfb_handle* h, double* Q, int per_filter);

/* set/getMin/MaxTimeDelta (:134-137) */
int ukfb_set_time_bounds(ukfb_handle* h, double min_dt, double max_dt);
int ukfb_get_time_bounds(const ukfb_handle* h, double* min_dt, double* max_dt);

/* set/getLastMeasurementTime (:131-133), int64 microseconds like base::Time. */
int ukfb_set_last_time(ukfb_handle* h, const int64_t* ts_us, int per_filter);
int ukfb_get_last_time(ukfb_handle* h, int64_t* ts_us);

/* The `accept` functor slot of ukfom::ukf::update.  The reference always passes
 * ukfom::accept_any_mahalanobis_distance (PoseUKF.cpp:116, OrientationUKF.cpp:69-71): that is the default here,
 * max_d2 = +inf.  A finite max_d2 gives ukfom::accept_mahalanobis_distance(max_d2) for every later update of this
 * handle: a measurement whose squared Mahalanobis distance innov^T S^-1 innov exceeds it is not integrated (state and
 * covariance untouched) and the filter's UKFB_STATUS_MEAS_REJECTED bit is set. */
int ukfb_set_mahalanobis_gate(ukfb_handle* h, double max_d2);
int ukfb_get_mahalanobis_gate(const ukfb_handle* h, double* max_d2);

/* OrientationUKF constructor arguments gyro_bias_tau, acc_bias_tau, location.latitude
 * (OrientationUKF.cpp:41-47): earth_rotation = (EARTHW cos lat, 0, EARTHW sin lat). */
int ukfb_set_orientation_params(ukfb_handle* h, double gyro_bias_tau, double acc_bias_tau, double latitude);
/* the same constructor arguments, one set per filter (B values each): every OrientationUKF object of the reference is
 * built with its own time constants and location. */
int ukfb_set_orientation_params_per_filter(ukfb_handle* h, const double* gyro_bias_tau, const double* acc_bias_tau,
                                           const double* latitude);

/* ---- predict -------------------------------------------------------------- */

/* predictionStep(delta_t) (:107-125) -> predictionStepImpl (PoseUKF.cpp:180-196 /
 * OrientationUKF.cpp:79-89) -> ukfom::ukf::predict.  dt: B values, or 1 when per_filter = 0. */
int ukfb_predict_dt(ukfb_handle* h, const double* dt, int per_filter);
int ukfb_predict_dt_dev(ukfb_handle* h, const double* d_dt, int per_filter);

/* predictionStepFromSampleTime(sample_time) (:83-100). */
int ukfb_predict_time(ukfb_handle* h, const int64_t* ts_us, int per_filter);
int ukfb_predict_time_dev(ukfb_handle* h, const int64_t* d_ts_us, int per_filter);

/* ---- measurements ----------------------------------------------------------- */

/* integrateMeasurement(<kind>) -> ukfom::ukf::update (PoseUKF.cpp:112-173,
 * OrientationUKF.cpp:65-72).  mu: B x m; cov: B x m x m, or m x m when
 * cov_per_filter = 0; mask: B bytes (0 = this filter has no such measurement now)
 * or NULL for all.  m = ukfb_meas_dim(kind). */
int ukfb_update(ukfb_handle* h, int meas_kind, const double* mu, const double* cov, int cov_per_filter,
                const uint8_t* mask);
/* A sensor's covariance rarely changes between samples.  ukfb_set_measurement_cov keeps one covariance for
 * `meas_kind` on the device (m x m, or B x m x m when per_filter = 1); afterwards the host-pointer calls ukfb_update,
 * ukfb_step and ukfb_step_async accept cov = NULL for that kind and use the kept one (cov_per_filter is then ignored),
 * so a streaming caller only sends the measurement vectors.  Same results as passing the covariance every time. */
int ukfb_set_measurement_cov(ukfb_handle* h, int meas_kind, const double* cov, int per_filter);
int ukfb_update_dev(ukfb_handle* h, int meas_kind, const double* d_mu, const double* d_cov, int cov_per_filter,
                    const uint8_t* d_mask);
int ukfb_meas_dim(int meas_kind);

/* Asynchronous mixed measurements (BASELINE.json config 5): kinds[b] is the kind
 * filter b integrates now (UKFB_MEAS_NONE = none).  mu: B x 3 and cov: B x 3 x 3,
 * the leading m / m x m block of each slot is used. */
/* (a kind of the other filter class: UKFB_ERR_INVALID from the host-pointer call, which can read the array; ignored and
 * flagged UKFB_STATUS_BAD_EVENT by the `_dev` call, whose kinds live on the device) */
int ukfb_update_mixed(ukfb_handle* h, const int8_t* kinds, const double* mu3, const double* cov33);
int ukfb_update_mixed_dev(ukfb_handle* h, const int8_t* d_kinds, const double* d_mu3, const double* d_cov33);

/* PoseUKF::integrateMeasurement(AccelerationMeasurement) (PoseUKF.cpp:175-178): stored
 * unchecked for the next predict; OrientationUKF::integrateMeasurement(Acceleration)
 * (OrientationUKF.cpp:59-63): finite-checked, then stored.  mu: B x 3, cov: B x 3 x 3
 * (or 3 x 3).  cov may be NULL = identity (Measurement.hpp:11). */
int ukfb_set_acceleration(ukfb_handle* h, const double* mu, const double* cov, int cov_per_filter,
                          const uint8_t* mask);
int ukfb_set_acceleration_dev(ukfb_handle* h, const double* d_mu, const double* d_cov, int cov_per_filter,
                              const uint8_t* d_mask);
/* OrientationUKF::integrateMeasurement(RotationRate) (OrientationUKF.cpp:53-57). */
int ukfb_set_rotation_rate(ukfb_handle* h, const double* mu, const double* cov, int cov_per_filter,
                           const uint8_t* mask);
int ukfb_set_rotation_rate_dev(ukfb_handle* h, const double* d_mu, const double* d_cov, int cov_per_filter,
                               const uint8_t* d_mask);
/* OrientationUKF::getRotationRate() (OrientationUKF.cpp:74-77): out B x 3. */
int ukfb_get_rotation_rate(ukfb_handle* h, double* out);

/* ---- fused step ------------------------------------------------------------- */

/* predictionStep(dt) followed by integrateMeasurement(kind) in ONE kernel launch; the
 * state makes one HBM round trip.  Same results as ukfb_predict_dt + ukfb_update. */
int ukfb_step(ukfb_handle* h, const double* dt, int dt_per_filter, int meas_kind, const double* mu,
              const double* cov, int cov_per_filter, const uint8_t* mask);
int ukfb_step_dev(ukfb_handle* h, const double* d_dt, int dt_per_filter, int meas_kind, const double* d_mu,
                  const double* d_cov, int cov_per_filter, const uint8_t* d_mask);

/* Pipelined host-pointer variants for streaming callers (the aggregator callbacks of the reference's oroGen tasks
 * deliver one sample set per tick): same arguments and results as ukfb_step / ukfb_get_state, but the calls only
 * enqueue.  Inputs travel on a copy-in stream into one of two staging slots while the previous step's kernel runs;
 * estimates are unpacked after the steps issued so far and travel on a copy-out stream while later steps run.
 * Host arrays (pinned memory for true overlap) must stay valid and unchanged until ukfb_synchronize(), which is also
 * when mu / sigma hold the estimates. */
int ukfb_step_async(ukfb_handle* h, const double* dt, int dt_per_filter, int meas_kind, const double* mu,
                    const double* cov, int cov_per_filter, const uint8_t* mask);
int ukfb_get_state_async(ukfb_handle* h, double* mu, double* sigma);

/* K consecutive fused steps with the state resident on chip between them.
 * dt: K x B (or K when dt_per_filter = 0); kinds: K measurement kinds (one per tick,
 * UKFB_MEAS_NONE = predict only); mu3: K x B x 3; cov33: K x B x 3 x 3, or K x 3 x 3
 * when cov_per_filter = 0.  For ORIENTATION handles imu: K x B x 6 (gyro xyz, acc xyz)
 * is stored before each predict (may be NULL). */
int ukfb_run_dev(ukfb_handle* h, int K, const double* d_dt, int dt_per_filter, const int8_t* kinds_host,
                 const double* d_mu3, const double* d_cov33, int cov_per_filter, const double* d_imu);

/* Event streams: the device-side form of the reference's caller loop.  The oroGen tasks around the reference run one
 * aggregator callback per sensor sample, in timestamp order, each doing
 *     filter.predictionStepFromSampleTime(ts);  filter.integrateMeasurement(sample);
 * (UnscentedKalmanFilter.hpp:83-100, PoseUKF.cpp:112-178, OrientationUKF.cpp:53-72).  Here every filter has its own
 * queue of such samples, K slots deep, slot-major:  ts[k * B + b] (int64 microseconds), kinds[k * B + b] (a
 * UKFB_MEAS_* kind of this filter class, a storing UKFB_EVENT_* kind, UKFB_MEAS_NONE = advance the time only, or
 * UKFB_EVENT_IDLE = filter b has no sample in slot k: nothing happens, not even the time latch), mu3[(k * B + b) * 3]
 * (the leading m values are used).  Covariances: cov_mode 0 = one table cov[UKFB_EVENT_KIND_COUNT][3][3] indexed by
 * kind (a sensor's covariance, leading m x m block), 1 = one per event, cov[(k * B + b) * 9].
 * All K slots of all filters run in ONE kernel launch with the filter state resident on chip; time guards, the
 * first-call latch, finite checks and status bits behave per event as in the single calls.  A sample whose time step is
 * negative or above max_dt is flagged (UKFB_STATUS_NEG_DT / DT_TOO_LARGE) and NOT integrated or stored: the reference's
 * callback leaves at the throw of predictionStep (:110-122), before its integrateMeasurement.  A kind the filter class
 * has no overload for is ignored and flagged UKFB_STATUS_BAD_EVENT. */
int ukfb_run_events_dev(ukfb_handle* h, int K, const int64_t* d_ts_us, const int8_t* d_kinds, const double* d_mu3,
                        const double* d_cov, int cov_mode);
int ukfb_run_events(ukfb_handle* h, int K, const int64_t* ts_us, const int8_t* kinds, const double* mu3,
                    const double* cov, int cov_mode);
/* the same, enqueue only (rules of ukfb_step_async: pinned host arrays that stay valid until ukfb_synchronize; the
 * queues of the next window are copied while the current one is being integrated) */
int ukfb_run_events_async(ukfb_handle* h, int K, const int64_t* ts_us, const int8_t* kinds, const double* mu3,
                          const double* cov, int cov_mode);

/* ---- status ------------------------------------------------------------------ */

int ukfb_get_status(ukfb_handle* h, uint32_t* flags); /* B words */
int ukfb_clear_status(ukfb_handle* h);
/* number of filters with any status bit set, and the OR of all words */
int ukfb_status_summary(ukfb_handle* h, int64_t* n_flagged, uint32_t* any_bits);
/* histogram of sigma_points_mean pass counts since the last clear: hist[k] = number
 * of state-mean loops that ran k passes (k = 1..7, 7 = "7 or more"; hist[0] unused). */
int ukfb_get_mean_iter_hist(ukfb_handle* h, uint64_t hist[8]);
int ukfb_clear_mean_iter_hist(ukfb_handle* h);

/* ---- per-filter access ------------------------------------------------------------------------------------------ */
/* A caller of the reference owns N filter objects and calls initializeFilter (UnscentedKalmanFilter.hpp:40-44) or
 * getCurrentState (:51-75) on the ONE it needs; these calls do that for the filters idx[0..n) of a batch and touch
 * nothing else (a filter whose status shows UKFB_STATUS_NOT_SPD fails every later factorisation: re-initialising it,
 * then clearing its status, is how it comes back without disturbing the others).
 *   - idx: n int64 GLOBAL filter indices (also on a sharded handle), in any order; row k of every data array belongs to
 *     filter idx[k].  n = 0 is a no-op returning UKFB_OK (null pointers allowed then).
 *   - host-pointer calls check n < 0, null pointers with n > 0, indices outside [0, B) and (ukfb_initialize_indexed)
 *     duplicates, and return UKFB_ERR_INVALID before anything is enqueued: a rejected call changes nothing, on any
 *     shard.  They stage n rows, never B.
 *   - `_dev` calls take device indices and cannot report per-index errors: they require valid indices (unique for
 *     initialize).  An index outside [0, B) is skipped (its row is neither read nor written); duplicates in initialize
 *     leave those filters' records unspecified.  On a sharded parent they return UKFB_ERR_INVALID, as every `_dev` call.
 *   - all work is plain launches and cudaMemcpyAsync on the handle's stream, in full stream order with the step
 *     launches before and after (also where those overlap one another tile by tile, see ukfb_overlapped_launch_count).
 */
/* getCurrentState of filters idx[0..n): mu n x MU, sigma n x n x n (full symmetric, as ukfb_get_state) or NULL.
 * Duplicates allowed.  Bit for bit the rows idx[k] of ukfb_get_state. */
int ukfb_get_state_indexed(ukfb_handle* h, int64_t n, const int64_t* idx, double* mu, double* sigma);
int ukfb_get_state_indexed_dev(ukfb_handle* h, int64_t n, const int64_t* d_idx, double* d_mu, double* d_sigma);
/* initializeFilter of filters idx[0..n) only: record replaced (mu, lower triangle of sigma), t_last = 0 (:43).
 * Q, the stored acceleration / rotation rate, orientation parameters, status words and every other filter are
 * untouched: status is left alone exactly as ukfb_initialize leaves it, recovery clears it explicitly.  The handle must
 * already be initialized (the first ukfb_initialize also does the OrientationUKF constructor's defaults):
 * UKFB_ERR_NOT_INITIALIZED otherwise. */
int ukfb_initialize_indexed(ukfb_handle* h, int64_t n, const int64_t* idx, const double* mu, const double* sigma);
int ukfb_initialize_indexed_dev(ukfb_handle* h, int64_t n, const int64_t* d_idx, const double* d_mu, const double* d_sigma);
/* filters whose status word has any bit of `bits`, ascending; the first min(max_n, count) are written to idx,
 * *n_found = count (idx may be NULL when max_n = 0: count only) */
int ukfb_find_status(ukfb_handle* h, uint32_t bits, int64_t max_n, int64_t* idx, int64_t* n_found);
/* status words of filters idx[0..n) set to 0 (ukfb_clear_status for a subset); duplicates allowed */
int ukfb_clear_status_indexed(ukfb_handle* h, int64_t n, const int64_t* idx);

/* ---- checkpoint / restore ---------------------------------------------------------------------------------------- */
/* One image of everything a batch holds for its filters, so that a stopped job resumes exactly where it stopped, on the
 * same or another number of devices and with any kernel family (UKFB_KERNEL):  records (mu, sigma), t_last, status
 * words, the stored acceleration / IMU sample, Q, per-filter orientation parameters, kept measurement covariances, and
 * the handle-wide values (time bounds, gate, orientation parameters, mean-pass histogram, initialized / first-init).
 * Launch configuration, pipeline slots, launch counters and the launch-overlap counters are not filter state and are
 * not saved.
 *
 * Image: a flat little-endian byte buffer, a 768-byte header, then one section per array.
 *   header    offset  type         field
 *             0       char[8]      magic "UKFBCKPT"
 *             8       uint32       version (UKFB_CHECKPOINT_VERSION)
 *             12      uint32       header bytes (768)
 *             16      uint64       total bytes of the image
 *             24      int32 x 3    kind, MU, n
 *             36      uint32       number of section-table entries (UKFB_CKPT_SECTIONS)
 *             40      int64        B
 *             48      uint32 x 2   initialized, first_init (0 / 1)
 *             56      double x 2   min_dt, max_dt
 *             72      double       Mahalanobis gate
 *             80      double x 6   tau_g, tau_a, latitude, earth[3] (the handle-wide orientation parameters)
 *             128     uint64 x 8   mean-pass histogram (ukfb_get_mean_iter_hist: summed over the handle's slots and shards)
 *             192     uint32 x 2   Q per filter (0 / 1), per-filter orientation parameters present (0 / 1)
 *             200     uint32 x 10  kept covariance of measurement kind k (ukfb_set_measurement_cov): 0 none,
 *                                  1 broadcast, 2 per filter
 *             240     16 zero bytes
 *             256     18 x 24      section table, entry i for section id i: uint32 id, uint32 0, uint64 offset,
 *                                  uint64 bytes; an absent section has offset 0 and bytes 0
 *   sections, at 256-byte aligned offsets in id order, filter-major, all B filters in global filter order:
 *     id 0        records       REC doubles per filter: mu, then the packed lower triangle of sigma (tri(r, c) order)
 *     id 1        t_last        int64
 *     id 2        status        uint32
 *     id 3, 4, 5  acc_mu (3), acc_cov (9), gyro_mu (3) doubles: the stored samples, NaN sentinel of PoseUKF included
 *     id 6        Q             the packed lower triangle (n (n + 1) / 2 doubles) per filter, or once when broadcast
 *     id 7        orientation parameters, 5 doubles per filter (-1/tau_g, -1/tau_a, earth xyz as stored); only if present
 *     id 8 + k    kept covariance of measurement kind k, m x m per filter, or once when broadcast; only if kept
 * The bytes of an image depend on the filters' state alone: not on the shard count, nor on the kernel family.  Per filter:
 * 860 bytes (PoseUKF) / 972 (OrientationUKF), + 624 / 728 with per-filter Q, + 40 with per-filter orientation parameters.
 *
 *   ukfb_checkpoint_size: bytes of this handle's image now (the modes above decide it).
 *   ukfb_checkpoint_save: UKFB_ERR_NOT_INITIALIZED on a handle never initialized; UKFB_ERR_INVALID for a null buffer or
 *     one smaller than ukfb_checkpoint_size.
 *   ukfb_checkpoint_restore: checks magic, version, kind, B, MU, n, every section's offset and size against the header's
 *     modes, and that the image fits `bytes`, before anything is enqueued on any shard: a rejected image (UKFB_ERR_INVALID)
 *     leaves the handle unchanged.  Then replaces every per-filter and handle-wide value above, reallocating Q, the
 *     orientation parameters and kept covariances whose mode differs, as the setters do; initialized / first_init come
 *     from the image (a later ukfb_initialize of a restored OrientationUKF handle does not apply the constructor's
 *     defaults again).  On a sharded handle shard i reads / writes rows [first_i, first_i + count_i) of every section;
 *     handle-wide values are saved from shard 0; a restored histogram goes to shard 0 whole.  An image of any shard
 *     count restores onto any other.
 *   `_dev` variants: the image in device memory of the handle's device (UKFB_ERR_INVALID on a sharded parent).  The save
 *     only enqueues; the restore reads the header (with a broadcast Q behind it) back in one small synchronous copy to
 *     validate it, the payload stays on the device: an in-device snapshot and rollback.
 *   Host-pointer calls move the record section through a device buffer of at most 64 MiB (kept by the handle, as every
 *   staging buffer); the other sections go straight between the caller's buffer and the handle's arrays.  A restore
 *   allocates every array whose size changes before it frees the old one: UKFB_ERR_NOMEM leaves a one-device handle as it
 *   was; on a sharded handle it names the shard that failed, the other shards are restored.
 * All work is plain launches and cudaMemcpyAsync on the handle's stream, in full stream order with earlier _async calls
 * and with step launches that overlap one another tile by tile. */
#define UKFB_CHECKPOINT_VERSION 1
#define UKFB_CKPT_HEADER_BYTES 768
#define UKFB_CKPT_SECTIONS 18
int ukfb_checkpoint_size(ukfb_handle* h, uint64_t* bytes);
int ukfb_checkpoint_save(ukfb_handle* h, void* buf, uint64_t bytes);
int ukfb_checkpoint_restore(ukfb_handle* h, const void* buf, uint64_t bytes);
int ukfb_checkpoint_save_dev(ukfb_handle* h, void* d_buf, uint64_t bytes);
int ukfb_checkpoint_restore_dev(ukfb_handle* h, const void* d_buf, uint64_t bytes);

/* ---- stream plumbing ------------------------------------------------------- */

int ukfb_synchronize(ukfb_handle* h);
/* the handle's cudaStream_t, as an opaque pointer (NULL for a sharded handle: see ukfb_shard) */
void* ukfb_stream(ukfb_handle* h);
/* Ordering against the caller's own CUDA streams, for the `_dev` entry points (they enqueue on the handle's stream, a
 * cudaStreamNonBlocking stream that does not synchronise with the legacy default stream either):
 *   ukfb_wait_for_stream: work enqueued on the handle from now on starts after everything enqueued so far on
 *     `cuda_stream` (a cudaStream_t; NULL = the legacy default stream) -- call it after producing `_dev` inputs;
 *   ukfb_stream_wait: work enqueued on `cuda_stream` from now on starts after everything enqueued so far on the
 *     handle -- call it before consuming `_dev` outputs (ukfb_get_state_dev, ...). */
int ukfb_wait_for_stream(ukfb_handle* h, void* cuda_stream);
int ukfb_stream_wait(ukfb_handle* h, void* cuda_stream);
/* CUDA events on the handle's stream, slots 0..15 */
int ukfb_event_record(ukfb_handle* h, int slot);
int ukfb_event_elapsed_ms(ukfb_handle* h, int slot_begin, int slot_end, float* ms);
/* number of engine kernels launched on this handle since creation */
int64_t ukfb_launch_count(const ukfb_handle* h);
/* ... and how many of them were launched to overlap with their predecessor.  Nothing in the reference corresponds to
 * this: its filters are stepped one call after the other (UnscentedKalmanFilter.hpp:83-125).  Here consecutive step
 * launches of one handle are ordered TILE BY TILE (a tile of 32 filters of launch n waits for the same tile of launch
 * n - 1) instead of launch by launch, so launch n starts in the multiprocessor slots the last, partial wave of launch n - 1
 * leaves empty.  Results are bit for bit those of launches in stream order; every other operation of the stream (copies,
 * get_state, ...) keeps full stream order.  The engine launches this way when the handle's batch is between 1 and
 * UKFB_OVERLAP_MAX_WAVES (12) waves of resident warps -- a shard of 40 Ki to 450 Ki filters on a B200 -- where it gains 4 to
 * 20 %; UKFB_OVERLAP_LAUNCHES=0 in the environment turns it off. */
int64_t ukfb_overlapped_launch_count(const ukfb_handle* h);
/* peak of an unrolled independent-DFMA microkernel on the handle's device, in
 * FLOP/s (FMA = 2), the FP64 roofline denominator (BASELINE.md section 2). */
int ukfb_measure_fp64_peak(ukfb_handle* h, double* flops_per_s);
/* self-test of the device arithmetic the kernels are built on (csrc/so3.cuh, csrc/simt.cuh): for i < n, with
 * o = out + UKFB_SELFTEST_STRIDE i:  o[0..3] = SO3 exp(v[3 i ..]) (x, y, z, w), o[4..6] = SO3 log of that quaternion,
 * o[7] = 1 / x[i], o[8], o[9] = sqrt(x[i]), 1 / sqrt(x[i]); o[10..12] = the fast kernels' branch-free log (no reciprocal)
 * of their polynomial exp of v, o[13] = 1 if v lies outside the range of that pair (the kernels then use the any-angle
 * pair), else 0; o[14..17] = the any-angle exp of v, o[18..20] = the any-angle log of that quaternion.
 * tests/ compare them with extended-precision values. */
#define UKFB_SELFTEST_STRIDE 21
int ukfb_selftest_so3(ukfb_handle* h, int64_t n, const double* v, const double* x, double* out);

#ifdef __cplusplus
}
#endif

#endif /* UKF_BATCH_H */
