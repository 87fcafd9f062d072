/* rbis_batch.h -- C ABI of the B200-native batched RBIS EKF (drop-in boundary).
 *
 * One handle = one ensemble of N independent 21-state RBIS filters resident on one B200.  Every
 * entry point replaces, for a whole ensemble at once, one piece of the reference's per-filter
 * interface under /root/reference/state-estimator/src/mav_state_est/ (cited per function as
 * MSE/<file>:<lines>).  Plain pointers and sizes only; no C++/torch types; never throws.
 *
 * Conventions
 *   - All floating point is IEEE double.  Indices are int32, time is int64 microseconds.
 *   - Ensemble arrays are structure-of-arrays with the FILTER INDEX FASTEST:
 *       vec  [21][N]   state vector, index layout of RBIS (MSE/rbis.hpp:22-24 + eigen_utils):
 *                      0-2 angular velocity, 3-5 body velocity, 6-8 chi, 9-11 position,
 *                      12-14 acceleration, 15-17 gyro bias, 18-20 accel bias
 *       quat [4][N]    orientation (w,x,y,z)
 *       cov  [441][N]  RBIM, element (r,c) at row r + 21*c (Eigen column-major, MSE/rbis.hpp:30,123)
 *       imu  [rows][6][N]  gyro xyz then accelerometer xyz per IMU sample row
 *       z    [rows][m][N], meas quat [rows][4][N]     (N -> cols under rbis_batch_set_column_map)
 *   - `mem` says where the caller's ensemble arrays live: host memory (copied by the library on the
 *     handle's stream; use pinned memory for truly asynchronous copies) or device memory (used in
 *     place; must stay valid until the call's work has completed).
 *   - Lifetime of host inputs: a call that takes host arrays with mem == RBIS_MEM_HOST returns once the copies are ENQUEUED
 *     (pageable memory is staged by the CUDA runtime before the call returns; PINNED memory is read later, by the copy
 *     engine).  Pinned input arrays of rbis_batch_run_fused must therefore stay valid and unchanged until a later
 *     rbis_batch_synchronize(), or a rbis_batch_wait() on a ticket recorded after the call, has returned.
 *   - Calls are stream-ordered on the handle and return once enqueued unless stated otherwise;
 *     rbis_batch_synchronize() waits.  A handle is not thread-safe (the reference is single
 *     threaded too: MSE/lcm_front_end.cpp:223-229).
 *   - Return value: 0 on success, negative rbis_status_t on error; rbis_last_error() gives the text.
 *   - The covariance is kept symmetric-packed on the device (upper triangle of `cov` is read on
 *     input; both triangles are written on output).  The reference never symmetrises, but its
 *     covariance is symmetric to rounding by construction.
 *   - There is no CPU fallback: every compute entry point runs CUDA kernels built for sm_100a and
 *     fails with RBIS_ERR_CUDA when no such device is present.
 */
#ifndef RBIS_BATCH_H_
#define RBIS_BATCH_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RBIS_NUM_STATES 21
#define RBIS_COV_ELEMS 441
#define RBIS_MAX_MEAS 9      /* largest index set any reference handler emits (SE/gpf/laser_gpf_lib.cpp:108-110) */
#define RBIS_MAX_STREAMS 8
#define RBIS_NUM_STATS 96    /* doubles per statistics chunk, see rbis_batch_stats */

typedef struct rbis_batch rbis_batch_t;

typedef enum {
  RBIS_OK = 0,
  RBIS_ERR_INVALID = -1,  /* bad argument */
  RBIS_ERR_CUDA = -2,     /* CUDA runtime failure, or no sm_100 device */
  RBIS_ERR_ALLOC = -3,
  RBIS_ERR_STATE = -4     /* call sequence error (e.g. restore of an empty snapshot slot) */
} rbis_status_t;

typedef enum {
  RBIS_MEM_HOST = 0,
  RBIS_MEM_DEVICE = 1,
  /* rbis_batch_run_fused only, OR-ed with one of the above: the sensor rows (imu, z, quat) are FLOAT arrays of the same shapes.  They
   * are widened to double exactly on the device, so the results equal those of the same values passed as doubles; a host log that is
   * float-valued (most sensor data is) then crosses PCIe in half the bytes.  Per-filter R arrays stay double. */
  RBIS_MEM_F32_ROWS = 4
} rbis_mem_t;

/* Fused-program op kinds. */
typedef enum {
  RBIS_OP_IMU = 0,       /* RBISIMUProcessStep::updateFilter, MSE/rbis_update_interface.cpp:30-52 */
  RBIS_OP_MEAS = 1,      /* RBISIndexed[PlusOrientation]Measurement::updateFilter, :54-107 */
  RBIS_OP_SNAPSHOT = 2,  /* save (state, cov, loglik) of every filter into ring slot `row` */
  RBIS_OP_RESTORE = 3,   /* load them back: the history rewind of MSE/mav_state_est.cpp:35-70 */
  RBIS_OP_RECORD = 4     /* write the fields of the handle's record set (rbis_batch_set_record) of every filter into record row
                            `row`: the trajectory a replay publishes (MSE/lcm_front_end.cpp:144-166).  Changes neither the filters
                            nor the ensemble's utime; `stream` and `dt` are ignored */
} rbis_op_kind_t;

typedef enum {
  RBIS_R_SHARED_FULL = 0,      /* one m x m column-major matrix for all filters (HOST pointer always) */
  RBIS_R_PER_FILTER_DIAG = 1,  /* diagonal, [m][N], located as `mem` says */
  RBIS_R_PER_ROW_FULL = 2      /* HOST [rows][m][m]: row r (column-major like the shared matrix) is the covariance of the update that
                                  reads row r of the stream -- the measurement_cov each RBISIndexed[PlusOrientation]Measurement carries
                                  (MSE/rbis_update_interface.hpp:90-96,111-117), e.g. leg odometry switching between its certain and
                                  uncertain R, or indexed_measurement_t's R_effective per message.  Shared by all filters as the log is;
                                  column maps do not apply to it.  The m rows are cut into chunks along the union of the off-diagonal
                                  non-zeros of all rows of the call, so rows that all equal one R run exactly as RBIS_R_SHARED_FULL
                                  with that R (same chunks, same kernel variant, same bits).  rbis_batch_run_fused and
                                  rbis_batch_run_fused_synth only: the single-update entry points reject it (one update has one R). */
} rbis_r_mode_t;

typedef struct {
  double g_val;            /* eigen_utils g_val, g_vec = (0,0,-g_val); default 9.8 (SURVEY.md 8c) */
  double chi_tol;          /* eigen_utils chiToQuat tolerance; default 1e-6 */
  int32_t ctor_folds_chi;  /* RigidBodyState(VectorXd) ctor folds chi into its quaternion; default 1 */
  int32_t renormalize_quat;/* 0 = reference behaviour (never renormalises, MSE/rbis.cpp:219-227);
                              1 = renormalise the quaternion after every applied delta */
  int32_t snapshot_slots;  /* ring slots for RBIS_OP_SNAPSHOT / RESTORE; 0 = none */
  int32_t device;          /* CUDA device ordinal */
  int32_t launch_groups;   /* fused launches are split into this many CTA ranges on separate streams so that
                              consecutive rbis_batch_run_fused calls overlap and the last, partially filled wave of
                              one launch does not idle SMs; 0 = automatic (6 when the CTAs do not fill whole
                              waves, else 1), 1 = off, max 8 */
  int32_t dense_only;      /* 0 (default) = automatic: fused programs run the "decoupled" kernel variant (only the
                              15x15 block of v, chi, p, b_g, b_a on chip, 384 filters per SM) whenever every filter's
                              covariance couplings to the omega / a rows are exactly zero -- true for every filter
                              started from the reference's diagonal initial covariance (MSE/rbis_initializer.cpp:85-91)
                              until a measurement indexes omega or a -- and no stream of the program indexes omega or a;
                              results are bit-identical to the dense variant.
                              1 = always run the dense variant (whole covariance on chip, 256 filters per SM). */
  int32_t mapping;         /* lanes that cooperate on one filter in the fused kernels.  1 = the lane-per-filter kernels (a
                              B200 needs ~57,000 filters to fill them); 2, 4, 8, 16 = the warp-group kernels for small or
                              split ensembles (BASELINE configs[1], a 65,536-filter ensemble sharded over 8 GPUs): the
                              covariance products of MSE/rbis.cpp:113-118,134-140 are split over the lanes of a group, the
                              covariance is carried as a full matrix in shared memory.
                              0 (default) = automatic by ensemble size.  Results of the two mappings agree
                              BIT FOR BIT (every covariance element is computed by the same expression in both;
                              tests/test_gpu_group.py), so the choice is invisible in the results. */
  int32_t lane_filters_per_cta; /* filters per CTA of the decoupled lane-per-filter kernels: 384 (three warps per scheduler, for
                              ensembles that fill the GPU), 256 or 128 (more SMs busy for 10-50 thousand filters); 0 = automatic.
                              Same bits for every value. */
  int32_t piece_ops;       /* with launch groups, a fused program of >= 2 * piece_ops ops is cut into consecutive pieces of about
                              this many ops over the same inputs, each piece one set of launches, so that the partially filled last
                              wave of CTAs of a piece overlaps the next piece (rbis_batch.cu).  0 = automatic (256).  Smaller
                              pieces (64-100) pay when the caller reads a result after every call, which keeps consecutive CALLS
                              from overlapping; results do not depend on it. */
  int32_t synth_materialize; /* rbis_batch_run_fused_synth: 0 (default) = decoupled programs with the fast generator (rbis_synth_t::mode 1)
                              draw their input rows INSIDE the fused kernel -- no per-filter input exists in HBM; 1 = always generate
                              the rows into device buffers first and run the ordinary fused kernels over them.  Same bits either way
                              (tests/test_gpu_synth.py). */
} rbis_batch_config_t;

/* One measurement stream = the constant part of an RBISIndexedMeasurement /
 * RBISIndexedPlusOrientationMeasurement constructor (MSE/rbis_update_interface.hpp:90-96,111-117)
 * plus where its per-row data live (with RBIS_R_PER_ROW_FULL the measurement covariance is per-row data too). */
typedef struct {
  int32_t m;                      /* 1..RBIS_MAX_MEAS */
  int32_t has_orientation;        /* 0 indexedMeasurement, 1 indexedPlusOrientationMeasurement */
  int32_t r_mode;                 /* rbis_r_mode_t */
  int32_t sensor_id;              /* RBISUpdateInterface::sensor_enum value, carried only */
  int32_t idx[RBIS_MAX_MEAS];     /* state indices, 0..20 */
  int32_t flags;                  /* RBIS_STREAM_* bits; 0 = none (every other bit is rejected) */
  const double* z;                /* [rows][m][N]; entries at chi indices are ignored when has_orientation */
  const double* quat;             /* [rows][4][N] or NULL */
  const double* R;                /* see rbis_r_mode_t */
  int64_t rows;
} rbis_stream_t;

/* rbis_stream_t::flags.
 * RBIS_STREAM_SKIP_NAN_ROWS: rows that some filters did not receive (sensor dropouts that differ from one realisation to the next,
 *   logs whose gaps fall in different places).  Row r is MISSING for filter n when any z value the update reads in filter n's
 *   column -- the column-map column where a map is set -- is NaN; the chi entries of an orientation stream are not read and do not
 *   count, quat is not inspected.  For that filter the RBIS_OP_MEAS op of row r does nothing: state, quaternion, covariance and
 *   log-likelihood keep their bits, and no addState runs (so renormalize_quat does not renormalise either).  Every other filter,
 *   the ensemble's utime, SNAPSHOT, RESTORE and RECORD proceed as usual.  Hence for an in-order or planner-built program, filter n
 *   ends exactly where the same program ends with the MEAS ops of its missing rows deleted.  Without the flag a NaN is used
 *   as a value (and poisons the filter).  rbis_batch_run_fused only (any mem, r_mode, chunk kind, column map, mapping);
 *   rbis_batch_run_fused_synth rejects it, its rows are drawn, not read. */
#define RBIS_STREAM_SKIP_NAN_ROWS 1

typedef struct {
  int32_t kind;    /* rbis_op_kind_t */
  int32_t stream;  /* RBIS_OP_MEAS: stream number */
  int64_t row;     /* IMU / MEAS: row in the stream; SNAPSHOT / RESTORE: ring slot; RECORD: record row */
  int64_t utime;   /* becomes the ensemble's utime (MSE/mav_state_est.cpp:60) */
  double dt;       /* RBIS_OP_IMU only */
} rbis_op_t;

const char* rbis_last_error(void);
void rbis_default_config(rbis_batch_config_t* cfg);

/* ---- lifetime: replaces `new MavStateEstimator(new RBISResetUpdate(...))`, MSE/mav_state_est.cpp:12-22.
 * The handle owns all device memory; the caller owns every buffer it passes in. */
int rbis_batch_create(rbis_batch_t** out, int64_t n_filters, const rbis_batch_config_t* cfg);
int rbis_batch_destroy(rbis_batch_t* h);
int rbis_batch_synchronize(rbis_batch_t* h);
int64_t rbis_batch_num_filters(const rbis_batch_t* h);
/* Raw CUDA stream (cudaStream_t) of the handle, for event timing by the caller.  With launch groups the fused
 * kernels run on internal streams that this stream joins at the next non-fused call: to time fused work, call
 * rbis_batch_record() (it joins) and then record the timing event on this stream. */
void* rbis_batch_stream(rbis_batch_t* h);
/* Kernels launched by this handle so far (bench.py's gpu_launches). */
int64_t rbis_batch_launch_count(const rbis_batch_t* h);
/* Kernel variant the last rbis_batch_run_fused / single-op call launched: 0 dense, 2 decoupled (see
 * rbis_batch_config_t::dense_only), +1 when the program has measurement chunks other than uncorrelated aligned index
 * triples (the instantiations that also contain the one-row and the correlated-block updates), +4 when the kernel drew its
 * input rows itself (rbis_batch_run_fused_synth, SYN instantiations), + 16 * lanes per filter for the warp-group kernels
 * (rbis_batch_config_t::mapping > 1), +8 for the REC instantiations, which run when the program records (RBIS_OP_RECORD) or a MEAS op
 * of it writes an innovation set (rbis_batch_set_innovations) and never otherwise, +1024 more when they carry the innovation path
 * (the program writes an innovation set: programs that only record do not run that code), +512 when a stream has RBIS_STREAM_SKIP_NAN_ROWS (the MASK instantiations, which contain the one-row and
 * correlated-block updates whatever +1 says); -1 before the first launch. */
int rbis_batch_last_kernel_variant(const rbis_batch_t* h);

/* ---- RBISResetUpdate::updateFilter (MSE/rbis_update_interface.cpp:23-28): posterior := given,
 * loglikelihood := 0 (or `loglik` [N] when non-NULL).  cov may be NULL to keep the current one. */
int rbis_batch_set_state(rbis_batch_t* h, const double* vec, const double* quat, const double* cov,
                         const double* loglik, int64_t utime, int mem);
/* MavStateEstimator::getHeadState + getMeasurementsLogLikelihood (MSE/mav_state_est.cpp:82-96).
 * Any output pointer may be NULL.  Synchronises when mem == RBIS_MEM_HOST. */
int rbis_batch_get_state(rbis_batch_t* h, double* vec, double* quat, double* cov, double* loglik,
                         int64_t* utime, int mem);
/* Single-filter (array-of-structures) access for the C++ shim: vec[21], quat[4], cov[441]. Synchronous. */
int rbis_batch_set_filter(rbis_batch_t* h, int64_t n, const double* vec, const double* quat, const double* cov,
                          double loglik);
int rbis_batch_get_filter(rbis_batch_t* h, int64_t n, double* vec, double* quat, double* cov, double* loglik);

/* ---- process noise = the q_* constructor arguments of RBISIMUProcessStep
 * (MSE/rbis_update_interface.hpp:70-75); variances, as InsHandler squares them
 * (MSE/sensor_handlers.cpp:18-25).  Either one value for all filters or one per filter. */
int rbis_batch_set_process_noise(rbis_batch_t* h, double q_gyro, double q_accel, double q_gyro_bias,
                                 double q_accel_bias);
int rbis_batch_set_process_noise_per_filter(rbis_batch_t* h, const double* q_gyro, const double* q_accel,
                                            const double* q_gyro_bias, const double* q_accel_bias, int mem);

/* ---- one update for every filter (each is a one-op fused program) ----
 * RBISIMUProcessStep::updateFilter: insUpdateState (MSE/rbis.cpp:37-75) + insUpdateCovariance
 * linearised at the PRIOR state (MSE/rbis.cpp:77-122, rbis_update_interface.cpp:38-39).
 * gyro/accel: [3][N]. */
int rbis_batch_ins_step(rbis_batch_t* h, const double* gyro, const double* accel, double dt, int64_t utime,
                        int mem);
/* indexedMeasurement + rbisApplyDelta (MSE/rbis.cpp:160-178,219-227).  z [m][N]; R per r_mode. */
int rbis_batch_indexed_update(rbis_batch_t* h, int m, const int32_t* idx, const double* z, const double* R,
                              int r_mode, int64_t utime, int mem);
/* indexedPlusOrientationMeasurement + rbisApplyDelta (MSE/rbis.cpp:189-227).  quat [4][N]. */
int rbis_batch_indexed_orient_update(rbis_batch_t* h, int m, const int32_t* idx, const double* z,
                                     const double* quat, const double* R, int r_mode, int64_t utime, int mem);

/* ---- column maps: filters that share input data (parameter sweeps in the style of the reference's noise
 * identification, state-estimator/matlab/ins_noise_opt_script_mex.m:38-61, where every parameter point replays
 * the SAME log; or one noise realisation evaluated under many parameter sets).  While a map is set, the
 * corresponding array handed to rbis_batch_run_fused has `cols` columns instead of N and filter n reads column
 * map[n]:  imu [rows][6][cols]  (which = -1),  z [rows][m][cols] and quat [rows][4][cols] of stream `which` >= 0.
 * map: HOST int32[N] with entries in [0, cols), copied by the call; NULL restores the identity (cols ignored).
 * Per-filter R ([m][N]) and everything else stay per filter.  The one-op entry points above ignore the maps.
 * Synchronises the handle. */
int rbis_batch_set_column_map(rbis_batch_t* h, int which, const int32_t* map, int64_t cols);

/* ---- records: selected per-filter fields at chosen points of a fused program, written from the values the kernel holds on chip.
 * Record row r holds, bit for bit, what an RBIS_OP_SNAPSHOT at the same program position would hold in those fields.  Field f is
 * recorded when bit f of `fields` is set:
 *   0..20  vec[f]        21..24  quat w, x, y, z        25  log-likelihood        26..46  covariance diagonal P(f-26, f-26)
 * After the fields a row can hold covariance BLOCKS: bit b of `cov_blocks` selects state block b, indices 3b..3b+2 (0 omega,
 * 1 v, 2 chi, 3 p, 4 a, 5 gyro bias, 6 accel bias).  With I the ascending selected indices and nb = |I| = 3 popcount(cov_blocks),
 * the packed upper triangle of P restricted to I follows the fields: P(I[ii], I[jj]), ii <= jj < nb, at field position
 * popcount(fields) + jj (jj + 1) / 2 + ii.  With all seven blocks that is the covariance part of a snapshot slot
 * (slot(i, j) = j (j + 1) / 2 + i, 231 entries); {v, chi, p} is the 9x9 block of the NEES, {p, chi} the pose covariance.
 * out is [rows][k][N], k = popcount(fields) + nb (nb + 1) / 2, the chosen fields in ascending bit order, then the covariance
 * entries, filter index fastest; column maps do not apply (records are always per filter).  Inactive filters of a launch write
 * nothing; rows no RECORD op names stay untouched.
 *   RBIS_MEM_DEVICE: the kernels write `out` in place.  It is valid once a ticket recorded after the call has been waited for
 *                    (rbis_batch_record / rbis_batch_wait) or after rbis_batch_synchronize.
 *   RBIS_MEM_HOST:   `out` must be PINNED host memory (pageable memory is rejected: a copy into it would synchronise).  The kernels
 *                    write the distinct rows the call records into a library-owned device staging buffer (double buffered across
 *                    calls), and after the call's launches one asynchronous copy per run of consecutive record rows, on a stream
 *                    of its own, moves them to their rows of `out`; rows between them keep their contents.  The next call's
 *                    launches do not wait for those copies.  `out` is valid, and must stay allocated,
 *                    until a ticket recorded after the call has been waited for or rbis_batch_synchronize has returned. */
typedef struct {
  uint64_t fields;   /* bit f: record field f, f < 47 */
  double* out;       /* [rows][k][N] */
  int64_t rows;
  int32_t mem;       /* RBIS_MEM_DEVICE or RBIS_MEM_HOST (pinned) */
  int32_t cov_blocks; /* bit b < 7: record the covariance block of state block b (0 = none; was a reserved zero field) */
} rbis_record_t;
/* Sets the record set used by the rbis_batch_run_fused / rbis_batch_run_fused_synth calls enqueued after it (handle state, like
 * the column maps; a copy of *rec is kept); NULL clears it.  Does not synchronise, so switching buffers between calls keeps the
 * device busy.  fields and cov_blocks must not both be empty; a cov_blocks bit >= 7 is RBIS_ERR_INVALID.  A RECORD op without a
 * record set fails with RBIS_ERR_STATE, a row outside [0, rows) with RBIS_ERR_INVALID, both before anything is enqueued.  The
 * single-update entry points do not record. */
int rbis_batch_set_record(rbis_batch_t* h, const rbis_record_t* rec);

/* ---- innovation sets: the innovation sequence of every measurement update, the consistency check that needs no truth (a log
 * replay, a sweep of R or Q).  For a MEAS op on a stream with index set idx[0..m-1], from the PRIOR state of the op (x-, P-) as
 * the reference's update forms them (MSE/rbis.cpp:124-143):
 *   y_a    = z_a - x-[idx_a]; at the chi indices of an orientation stream, component idx_a - 6 of subtract_quats(meas_quat, quat)
 *   S(a,a) = P-(idx_a, idx_a) + R(a,a), R's diagonal from the shared table, the row's table (RBIS_R_PER_ROW_FULL) or R[a][n]
 *            (RBIS_R_PER_FILTER_DIAG)
 *   NIS    = y^T S^-1 y with the full S: the sum of the quadratic forms of the update's chunks (the kernels apply an update as
 *            chunks of uncorrelated rows, and decorrelated scalar rows inside a correlated block); by the chain rule of the Gaussian
 *            likelihood that equals the single update's y^T S^-1 y up to rounding.  A consistent filter has NIS ~ chi2(m).
 * out is DEVICE memory [rows][k][N], k = NIS + m Y + m S_DIAG: the chosen fields in the order NIS, y_0..y_m-1, S(0,0)..S(m-1,m-1),
 * filter index fastest.  Every MEAS op on stream slot `stream` of a later rbis_batch_run_fused / rbis_batch_run_fused_synth call
 * writes row op.row for every active filter:
 *   - a filter that skips the row (RBIS_STREAM_SKIP_NAN_ROWS) writes NaN into all k entries;
 *   - a row applied more than once holds the values of its last application (after a RESTORE and replay, the replayed one);
 *   - rows no MEAS op writes keep their contents; column maps do not apply (the values are per filter).
 * `out` is valid once a ticket recorded after the call has been waited for (rbis_batch_record / rbis_batch_wait) or after
 * rbis_batch_synchronize.  The single-update entry points, and calls with fewer than stream + 1 streams, ignore the set. */
#define RBIS_INNOV_NIS    1   /* y^T S^-1 y: 1 entry */
#define RBIS_INNOV_Y      2   /* the innovation y: m entries */
#define RBIS_INNOV_S_DIAG 4   /* S(a,a) = P-(idx_a, idx_a) + R(a,a): m entries */
typedef struct {
  uint32_t fields;   /* RBIS_INNOV_* bits, not 0 */
  int32_t  m;        /* the stream's measurement dimension; a call whose stream `stream` has another m fails */
  double*  out;      /* DEVICE [rows][k][N], k = NIS + m*Y + m*S_DIAG, in that order, filter index fastest */
  int64_t  rows;
} rbis_innovation_t;
/* Sets the innovation set of stream slot `stream` (0..RBIS_MAX_STREAMS-1) used by the fused calls enqueued after it (handle state
 * per slot, like the column maps and the record set; a copy of *spec is kept); NULL clears it.  Does not synchronise.  A bad slot,
 * an unknown or empty `fields`, m outside 1..RBIS_MAX_MEAS and a NULL or non-device `out` are RBIS_ERR_INVALID.  A fused call
 * whose stream `stream` has another m, or whose MEAS op on it names a row outside [0, rows), fails with RBIS_ERR_INVALID before
 * anything is enqueued.  Programs that write an innovation set run the REC kernel instantiations with the innovation path
 * (rbis_batch_last_kernel_variant +8 +1024). */
int rbis_batch_set_innovations(rbis_batch_t* h, int32_t stream, const rbis_innovation_t* spec);

/* ---- the fused hot path: run `n_ops` ops (host array, executed in order) for every filter in ONE
 * kernel launch, state and covariance resident on chip throughout.  This is the batch form of the
 * roll-forward loop MSE/mav_state_est.cpp:50-70.  imu may be NULL when no IMU op is present. */
int rbis_batch_run_fused(rbis_batch_t* h, int64_t n_ops, const rbis_op_t* ops, const double* imu,
                         int64_t imu_rows, int n_streams, const rbis_stream_t* streams, int mem);

/* ---- on-device synthesis of per-filter sensor streams for Monte-Carlo noise sweeps (SURVEY.md 8d): every filter reads the
 * same noise-free log plus its own noise realisation, so the host passes the noise-free rows and a seed and the per-filter
 * rows are produced in HBM, never crossing PCIe.  Counter-based generator, one draw per (seed, GLOBAL filter index, step
 * counter, channel): key = seed ^ filter*K1 ^ step*K2 ^ channel*K3, a = splitmix64(key), b = splitmix64(a), Box-Muller.
 * mode 0 (exact): u1, u2 from 53 bits, sqrt(-2 ln u1) cos(2 pi u2) in double -- pronto_b200/synth.py:normal is its numpy
 * statement (bit-exact integers, libm calls within an ulp or two); mode 1 (fast): same counters and hash, 24-bit uniforms,
 * single-precision SFU ln / sqrt / cos.  Channels follow SURVEY.md 8d: 0-2 gyro, 3-5 accelerometer, then per stream. */
typedef struct {
  int32_t m;                      /* columns of z */
  int32_t has_orientation;        /* also draw a measured orientation: mean_quat (x) Exp(sigma_rot * n) */
  int32_t channel;                /* column a draws channel + a */
  int32_t channel_rot;            /* the rotation perturbation draws channel_rot + 0..2 */
  const double* mean;             /* HOST [rows][m] noise-free rows */
  const double* mean_quat;        /* HOST [rows][4] (w,x,y,z) or NULL */
  const int64_t* step;            /* HOST [rows] counter value of each row (the global time-step index) */
  double sigma[RBIS_MAX_MEAS];    /* standard deviation per column */
  double sigma_rot[3];
  int64_t rows;
} rbis_synth_stream_t;
typedef struct {
  uint64_t seed;
  int64_t first_filter;           /* global index of the handle's filter 0: shards of one ensemble draw the same noise for any GPU count */
  int32_t mode;                   /* 0 exact (double precision, one hash pair per sample: pronto_b200/synth.py:normal), 1 fast (one hash per
                                     PAIR of channels, single-precision Box-Muller; the mode the fused kernels can draw in-kernel) */
  int32_t n_streams;
  const double* imu_mean;         /* HOST [imu_rows][6]: noise-free gyro xyz, accelerometer xyz readings */
  const int64_t* imu_step;        /* HOST [imu_rows] */
  int64_t imu_rows;
  double sigma_gyro, sigma_accel; /* >= 0: standard deviations for all filters; < 0: per filter sqrt(q_gyro / dt), sqrt(q_accel / dt) from
                                     the handle's process noise, i.e. sample noise consistent with Qd = q dt (MSE/rbis.cpp:116) */
  double dt;
  const rbis_synth_stream_t* streams;
} rbis_synth_t;
/* Materialise the streams into DEVICE arrays imu_out [imu_rows][6][N], z_out[s] [rows][m][N], quat_out[s] [rows][4][N]
 * (enqueued on the handle's stream; the host arrays of `syn` are consumed before the call returns).  This is also how a
 * test feeds the CPU oracle exactly what the device drew. */
int rbis_batch_synthesize(rbis_batch_t* h, const rbis_synth_t* syn, double* imu_out, double* const* z_out, double* const* quat_out);
/* rbis_batch_run_fused with synthesised inputs: streams[s].z / .quat / .rows are ignored (taken from syn->streams[s]; a per-filter R
 * is a DEVICE array on this path).  Mode 1 on a decoupled ensemble (rbis_batch_config_t::dense_only): the fused kernel draws every row
 * it consumes itself, from the noise-free row and the filter's counters -- nothing is materialised, the launch reads no per-filter input.
 * Otherwise (mode 0, dense kernels, rbis_batch_config_t::synth_materialize) the rows are generated into library-owned device buffers
 * (double buffered across calls) and consumed by the ordinary fused launch; both ways give the same bits as rbis_batch_synthesize +
 * rbis_batch_run_fused.  Host -> device traffic per call: the op list and the noise-free rows. */
int rbis_batch_run_fused_synth(rbis_batch_t* h, int64_t n_ops, const rbis_op_t* ops, int n_streams, const rbis_stream_t* streams,
                               const rbis_synth_t* syn);

/* ---- delayed measurements: the batch form of MavStateEstimator::addUpdate's out-of-order insert +
 * replay (MSE/mav_state_est.cpp:28-80) over updateHistory's time-ordered multimap
 * (MSE/update_history.cpp:16-54), for an ensemble whose filters share one arrival schedule.
 * The planner keeps the time-ordered list of updates (equal utime keeps arrival order, as the hinted
 * multimap insert does) and turns arrivals into an op program for rbis_batch_run_fused: in-order
 * arrivals append ops; an arrival older than the head becomes RESTORE(nearest earlier snapshot) +
 * the replay of every update from there to the head.  Where the reference keeps a full posterior in
 * every history node, the device keeps a ring of `snapshot_slots` ensemble snapshots taken every
 * `snapshot_period_us` (at utimes u with (u - snapshot_phase_us) % period == 0, after the last
 * update stamped u), plus one at the start.  Updates older than the oldest retained history entry are
 * discarded as in update_history.cpp:28-39; so are updates that no retained snapshot precedes.
 * History is truncated to `history_span_us` behind the newest update after every roll-forward
 * (mav_state_est.cpp:74-77).  The rewind window is therefore ~ snapshot_slots x snapshot_period_us: choose them so that it
 * covers history_span_us when every update the reference would replay must be replayed (rbis_planner_create leaves a
 * warning in rbis_last_error() when it does not; the C++ shim's default does).  Host-side only; no device work.
 *
 * ONE SCHEDULE PER HANDLE.  A planner serves one rbis_batch_t: all of its filters see the same arrivals in the same order --
 * the shape of every workload in BASELINE.json (a noise sweep or a parameter sweep replays ONE log; delayed pose fixes are
 * late for every realisation alike).  One schedule, but rows may be MISSING per filter: with RBIS_STREAM_SKIP_NAN_ROWS a
 * filter whose row is NaN skips that update, so dropouts that differ between realisations stay in one handle and one
 * planner (the program is planned as if every filter received every row).  Filters whose measurements arrive in a
 * different ORDER or with different latency belong in different handles,
 * one planner each: handles are independent (own streams, own snapshot ring), their launches run concurrently on the device,
 * and the warp-group kernels keep small sub-ensembles efficient; tests/test_gpu_parity.py
 * (test_two_arrival_schedules_as_two_handles) runs two schedules side by side against the oracle's per-filter histories. */
typedef struct rbis_planner rbis_planner_t;
int rbis_planner_create(rbis_planner_t** out, int64_t utime0, int32_t snapshot_slots, int64_t snapshot_period_us,
                        int64_t snapshot_phase_us, int64_t history_span_us);
int rbis_planner_destroy(rbis_planner_t* p);
/* addUpdate(update, roll_forward): update->kind is RBIS_OP_IMU or RBIS_OP_MEAS.  Returns 0 = accepted,
 * 1 = discarded (too old), negative = error.  With roll_forward == 0 the update only enters the
 * history; the next roll-forward processes everything outstanding in one replay. */
int rbis_planner_add_update(rbis_planner_t* p, const rbis_op_t* update, int roll_forward);
/* Ops planned so far and not yet taken. */
int64_t rbis_planner_pending(const rbis_planner_t* p);
/* Copy out (and clear) the pending program; fails with RBIS_ERR_INVALID if cap is too small. */
int rbis_planner_take(rbis_planner_t* p, rbis_op_t* out, int64_t cap, int64_t* n_out);
/* Counters: [0] updates accepted, [1] discarded, [2] rewinds, [3] updates replayed (re-applied),
 * [4] snapshots taken, [5] history entries retained. */
int rbis_planner_counters(const rbis_planner_t* p, int64_t out[6]);

/* ---- EKF smoother ("next" row 1 of SURVEY.md 8f): ekfSmoothingStep (MSE/rbis.cpp:234-266) driven as
 * MavStateEstimator::EKFSmoothBackwardsPass (MSE/mav_state_est.cpp:98-189).  Where the reference keeps a posterior in
 * every history node, the ensemble keeps the posteriors it wants smoothed in the snapshot ring: the forward program
 * stores the posterior of update u into ring slot slot[u] with RBIS_OP_SNAPSHOT.
 *
 * rbis_smooth_plan: host-side mirror of the reference's backwards traversal over a history of n updates in history
 * order (is_ins[u] != 0 for IMU process steps; every other update counts as a measurement, as the reset at the front
 * of the reference's history does).  It reproduces the traversal statement by statement, including the extra
 * decrement after trailing measurements (mav_state_est.cpp:130).  Outputs: the two slots the recursion starts from,
 * the smoothing steps in execution (backward-in-time) order (capacity n), and alias[u] = the slot that holds update
 * u's posterior after smoothing (the reference copies the smoothed posterior into the measurement updates that follow
 * an IMU step, :163-169; here they alias the IMU step's slot).  Returns the number of steps, or a negative status. */
typedef struct {
  int32_t cur_slot;       /* posterior being smoothed: the last measurement of the time step, or the IMU step's own */
  int32_t cur_pred_slot;  /* the IMU step's posterior of that time step (becomes the next step's prediction) */
  int32_t out_slot;       /* where the smoothed state and covariance are written (the IMU step's slot) */
  int32_t reserved;
} rbis_smooth_step_t;
int64_t rbis_smooth_plan(int64_t n, const uint8_t* is_ins, const int32_t* slot, int32_t* next_pred_slot,
                         int32_t* next_slot, rbis_smooth_step_t* steps, int32_t* alias);
/* Runs the steps on the device, one warp per filter (rbis_smooth.cuh); dt as passed to EKFSmoothBackwardsPass.
 * Slots must hold snapshots; `steps` is a HOST array.  Stream-ordered like every other call. */
int rbis_batch_smooth_backward(rbis_batch_t* h, int32_t next_pred_slot, int32_t next_slot, int64_t n_steps,
                               const rbis_smooth_step_t* steps, double dt);
/* Read a ring slot back: vec [21][N], quat [4][N], cov [441][N], loglik [N]; any may be NULL. */
int rbis_batch_get_snapshot(rbis_batch_t* h, int32_t slot, double* vec, double* quat, double* cov, double* loglik, int mem);

/* ---- IMU conditioning ("next" row 4 of SURVEY.md 8f): the accelerometer notch cascade of the Atlas INS path,
 * InsHandler::doFilter (MSE/sensor_handlers.cpp:155-162) over IIRNotch (estimate_tools/src/estimate_tools/
 * iir_notch.cpp:3-60), for every column of an IMU chunk at once.
 * configure: n_stages filters at notch_freq * 2^i, i = 0.., sample rate fs (the reference: 3 stages, fs = 1000,
 * MSE/sensor_handlers.cpp:29-41), for chunks of `cols` columns (N, or the column count of the IMU column map); resets
 * the carried samples to zero as the IIRNotch constructor does.
 * filter: filters rows 3..5 (accelerometer x,y,z) of imu [rows][6][cols] IN PLACE, continuing from the state the
 * previous call left, so a log can be conditioned chunk by chunk before rbis_batch_run_fused consumes it. */
int rbis_batch_notch_configure(rbis_batch_t* h, double notch_freq, double fs, int n_stages, int64_t cols);
int rbis_batch_notch_filter(rbis_batch_t* h, double* imu, int64_t rows, int mem);

/* ---- ensemble statistics against a truth state (error definition of
 * SE/noise_id/noise_id.cpp:37-38; NEES over velocity+chi+position as roll_forward.cpp:54-57).
 * truth_vec [21] / truth_quat [4] (host) shared by all filters, or per-filter [21][N] / [4][N] (`mem`)
 * when per_filter != 0.  Filters are reduced in chunks of `chunk` filters (power of two, <= 1024)
 * in a fixed tree order; out_chunks (host) receives [n_chunks][RBIS_NUM_STATS]:
 *   [0..20] sum e_i, [21..41] sum e_i^2, [42] sum NEES, [43] sum NEES^2, [44] sum loglik,
 *   [45] count non-finite filters, [46] count filters, [47] count NEES within the 95% chi2(9) bounds,
 *   rest reserved (0).
 * out_per_filter (optional, `mem`): [23][N] = e[21], NEES, loglik per filter.  Synchronous. */
int rbis_batch_stats(rbis_batch_t* h, const double* truth_vec, const double* truth_quat, int per_filter,
                     int chunk, double* out_chunks, int64_t* n_chunks, double* out_per_filter, int mem);
/* Same reduction, enqueued on the handle's stream without waiting: truth is shared ([21], [4], host),
 * out_chunks must be PINNED host memory and is valid once a ticket recorded after this call has been
 * waited for.  Lets a caller read per-chunk results every step without stalling the input copies of
 * the next step. */
int rbis_batch_stats_enqueue(rbis_batch_t* h, const double* truth_vec, const double* truth_quat, int chunk,
                             double* out_chunks, int64_t* n_chunks);
/* The same statistics over SNAPSHOT SLOT `slot` (written by an RBIS_OP_SNAPSHOT of an earlier fused program) instead of the live
 * ensemble, on a side stream: the pass is ordered after the launch that wrote the slot and nothing waits for it -- the fused
 * launches that follow keep overlapping the ones before, which a read of the LIVE state (rbis_batch_stats_enqueue) prevents.
 * A later program that snapshots into the same slot waits for this pass.  out_chunks must be PINNED host memory; it is valid
 * once rbis_batch_wait(*ticket) returns.  This is how a Monte-Carlo driver reads the ensemble error / NEES every step of a long
 * replay (append RBIS_OP_SNAPSHOT to the step's last program, alternate two slots) without draining the device. */
int rbis_batch_stats_snapshot_enqueue(rbis_batch_t* h, int32_t slot, const double* truth_vec, const double* truth_quat, int chunk,
                                      double* out_chunks, int64_t* n_chunks, int32_t* ticket);
/* The same statistics over RECORD ROWS first_row .. first_row + n_rows - 1 of the current record set, one chunk table per row:
 * the table of row r is bit-identical to rbis_batch_stats_snapshot_enqueue over a SNAPSHOT taken where the RECORD op that wrote
 * row r stands, with the same truth and chunk.  One pass over all rows, on the same side stream and with the same ordering as
 * rbis_batch_stats_snapshot_enqueue (after the launches of the last fused call; the fused calls that follow do not wait for it).
 * The record set must be in device memory, have every field 0..25 (vec, quat, loglik) and the covariance blocks 1, 2 and 3
 * (v, chi, p: the NEES block), and the rows must lie in [0, rows); otherwise the call fails before anything is enqueued.
 *   truth_vec [n_rows][21] / truth_quat [n_rows][4]: host; row r is the truth at record row first_row + r.
 *   out_chunks: PINNED host [n_rows][n_chunks][RBIS_NUM_STATS].  out_totals: PINNED host [n_rows][RBIS_NUM_STATS] or NULL, each
 *   row's table summed in ascending chunk order (= rbis_stats_reduce_chunks).  Both are valid once rbis_batch_wait(*ticket)
 *   returns.
 * A later fused call whose RECORD ops write into the buffer a pending pass reads waits for that pass on the device.  To keep
 * calls overlapping, alternate two record buffers with rbis_batch_set_record (which does not synchronise), as a driver
 * alternates two snapshot slots. */
int rbis_batch_stats_records_enqueue(rbis_batch_t* h, int64_t first_row, int64_t n_rows, const double* truth_vec,
                                     const double* truth_quat, int chunk, double* out_chunks, double* out_totals, int64_t* n_chunks,
                                     int32_t* ticket);
/* Ensemble statistics of INNOVATION ROWS first_row .. first_row + n_rows - 1 of stream slot `stream`'s innovation set, which must
 * include RBIS_INNOV_NIS; one chunk table per row, with the side stream, outputs, ticket and ordering of
 * rbis_batch_stats_records_enqueue (a later fused call whose MEAS ops write into the buffer a pending pass reads waits for it on
 * the device; alternate two innovation buffers to keep calls overlapping).  Table entries (all others zero):
 *   [0] sum NIS   [1] sum NIS^2   [2] filters with a finite NIS   [3] of them, NIS inside the central 95 % of chi2(m)
 *   [4] filters with a non-finite NIS (skipped rows, poisoned filters)   [5] filters
 *   [6 + a] sum y_a, [15 + a] sum y_a^2 (with RBIS_INNOV_Y)   [24 + a] sum y_a^2 / S(a,a) (with RBIS_INNOV_Y and RBIS_INNOV_S_DIAG)
 * Only filters with a finite NIS enter [0], [1], [3] and [6..32].  Each chunk is reduced with the fixed binary tree of the other
 * statistics, so tables of chunk-aligned shards concatenate and reduce with rbis_stats_reduce_chunks.  ANIS = [0] / [2]; for a
 * consistent filter ANIS is near m and [15 + a] / [2] near the mean S(a,a), i.e. [24 + a] / [2] near 1 for every axis a. */
int rbis_batch_stats_innovations_enqueue(rbis_batch_t* h, int32_t stream, int64_t first_row, int64_t n_rows, int chunk,
                                         double* out_chunks, double* out_totals, int64_t* n_chunks, int32_t* ticket);
/* ---- statistics of a SHARDED ensemble (SURVEY.md 8e): one process per GPU, each handle holds the contiguous filter range
 * [first_chunk * chunk, first_chunk * chunk + N) of an ensemble of total_chunks chunks.  The shard's chunk partials are written
 * into its rows of a zero-initialised DEVICE table [total_chunks][RBIS_NUM_STATS], the table is summed over the ranks with
 * ncclAllReduce on the handle's stream (exact: every row has one non-zero contributor), and reduced on the device in
 * ascending chunk order -- no host round trip before the collective.  The totals (and the table) are therefore bit-identical
 * on every rank and for every GPU count, and equal to rbis_batch_stats + rbis_stats_reduce_chunks on one GPU.
 *   nccl_comm: the caller's ncclComm_t (as void*), one rank per handle, created on the handle's device; NULL = single
 *              process (no collective; first_chunk = 0, total_chunks = the shard's own count).  The library resolves
 *              ncclAllReduce from the NCCL already loaded in the calling process and has no link-time NCCL dependency.
 *   truth_vec [21] / truth_quat [4]: host, shared by all filters.  out_totals: host [RBIS_NUM_STATS].
 *   out_table: host [total_chunks][RBIS_NUM_STATS] or NULL.  Synchronous (collective: every rank of the communicator calls it). */
int rbis_batch_stats_allreduce(rbis_batch_t* h, void* nccl_comm, const double* truth_vec, const double* truth_quat, int chunk,
                               int64_t first_chunk, int64_t total_chunks, double* out_totals, double* out_table);

/* ---- windowed noise-identification likelihood: the per-window term of sampleProcessForward + negLogLikelihood
 * (state-estimator/src/noise_id/noise_id.cpp:36-40,44-65; SURVEY.md 8f row 2) for every filter at once.  With the
 * filters' heads = states rolled forward over one window from the truth, truth_vec [21][N] / truth_quat [4][N] = the
 * truth at the window ends, and base_cov [441][base_cols] = the covariance the same window accumulates under ZERO
 * process noise (column base_map[n] for filter n; base_map HOST int32[N], NULL = column n):
 *   e = head (-) truth (subtractState + quatToChi),  C = cov - base_cov[:, base_map[n]],
 *   out[n] = -loglike_normalized(e_A, 0, C_AA) = log det C_AA + e_A^T C_AA^-1 e_A     (A = active_idx, host int32[n_active])
 * Summing out over the windows of one parameter point gives negLogLikelihood.  truth, base_cov, out live as `mem`
 * says.  Synchronous. */
int rbis_batch_window_neg_loglik(rbis_batch_t* h, const double* truth_vec, const double* truth_quat, const double* base_cov,
                                 const int32_t* base_map, int64_t base_cols, int n_active, const int32_t* active_idx,
                                 double* out, int mem);

/* ---- wire structs and IMU decode (SURVEY.md 8f row 4) -- host side.  Struct-level layouts of the reference's LCM types;
 * the LCM byte encoding (big-endian marshalling + fingerprint) is not produced here (no LCM, no lcm-gen, no log to check
 * an encoder against).
 * filter_state_t (pronto-lcmtypes/lcmtypes/pronto_filter_state_t.lcm) as rbisCreateFilterStateMessage writes it
 * (MSE/rbis.cpp:268-285: quat (w,x,y,z), state = vec, cov = Map<RBIM> i.e. COLUMN-major although the .lcm comment says row
 * major) and RBIS(const pronto_filter_state_t*) reads it (MSE/rbis.hpp:58-67). */
typedef struct {
  int64_t utime;
  double quat[4];
  int32_t num_states;        /* 21 */
  int32_t reserved0;
  double state[RBIS_NUM_STATES];
  int32_t num_cov_elements;  /* 441 */
  int32_t reserved1;
  double cov[RBIS_COV_ELEMS];
} rbis_filter_state_t;
/* One message per filter first..first+count-1 (synchronous; reads the whole ensemble: a logging path). */
int rbis_batch_get_filter_states(rbis_batch_t* h, int64_t first, int64_t count, rbis_filter_state_t* out);
/* Filters first..first+count-1 := the messages (state, quaternion, covariance; log-likelihood 0), as RBIS(msg) +
 * Map<const RBIM>(msg->cov) of the reference's log loader (state-estimator/src/noise_id/noise_id.cpp:83-86). */
int rbis_batch_set_filter_states(rbis_batch_t* h, int64_t first, int64_t count, const rbis_filter_state_t* msgs);
/* One filter_state_t message per filter first..first+count-1 of a record row that is already on the
 * host: row is [k][n_filters] in the layout above, with every field 0..24 and all seven covariance blocks (fields bit 25 and
 * bits 26.. may be set too).  The messages are what rbis_batch_get_filter_states writes for the same state: both triangles of the
 * covariance, column-major (MSE/rbis.cpp:282), utime = `utime`.  Host only; it hides the packed layout from a caller that
 * publishes the reference's message per recorded head (MSE/lcm_front_end.cpp:144-166). */
int rbis_record_filter_states(uint64_t fields, int32_t cov_blocks, const double* row, int64_t n_filters, int64_t utime,
                              int64_t first, int64_t count, rbis_filter_state_t* out);

/* indexed_measurement_t (pronto-lcmtypes/lcmtypes/pronto_indexed_measurement_t.lcm), bounded to RBIS_MAX_MEAS rows. */
typedef struct {
  int64_t utime, state_utime;
  int32_t measured_dim;
  int32_t measured_cov_dim;                      /* measured_dim^2 */
  double z_effective[RBIS_MAX_MEAS];
  int32_t z_indices[RBIS_MAX_MEAS];
  int32_t reserved;
  double R_effective[RBIS_MAX_MEAS * RBIS_MAX_MEAS];
} rbis_indexed_measurement_t;
/* IndexedMeasurementHandler::processMessage (MSE/sensor_handlers.cpp:576-582): the constant part of a stream (index set,
 * R = Map<MatrixXd>(R_effective, m, m), column-major, copied to R_out[m*m]; sensor_id = indexed_sensor).  z rows are the
 * messages' z_effective; out->z / rows stay for the caller to fill. */
int rbis_stream_from_indexed_measurement(const rbis_indexed_measurement_t* msg, rbis_stream_t* out, double* R_out);
/* The same for a sequence of `count` messages that become rows 0..count-1 of ONE stream: all must have message 0's measured_dim,
 * measured_cov_dim and index set (else RBIS_ERR_INVALID).  R_out [count][m][m] receives every message's R_effective; r_mode is
 * RBIS_R_SHARED_FULL when all of them are bit-identical (R_out's first matrix is then the stream's R), else RBIS_R_PER_ROW_FULL.
 * out->rows = count; out->z stays for the caller to fill. */
int rbis_stream_from_indexed_measurements(const rbis_indexed_measurement_t* msgs, int64_t count, rbis_stream_t* out, double* R_out);

/* KVH raw IMU batches of the Atlas INS path.  rbis_kvh_packet_t = bot_core::kvh_raw_imu_t; a batch message carries
 * num_packets of them, NEWEST FIRST, most of which were already seen in earlier batches.
 * rbis_kvh_decode_batch = IMUStream::convertFromLCMBatch (estimate_tools/src/estimate_tools/imu_stream.cpp:62-97): the
 * packets newer than the last one seen come back in out_new, oldest first, with utime_delta = time since the previous new
 * packet; the others in out_old (optional) with the reference's obfuscated delta; a packet counter that runs backwards
 * resets the stream.  Both output arrays need room for num_packets entries. */
typedef struct {
  int64_t utime;
  int64_t packet_count;
  double delta_rotation[3];
  double linear_acceleration[3];
} rbis_kvh_packet_t;
typedef struct {
  int64_t utime_raw, utime_batch, utime, utime_delta, packet_count;
  double delta_rotation[3];
  double linear_acceleration[3];
} rbis_imu_packet_t;
typedef struct rbis_kvh_stream rbis_kvh_stream_t;
int rbis_kvh_stream_create(rbis_kvh_stream_t** out);
int rbis_kvh_stream_destroy(rbis_kvh_stream_t* s);
int rbis_kvh_decode_batch(rbis_kvh_stream_t* s, int64_t batch_utime, int32_t num_packets, const rbis_kvh_packet_t* raw,
                          rbis_imu_packet_t* out_new, int32_t* n_new, rbis_imu_packet_t* out_old, int32_t* n_old);
/* InsHandler::processMessageAtlas after the decode (MSE/sensor_handlers.cpp:186-251): the newest new packet of a batch
 * (after the notch cascade, rbis_batch_notch_filter, when the Atlas filter is on) -> gyro = R (delta_rotation / raw_dt),
 * accel = T linear_acceleration (rotation and translation, as the reference applies bot_trans_apply_vec), and the
 * integration dt = default_dt for the first message, else the batch utime difference.  *prev_utime: 0 before the first. */
int rbis_kvh_imu_step(const rbis_imu_packet_t* newest, int64_t batch_utime, const double ins_to_body_quat[4],
                      const double ins_to_body_trans[3], double default_dt, int64_t* prev_utime, double gyro[3], double accel[3],
                      double* dt);

/* Stream-ordered completion tickets: record marks "everything enqueued so far", wait blocks the host
 * until that point has completed.  Up to 8 tickets may be outstanding. */
int rbis_batch_record(rbis_batch_t* h, int32_t* ticket);
int rbis_batch_wait(rbis_batch_t* h, int32_t ticket);
/* Fixed-order final reduction of chunk partials (ascending chunk index): out[RBIS_NUM_STATS]. */
int rbis_stats_reduce_chunks(const double* chunks, int64_t n_chunks, double* out);

/* ---- FP64 roofline denominators measured on the handle's device: register-resident independent
 * DFMA chains, and mma.sync.m8n8k4.f64 (DMMA) for comparison.  TFLOP/s.  Synchronous. */
int rbis_measure_fp64_peak(int device, int iters, double* dfma_tflops, double* dmma_tflops);

#ifdef __cplusplus
}
#endif
#endif /* RBIS_BATCH_H_ */
