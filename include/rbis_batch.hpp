// rbis_batch.hpp -- header-only C++ mirror of the reference's operator interface over the C ABI of
// rbis_batch.h.  Same class names, constructor argument order and member names as
//   MavStateEst::RBIS / RBIM                         MSE/rbis.hpp:19-123
//   MavStateEst::RBISUpdateInterface + 4 subclasses  MSE/rbis_update_interface.hpp:8-120
//   MavStateEst::MavStateEstimator                   MSE/mav_state_est.hpp:10-27
// (MSE = /root/reference/state-estimator/src/mav_state_est), with two differences that the batch
// setting forces: (1) an update object carries its data for ALL N filters of an ensemble
// (structure of arrays, filter index fastest) and updateFilter() advances the whole ensemble on the
// GPU in place -- the posterior lives in the ensemble, not in the update object; (2) Eigen types are
// replaced by plain arrays (Eigen is not a dependency of this library).  All arithmetic runs in
// librbis_b200.so (CUDA, sm_100a); nothing here computes filter math on the host.
#ifndef RBIS_BATCH_HPP_
#define RBIS_BATCH_HPP_

#include <algorithm>
#include <array>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "rbis_batch.h"

namespace MavStateEst {
namespace batch {

struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& what) : std::runtime_error(what), code(c) {}
};
inline void check(int rc) {
  if (rc < 0) throw Error(rc, rbis_last_error());
}

// One filter's state: MavStateEst::RBIS without Eigen (MSE/rbis.hpp:19-121; index enum of
// eigen_utils::RigidBodyState as pinned in SURVEY.md 8.0).
struct RBIS {
  enum {
    angular_velocity_ind = 0, velocity_ind = 3, chi_ind = 6, position_ind = 9, acceleration_ind = 12, basic_num_states = 15,
    gyro_bias_ind = 15, accel_bias_ind = 18, rbis_num_states = 21
  };
  std::array<double, rbis_num_states> vec{};
  std::array<double, 4> quat{{1.0, 0.0, 0.0, 0.0}};  // w, x, y, z
  int64_t utime = 0;
  double* angularVelocity() { return &vec[angular_velocity_ind]; }
  double* velocity() { return &vec[velocity_ind]; }
  double* chi() { return &vec[chi_ind]; }
  double* position() { return &vec[position_ind]; }
  double* acceleration() { return &vec[acceleration_ind]; }
  double* gyroBias() { return &vec[gyro_bias_ind]; }
  double* accelBias() { return &vec[accel_bias_ind]; }
  const double* velocity() const { return &vec[velocity_ind]; }
  const double* position() const { return &vec[position_ind]; }
  const double* gyroBias() const { return &vec[gyro_bias_ind]; }
  const double* accelBias() const { return &vec[accel_bias_ind]; }
};
typedef std::array<double, RBIS::rbis_num_states * RBIS::rbis_num_states> RBIM;  // column-major, (r,c) at r + 21 c

// An ensemble of N filters resident on one GPU (owns an rbis_batch_t).
class RBISEnsemble {
 public:
  explicit RBISEnsemble(int64_t n_filters, const rbis_batch_config_t* cfg = nullptr) { check(rbis_batch_create(&h_, n_filters, cfg)); }
  ~RBISEnsemble() { rbis_batch_destroy(h_); }
  RBISEnsemble(const RBISEnsemble&) = delete;
  RBISEnsemble& operator=(const RBISEnsemble&) = delete;

  int64_t size() const { return rbis_batch_num_filters(h_); }
  rbis_batch_t* handle() { return h_; }
  void synchronize() { check(rbis_batch_synchronize(h_)); }
  // vec [21][N], quat [4][N], cov [441][N] (may be null), loglik [N] (null = zeros)
  void setState(const double* vec, const double* quat, const double* cov, const double* loglik, int64_t utime, int mem = RBIS_MEM_HOST) {
    check(rbis_batch_set_state(h_, vec, quat, cov, loglik, utime, mem));
  }
  void getState(double* vec, double* quat, double* cov, double* loglik, int64_t* utime, int mem = RBIS_MEM_HOST) {
    check(rbis_batch_get_state(h_, vec, quat, cov, loglik, utime, mem));
  }
  void setFilter(int64_t i, const RBIS& s, const RBIM& cov, double loglik = 0.0) {
    check(rbis_batch_set_filter(h_, i, s.vec.data(), s.quat.data(), cov.data(), loglik));
  }
  void getFilter(int64_t i, RBIS& s, RBIM& cov, double* loglik = nullptr) {
    check(rbis_batch_get_filter(h_, i, s.vec.data(), s.quat.data(), cov.data(), loglik));
    check(rbis_batch_get_state(h_, nullptr, nullptr, nullptr, nullptr, &s.utime, RBIS_MEM_DEVICE));
  }
  // process noise of the next IMU steps (cached: repeated identical values cost nothing)
  void setProcessNoise(double q_gyro, double q_accel, double q_gyro_bias, double q_accel_bias) {
    const std::array<double, 4> q{{q_gyro, q_accel, q_gyro_bias, q_accel_bias}};
    if (have_q_ && q == q_) return;
    check(rbis_batch_set_process_noise(h_, q_gyro, q_accel, q_gyro_bias, q_accel_bias));
    q_ = q;
    have_q_ = true;
  }
  void setProcessNoisePerFilter(const double* q_gyro, const double* q_accel, const double* q_gyro_bias, const double* q_accel_bias,
                                int mem = RBIS_MEM_HOST) {
    check(rbis_batch_set_process_noise_per_filter(h_, q_gyro, q_accel, q_gyro_bias, q_accel_bias, mem));
    have_q_ = false;
  }

 private:
  rbis_batch_t* h_ = nullptr;
  std::array<double, 4> q_{};
  bool have_q_ = false;
};

class MavStateEstimator;

// MSE/rbis_update_interface.hpp:8-42
class RBISUpdateInterface {
 public:
  typedef enum {
    ins, gps, vicon, laser, laser_gpf, scan_matcher, optical_flow, reset, invalid, rgbd, fovis, legodo, pose_meas, altimeter,
    airspeed, sideslip, init_message, viewer, yawlock
  } sensor_enum;

  int64_t utime;
  sensor_enum sensor_id;

  RBISUpdateInterface(sensor_enum sensor_id_, int64_t utime_) : utime(utime_), sensor_id(sensor_id_) {}
  virtual ~RBISUpdateInterface() {}

  // Applies the update to every filter: prior = the ensemble's head, posterior written in place;
  // the ensemble's log-likelihoods follow MSE/rbis_update_interface.cpp:25-27,42,87,106.
  virtual void updateFilter(RBISEnsemble& filters) = 0;

 protected:
  friend class MavStateEstimator;
  virtual int opKind() const { return -1; }
};

// MSE/rbis_update_interface.hpp:44-58.  reset_state [21][N] + [4][N], reset_cov [441][N]; the
// single-filter form broadcasts one state to the whole ensemble.
class RBISResetUpdate : public RBISUpdateInterface {
 public:
  std::vector<double> reset_vec, reset_quat, reset_cov;
  RBISResetUpdate(std::vector<double> vec, std::vector<double> quat, std::vector<double> cov, sensor_enum sensor_id_, int64_t utime_)
      : RBISUpdateInterface(sensor_id_, utime_), reset_vec(std::move(vec)), reset_quat(std::move(quat)), reset_cov(std::move(cov)) {}
  RBISResetUpdate(const RBIS& state, const RBIM& cov, int64_t n_filters, sensor_enum sensor_id_, int64_t utime_)
      : RBISUpdateInterface(sensor_id_, utime_), reset_vec(21 * n_filters), reset_quat(4 * n_filters), reset_cov(441 * n_filters) {
    for (int64_t n = 0; n < n_filters; n++) {
      for (int i = 0; i < 21; i++) reset_vec[i * n_filters + n] = state.vec[i];
      for (int i = 0; i < 4; i++) reset_quat[i * n_filters + n] = state.quat[i];
      for (int i = 0; i < 441; i++) reset_cov[i * n_filters + n] = cov[i];
    }
  }
  void updateFilter(RBISEnsemble& f) override { f.setState(reset_vec.data(), reset_quat.data(), reset_cov.data(), nullptr, utime); }
};

// MSE/rbis_update_interface.hpp:60-82.  gyro, accelerometer: [3][N].
class RBISIMUProcessStep : public RBISUpdateInterface {
 public:
  std::vector<double> gyro, accelerometer;
  double dt, q_gyro, q_accel, q_gyro_bias, q_accel_bias;
  RBISIMUProcessStep(std::vector<double> gyro_, std::vector<double> accelerometer_, double q_gyro_, double q_accel_,
                     double q_gyro_bias_, double q_accel_bias_, double dt_, int64_t utime_)
      : RBISUpdateInterface(ins, utime_), gyro(std::move(gyro_)), accelerometer(std::move(accelerometer_)), dt(dt_), q_gyro(q_gyro_),
        q_accel(q_accel_), q_gyro_bias(q_gyro_bias_), q_accel_bias(q_accel_bias_) {}
  void updateFilter(RBISEnsemble& f) override {
    f.setProcessNoise(q_gyro, q_accel, q_gyro_bias, q_accel_bias);
    check(rbis_batch_ins_step(f.handle(), gyro.data(), accelerometer.data(), dt, utime, RBIS_MEM_HOST));
  }

 protected:
  int opKind() const override { return RBIS_OP_IMU; }
};

// MSE/rbis_update_interface.hpp:84-102.  measurement [m][N]; measurement_cov m x m column-major, shared.
class RBISIndexedMeasurement : public RBISUpdateInterface {
 public:
  std::vector<int32_t> index;
  std::vector<double> measurement, measurement_cov;
  RBISIndexedMeasurement(std::vector<int32_t> index_, std::vector<double> measurement_, std::vector<double> measurement_cov_,
                         sensor_enum sensor_id_, int64_t utime_)
      : RBISUpdateInterface(sensor_id_, utime_), index(std::move(index_)), measurement(std::move(measurement_)),
        measurement_cov(std::move(measurement_cov_)) {}
  void updateFilter(RBISEnsemble& f) override {
    check(rbis_batch_indexed_update(f.handle(), (int)index.size(), index.data(), measurement.data(), measurement_cov.data(),
                                    RBIS_R_SHARED_FULL, utime, RBIS_MEM_HOST));
  }
  virtual const std::vector<double>* orientationRows() const { return nullptr; }

 protected:
  int opKind() const override { return RBIS_OP_MEAS; }
};

// MSE/rbis_update_interface.hpp:104-120.  orientation [4][N] (w,x,y,z).
class RBISIndexedPlusOrientationMeasurement : public RBISIndexedMeasurement {
 public:
  std::vector<double> orientation;
  RBISIndexedPlusOrientationMeasurement(std::vector<int32_t> index_, std::vector<double> measurement_,
                                        std::vector<double> measurement_cov_, std::vector<double> orientation_,
                                        sensor_enum sensor_id_, int64_t utime_)
      : RBISIndexedMeasurement(std::move(index_), std::move(measurement_), std::move(measurement_cov_), sensor_id_, utime_),
        orientation(std::move(orientation_)) {}
  void updateFilter(RBISEnsemble& f) override {
    check(rbis_batch_indexed_orient_update(f.handle(), (int)index.size(), index.data(), measurement.data(), orientation.data(),
                                           measurement_cov.data(), RBIS_R_SHARED_FULL, utime, RBIS_MEM_HOST));
  }
  const std::vector<double>* orientationRows() const override { return &orientation; }
};

// MSE/mav_state_est.hpp:10-27 + MSE/mav_state_est.cpp:12-96 for an ensemble whose filters share one
// arrival schedule.  addUpdate takes ownership of the update (as updateHistory does,
// MSE/update_history.cpp:9-14); out-of-order updates rewind to a device snapshot and replay
// (rbis_planner_*), too-old updates are dropped.  Every roll-forward is ONE fused kernel launch.
class MavStateEstimator {
 public:
  int64_t utime_history_span;

  // snapshot_period_us = 0 (default): chosen so that the snapshot ring covers the whole history span (slots x period >=
  // utime_history_span, whole milliseconds), i.e. every update the reference would still replay (update_history.cpp:28-39) can be
  // rewound to; an explicit, shorter period trades a shorter rewind window for shorter replays (rbis_planner_create).
  MavStateEstimator(int64_t n_filters, RBISResetUpdate* init_state, int64_t utime_history_span_us, int32_t snapshot_slots = 4,
                    int64_t snapshot_period_us = 0, const rbis_batch_config_t* cfg = nullptr)
      : utime_history_span(utime_history_span_us), filters_(make_ensemble(n_filters, snapshot_slots, cfg)) {
    std::unique_ptr<RBISResetUpdate> init(init_state);
    init->updateFilter(*filters_);  // MSE/mav_state_est.cpp:16
    if (snapshot_period_us <= 0 && snapshot_slots > 0) {
      const int64_t per = (utime_history_span_us + snapshot_slots - 1) / snapshot_slots;
      snapshot_period_us = std::max<int64_t>(1000, (per + 999) / 1000 * 1000);
    }
    check(rbis_planner_create(&planner_, init->utime, snapshot_slots, snapshot_period_us, init->utime, utime_history_span_us));
  }
  ~MavStateEstimator() { rbis_planner_destroy(planner_); }
  MavStateEstimator(const MavStateEstimator&) = delete;
  MavStateEstimator& operator=(const MavStateEstimator&) = delete;

  RBISEnsemble& filters() { return *filters_; }

  // Returns false when the update was discarded as too old (the reference prints and drops it).
  bool addUpdate(RBISUpdateInterface* update, bool roll_forward) {
    std::unique_ptr<RBISUpdateInterface> own(update);
    const int kind = update->opKind();
    if (kind < 0) throw Error(RBIS_ERR_INVALID, "addUpdate: only IMU and measurement updates enter the history");
    rbis_op_t op;
    std::memset(&op, 0, sizeof(op));
    op.kind = kind;
    op.row = next_id_;
    op.utime = update->utime;
    if (kind == RBIS_OP_IMU) op.dt = static_cast<RBISIMUProcessStep*>(update)->dt;
    const int rc = rbis_planner_add_update(planner_, &op, roll_forward ? 1 : 0);
    check(rc);
    if (rc == 1) return false;
    if (update->utime > newest_) newest_ = update->utime;
    updates_[next_id_++] = std::move(own);
    if (roll_forward) execute_pending();
    return true;
  }
  void getHeadState(int64_t filter, RBIS& head_state, RBIM& head_cov) { filters_->getFilter(filter, head_state, head_cov); }
  double getMeasurementsLogLikelihood(int64_t filter) {
    RBIS s; RBIM c; double ll = 0;
    filters_->getFilter(filter, s, c, &ll);
    return ll;
  }
  int64_t launches() const { return launches_; }

 private:
  static std::unique_ptr<RBISEnsemble> make_ensemble(int64_t n, int32_t slots, const rbis_batch_config_t* cfg) {
    rbis_batch_config_t c;
    if (cfg) c = *cfg; else rbis_default_config(&c);
    c.snapshot_slots = slots;
    return std::unique_ptr<RBISEnsemble>(new RBISEnsemble(n, &c));
  }
  struct StreamBuild {
    const RBISIndexedMeasurement* proto;
    std::vector<double> z, quat;
    std::vector<double> R;  // [rows][m][m]: every row's measurement_cov
    bool same_R = true;     // all rows carry proto's measurement_cov
    int64_t rows = 0;
  };
  // Updates share a stream when they share the index set, the orientation flag and the off-diagonal zero pattern of R: each row then
  // runs the chunk plan and decorrelation of its own R (rbis_r_mode_t), whatever the values -- a new R does not cost a flush.
  static bool same_stream(const RBISIndexedMeasurement* a, const RBISIndexedMeasurement* b) {
    if (a->index != b->index || (a->orientationRows() != nullptr) != (b->orientationRows() != nullptr)) return false;
    if (a->measurement_cov.size() != b->measurement_cov.size()) return false;
    const size_t m = a->index.size();
    for (size_t i = 0; i < m; i++)
      for (size_t j = 0; j < m; j++)
        if (i != j && (a->measurement_cov[i + m * j] != 0.0) != (b->measurement_cov[i + m * j] != 0.0)) return false;
    return true;
  }
  void flush(std::vector<rbis_op_t>& ops, std::vector<double>& imu, int64_t& imu_rows, std::vector<StreamBuild>& sb) {
    if (ops.empty()) return;
    std::vector<rbis_stream_t> st(sb.size());
    for (size_t s = 0; s < sb.size(); s++) {
      std::memset(&st[s], 0, sizeof(rbis_stream_t));
      const RBISIndexedMeasurement* m = sb[s].proto;
      st[s].m = (int32_t)m->index.size();
      st[s].has_orientation = m->orientationRows() ? 1 : 0;
      st[s].r_mode = sb[s].same_R ? RBIS_R_SHARED_FULL : RBIS_R_PER_ROW_FULL;
      st[s].sensor_id = (int32_t)m->sensor_id;
      for (size_t a = 0; a < m->index.size(); a++) st[s].idx[a] = m->index[a];
      st[s].z = sb[s].z.data();
      st[s].quat = st[s].has_orientation ? sb[s].quat.data() : nullptr;
      st[s].R = sb[s].same_R ? m->measurement_cov.data() : sb[s].R.data();
      st[s].rows = sb[s].rows;
    }
    check(rbis_batch_run_fused(filters_->handle(), (int64_t)ops.size(), ops.data(), imu_rows ? imu.data() : nullptr, imu_rows,
                               (int)st.size(), st.data(), RBIS_MEM_HOST));
    filters_->synchronize();  // the staging arrays die with this scope
    launches_++;
    ops.clear(); imu.clear(); imu_rows = 0; sb.clear();
  }
  void execute_pending() {
    const int64_t n = rbis_planner_pending(planner_);
    if (n == 0) return;
    std::vector<rbis_op_t> prog((size_t)n);
    int64_t got = 0;
    check(rbis_planner_take(planner_, prog.data(), n, &got));
    const int64_t N = filters_->size();
    std::vector<rbis_op_t> ops;
    std::vector<double> imu;
    int64_t imu_rows = 0;
    std::vector<StreamBuild> sb;
    for (int64_t i = 0; i < got; i++) {
      rbis_op_t op = prog[(size_t)i];
      if (op.kind == RBIS_OP_IMU) {
        auto* u = static_cast<RBISIMUProcessStep*>(updates_.at(op.row).get());
        const std::array<double, 4> q{{u->q_gyro, u->q_accel, u->q_gyro_bias, u->q_accel_bias}};
        if (have_cur_q_ && !ops.empty() && q != cur_q_) flush(ops, imu, imu_rows, sb);  // process noise is per launch
        cur_q_ = q;
        have_cur_q_ = true;
        filters_->setProcessNoise(q[0], q[1], q[2], q[3]);
        imu.insert(imu.end(), u->gyro.begin(), u->gyro.end());
        imu.insert(imu.end(), u->accelerometer.begin(), u->accelerometer.end());
        op.row = imu_rows++;
      } else if (op.kind == RBIS_OP_MEAS) {
        auto* u = static_cast<RBISIndexedMeasurement*>(updates_.at(op.row).get());
        size_t s = 0;
        for (; s < sb.size(); s++)
          if (same_stream(sb[s].proto, u)) break;
        if (s == sb.size()) {
          if (sb.size() == RBIS_MAX_STREAMS) { flush(ops, imu, imu_rows, sb); s = 0; }
          sb.push_back(StreamBuild{u, {}, {}, {}, true, 0});
        }
        sb[s].same_R = sb[s].same_R && u->measurement_cov == sb[s].proto->measurement_cov;
        sb[s].R.insert(sb[s].R.end(), u->measurement_cov.begin(), u->measurement_cov.end());
        sb[s].z.insert(sb[s].z.end(), u->measurement.begin(), u->measurement.begin() + (long)(u->index.size() * (size_t)N));
        if (const std::vector<double>* q = u->orientationRows()) sb[s].quat.insert(sb[s].quat.end(), q->begin(), q->end());
        op.stream = (int32_t)s;
        op.row = sb[s].rows++;
      }
      ops.push_back(op);
    }
    flush(ops, imu, imu_rows, sb);
    // updates at or before (newest - span) can never be replayed again (MSE/mav_state_est.cpp:74-77)
    if (utime_history_span > 0) {
      const int64_t cutoff = newest_ - utime_history_span;
      for (auto it = updates_.begin(); it != updates_.end();)
        if (it->second->utime <= cutoff) it = updates_.erase(it); else ++it;
    }
  }

  std::unique_ptr<RBISEnsemble> filters_;
  rbis_planner_t* planner_ = nullptr;
  std::map<int64_t, std::unique_ptr<RBISUpdateInterface>> updates_;
  int64_t next_id_ = 0, newest_ = INT64_MIN, launches_ = 0;
  std::array<double, 4> cur_q_{};
  bool have_cur_q_ = false;
};

// ------------------------------------------------------------------------------------------------
// Leg-odometry measurement formation for an ensemble: MavStateEst::LegOdoCommon
// (motion_estimate/src/mav_est_legodo/rbis_legodo_common.{hpp,cpp}; SURVEY.md 8f row 3), the step
// immediately before RBISIndexedMeasurement.  Pure input shaping (no filter math): delta pose ->
// body velocity, index set and R by mode, "uncertain" R while a foot breaks contact.  Per-filter
// arrays are [k][N]; the status flags are shared by the ensemble (one robot, N replicas).
// ------------------------------------------------------------------------------------------------
class LegOdoCommon {
 public:
  typedef enum { MODE_LIN_RATE, MODE_ROT_RATE, MODE_LIN_AND_ROT_RATE, MODE_POSITION_AND_LIN_RATE } LegOdoCommonMode;  // rbis_legodo_common.hpp:15-17
  LegOdoCommonMode mode_;
  double R_legodo_xyz_, R_legodo_vxyz_, R_legodo_vang_, R_legodo_vxyz_uncertain_, R_legodo_vang_uncertain_;

  // the config keys state_estimator.legodo.{mode,r_xyz,r_vxyz,r_vang,r_vxyz_uncertain,r_vang_uncertain} (rbis_legodo_common.cpp:9-33)
  LegOdoCommon(LegOdoCommonMode mode, double r_xyz, double r_vxyz, double r_vang, double r_vxyz_uncertain, double r_vang_uncertain)
      : mode_(mode), R_legodo_xyz_(r_xyz), R_legodo_vxyz_(r_vxyz), R_legodo_vang_(r_vang), R_legodo_vxyz_uncertain_(r_vxyz_uncertain),
        R_legodo_vang_uncertain_(r_vang_uncertain) {}

  // rbis_legodo_common.cpp:35-88.  cov_legodo: m x m column-major (diagonal).
  void getCovariance(LegOdoCommonMode mode_current, bool delta_certain, std::vector<double>& cov_legodo, std::vector<int32_t>& z_indices) const {
    const double vxyz = delta_certain ? R_legodo_vxyz_ : R_legodo_vxyz_uncertain_;
    const double vang = delta_certain ? R_legodo_vang_ : R_legodo_vang_uncertain_;
    std::vector<double> R;
    auto sq = [](double v) { return v * v; };
    if (mode_current == MODE_LIN_AND_ROT_RATE) {
      R = {sq(vxyz), sq(vxyz), sq(vxyz), sq(vang), sq(vang), sq(vang)};
      z_indices = {RBIS::velocity_ind, RBIS::velocity_ind + 1, RBIS::velocity_ind + 2, RBIS::angular_velocity_ind,
                   RBIS::angular_velocity_ind + 1, RBIS::angular_velocity_ind + 2};
    } else if (mode_current == MODE_LIN_RATE) {
      R = {sq(vxyz), sq(vxyz), sq(vxyz)};
      z_indices = {RBIS::velocity_ind, RBIS::velocity_ind + 1, RBIS::velocity_ind + 2};
    } else if (mode_current == MODE_POSITION_AND_LIN_RATE) {
      R = {sq(R_legodo_xyz_), sq(R_legodo_xyz_), sq(R_legodo_xyz_), sq(vxyz), sq(vxyz), sq(vxyz)};
      z_indices = {RBIS::position_ind, RBIS::position_ind + 1, RBIS::position_ind + 2, RBIS::velocity_ind, RBIS::velocity_ind + 1,
                   RBIS::velocity_ind + 2};
    } else {
      throw Error(RBIS_ERR_INVALID, "LegOdoCommon: mode not supported");  // the reference leaves the vectors unsized here
    }
    const size_t m = R.size();
    cov_legodo.assign(m * m, 0.0);
    for (size_t a = 0; a < m; a++) cov_legodo[a + m * a] = R[a];
  }

  // libbot bot_quat_to_roll_pitch_yaw (q = w,x,y,z)
  static void quatToRollPitchYaw(const double q[4], double rpy[3]) {
    rpy[0] = std::atan2(2 * (q[0] * q[1] + q[2] * q[3]), 1 - 2 * (q[1] * q[1] + q[2] * q[2]));
    rpy[1] = std::asin(2 * (q[0] * q[2] - q[3] * q[1]));
    rpy[2] = std::atan2(2 * (q[0] * q[3] + q[1] * q[2]), 1 - 2 * (q[2] * q[2] + q[3] * q[3]));
  }

  // rbis_legodo_common.cpp:110-170.  odo_position_xyz [3][N]: pelvis position; odo_delta_xyz [3][N] and
  // odo_delta_quat [4][N]: pose increment since prev_utime.  The velocity is delta / elapsed time
  // (pronto_conversions_lcm.hpp:38-87 getDeltaAsVelocity); the caller owns the returned update (or hands it to addUpdate).
  RBISUpdateInterface* createMeasurement(const std::vector<double>& odo_position_xyz, const std::vector<double>& odo_delta_xyz,
                                         const std::vector<double>& odo_delta_quat, int64_t n_filters, int64_t utime, int64_t prev_utime,
                                         int odo_position_status, float odo_delta_status) const {
    const size_t N = (size_t)n_filters;
    const double elapsed_time = (double)(utime - prev_utime) * 1E-6;
    LegOdoCommonMode mode_current = mode_;
    if (mode_current == MODE_POSITION_AND_LIN_RATE && !odo_position_status) mode_current = MODE_LIN_RATE;  // :117-121
    const bool delta_certain = odo_delta_status < 0.5f;                                                  // :123-128
    std::vector<double> cov_legodo;
    std::vector<int32_t> z_indices;
    getCovariance(mode_current, delta_certain, cov_legodo, z_indices);
    std::vector<double> vel(3 * N);
    for (size_t k = 0; k < 3 * N; k++) vel[k] = odo_delta_xyz[k] / elapsed_time;
    std::vector<double> z;
    if (mode_current == MODE_LIN_AND_ROT_RATE) {   // :135-153
      z.resize(6 * N);
      std::copy(vel.begin(), vel.end(), z.begin());
      for (size_t n = 0; n < N; n++) {
        const double q[4] = {odo_delta_quat[n], odo_delta_quat[N + n], odo_delta_quat[2 * N + n], odo_delta_quat[3 * N + n]};
        double rpy[3];
        quatToRollPitchYaw(q, rpy);
        for (int k = 0; k < 3; k++) z[(3 + (size_t)k) * N + n] = rpy[k] / elapsed_time;
      }
    } else if (mode_current == MODE_LIN_RATE) {    // :154-157
      z = vel;
    } else {                                       // MODE_POSITION_AND_LIN_RATE, :158-165
      z.resize(6 * N);
      std::copy(odo_position_xyz.begin(), odo_position_xyz.begin() + (long)(3 * N), z.begin());
      std::copy(vel.begin(), vel.end(), z.begin() + (long)(3 * N));
    }
    return new RBISIndexedMeasurement(z_indices, z, cov_legodo, RBISUpdateInterface::legodo, utime);
  }
};

// MavStateEstimator::EKFSmoothBackwardsPass (MSE/mav_state_est.cpp:98-189) for an ensemble whose forward program stored
// the posterior of history entry u (entry 0 = the reset, is_ins[u] for IMU process steps) in snapshot slot slot[u].
// Plans the reference's backwards traversal on the host (rbis_smooth_plan) and runs ekfSmoothingStep
// (MSE/rbis.cpp:234-266) for every filter on the device.  Returns, per history entry, the slot that now holds its
// smoothed posterior (the reference copies the smoothed posterior of an IMU step into the measurement updates that
// follow it; here they alias its slot) -- read with rbis_batch_get_snapshot.
inline std::vector<int32_t> EKFSmoothBackwardsPass(RBISEnsemble& filters, const std::vector<uint8_t>& is_ins,
                                                   const std::vector<int32_t>& slot, double dt) {
  if (is_ins.size() != slot.size() || is_ins.empty()) throw Error(RBIS_ERR_INVALID, "EKFSmoothBackwardsPass: bad history description");
  std::vector<rbis_smooth_step_t> steps(is_ins.size());
  std::vector<int32_t> alias(is_ins.size());
  int32_t next_pred = 0, next = 0;
  const int64_t n_steps = rbis_smooth_plan((int64_t)is_ins.size(), is_ins.data(), slot.data(), &next_pred, &next, steps.data(), alias.data());
  if (n_steps < 0) check((int)n_steps);
  check(rbis_batch_smooth_backward(filters.handle(), next_pred, next, n_steps, steps.data(), dt));
  return alias;
}

}  // namespace batch
}  // namespace MavStateEst

#endif  // RBIS_BATCH_HPP_
