// rbis_wire.cpp -- host-side wire structs of the RBIS path (SURVEY.md 8f row 4): the struct-level layout of
// pronto::filter_state_t as rbisCreateFilterStateMessage / RBIS(const pronto_filter_state_t*) write and read it
// (MSE/rbis.cpp:268-285, MSE/rbis.hpp:58-67), pronto::indexed_measurement_t as IndexedMeasurementHandler::processMessage
// reads it (MSE/sensor_handlers.cpp:576-582), and the KVH batch decode of the Atlas INS path (estimate_tools/src/
// estimate_tools/imu_stream.cpp:62-97 + MSE/sensor_handlers.cpp:165-251).  The LCM byte encoding itself (big-endian
// marshalling + type fingerprint) is NOT produced: LCM and lcm-gen are absent and no log exists to check an encoder against.
#include <cuda_runtime.h>

#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include "../../include/rbis_batch.h"

int rbis_set_error(int code, const char* fmt, ...);  // rbis_batch.cu

struct rbis_kvh_stream {
  int64_t last_packet = -1, last_packet_utime = 0;  // IMUStream::IMUStream, imu_stream.cpp:4-8
  int32_t counter = 0;
};

extern "C" {

// ---- filter_state_t ----
int rbis_batch_get_filter_states(rbis_batch_t* h, int64_t first, int64_t count, rbis_filter_state_t* out) {
  if (!h || !out) return rbis_set_error(RBIS_ERR_INVALID, "null argument");
  const int64_t N = rbis_batch_num_filters(h);
  if (first < 0 || count < 0 || first + count > N) return rbis_set_error(RBIS_ERR_INVALID, "filter range out of bounds");
  if (count == 0) return 0;
  // whole-ensemble read, then the gather into array-of-structures messages (a few hundred MB at 65,536 filters: this is a
  // logging path, not the hot path)
  std::vector<double> vec((size_t)21 * N), quat((size_t)4 * N), cov((size_t)441 * N);
  int64_t utime = 0;
  if (int rc = rbis_batch_get_state(h, vec.data(), quat.data(), cov.data(), nullptr, &utime, RBIS_MEM_HOST)) return rc;
  for (int64_t k = 0; k < count; k++) {
    const int64_t n = first + k;
    rbis_filter_state_t& m = out[k];
    m.utime = utime;                                              // msg->utime = state.utime, rbis.cpp:272
    m.num_states = RBIS_NUM_STATES;                               // :274
    m.num_cov_elements = RBIS_NUM_STATES * RBIS_NUM_STATES;       // :275
    m.reserved0 = m.reserved1 = 0;
    for (int i = 0; i < 4; i++) m.quat[i] = quat[(size_t)i * N + n];            // quaternionToBotDouble: (w,x,y,z), :276
    for (int i = 0; i < 21; i++) m.state[i] = vec[(size_t)i * N + n];           // Map<VectorNd>(msg->state) = state.vec, :281
    for (int e = 0; e < 441; e++) m.cov[e] = cov[(size_t)e * N + n];            // Map<RBIM>(msg->cov) = cov: COLUMN-major, :282
  }
  return 0;
}

int rbis_record_filter_states(uint64_t fields, int32_t cov_blocks, const double* row, int64_t n_filters, int64_t utime,
                              int64_t first, int64_t count, rbis_filter_state_t* out) {
  if (!row || !out) return rbis_set_error(RBIS_ERR_INVALID, "null argument");
  if ((fields & 0x1FFFFFFull) != 0x1FFFFFFull || (fields >> 47) != 0)
    return rbis_set_error(RBIS_ERR_INVALID, "record fields 0x%llx: need fields 0..24 (vec, quat) and nothing above 46", (unsigned long long)fields);
  if (cov_blocks != 0x7F) return rbis_set_error(RBIS_ERR_INVALID, "record cov_blocks 0x%x: need all seven blocks (0x7f)", (unsigned)cov_blocks);
  if (n_filters <= 0 || first < 0 || count < 0 || first + count > n_filters)
    return rbis_set_error(RBIS_ERR_INVALID, "filter range out of bounds");
  // all seven blocks: packed covariance index = state index, so P(i, j) sits at kf + slot(i, j)
  const int64_t kf = __builtin_popcountll(fields);
  for (int64_t k = 0; k < count; k++) {
    const int64_t n = first + k;
    rbis_filter_state_t& m = out[k];
    m.utime = utime;
    m.num_states = RBIS_NUM_STATES;
    m.num_cov_elements = RBIS_NUM_STATES * RBIS_NUM_STATES;
    m.reserved0 = m.reserved1 = 0;
    for (int i = 0; i < 4; i++) m.quat[i] = row[(21 + i) * n_filters + n];
    for (int i = 0; i < 21; i++) m.state[i] = row[i * n_filters + n];
    for (int j = 0; j < 21; j++)
      for (int i = 0; i < 21; i++) {
        const int64_t s = i <= j ? j * (j + 1) / 2 + i : i * (i + 1) / 2 + j;
        m.cov[i + 21 * j] = row[(kf + s) * n_filters + n];  // column-major, both triangles (rbis.cpp:282)
      }
  }
  return 0;
}

int rbis_batch_set_filter_states(rbis_batch_t* h, int64_t first, int64_t count, const rbis_filter_state_t* msgs) {
  if (!h || !msgs) return rbis_set_error(RBIS_ERR_INVALID, "null argument");
  const int64_t N = rbis_batch_num_filters(h);
  if (first < 0 || count < 0 || first + count > N) return rbis_set_error(RBIS_ERR_INVALID, "filter range out of bounds");
  for (int64_t k = 0; k < count; k++) {
    const rbis_filter_state_t& m = msgs[k];
    if (m.num_states != RBIS_NUM_STATES)  // rbis.hpp:61-63 only warns; a batch cannot hold another size
      return rbis_set_error(RBIS_ERR_INVALID, "message %lld: num_states %d, expected %d", (long long)k, m.num_states, RBIS_NUM_STATES);
    if (m.num_cov_elements != RBIS_NUM_STATES * RBIS_NUM_STATES) return rbis_set_error(RBIS_ERR_INVALID, "message %lld: bad num_cov_elements", (long long)k);
    // RBIS(msg): vec = state, quat = botDoubleToQuaternion(msg->quat), utime (rbis.hpp:58-67); covariance = Map<const RBIM>(cov)
    // as the noise-id loader reads it (noise_id.cpp:83-86)
    if (int rc = rbis_batch_set_filter(h, first + k, m.state, m.quat, m.cov, 0.0)) return rc;
  }
  return 0;
}

// ---- indexed_measurement_t ----
int rbis_stream_from_indexed_measurement(const rbis_indexed_measurement_t* msg, rbis_stream_t* out, double* R_out) {
  if (!msg || !out || !R_out) return rbis_set_error(RBIS_ERR_INVALID, "null argument");
  const int m = msg->measured_dim;
  if (m < 1 || m > RBIS_MAX_MEAS) return rbis_set_error(RBIS_ERR_INVALID, "measured_dim %d out of range", m);
  if (msg->measured_cov_dim != m * m) return rbis_set_error(RBIS_ERR_INVALID, "measured_cov_dim %d is not measured_dim^2", msg->measured_cov_dim);
  std::memset(out, 0, sizeof(*out));
  out->m = m;
  out->has_orientation = 0;          // RBISIndexedMeasurement, sensor_handlers.cpp:578
  out->r_mode = RBIS_R_SHARED_FULL;
  out->sensor_id = 5;                // RBISUpdateInterface::indexed_sensor (rbis_update_interface.hpp sensor_enum)
  for (int a = 0; a < m; a++) {
    if (msg->z_indices[a] < 0 || msg->z_indices[a] >= RBIS_NUM_STATES) return rbis_set_error(RBIS_ERR_INVALID, "z_indices[%d] out of range", a);
    out->idx[a] = msg->z_indices[a];
  }
  // Map<const MatrixXd>(R_effective, m, m): column-major, exactly what rbis_stream_t.R expects
  std::memcpy(R_out, msg->R_effective, sizeof(double) * (size_t)m * m);
  out->R = R_out;
  return 0;
}

int rbis_stream_from_indexed_measurements(const rbis_indexed_measurement_t* msgs, int64_t count, rbis_stream_t* out, double* R_out) {
  if (!msgs || !out || !R_out || count < 1) return rbis_set_error(RBIS_ERR_INVALID, "null argument or count < 1");
  if (int rc = rbis_stream_from_indexed_measurement(&msgs[0], out, R_out)) return rc;
  const int m = out->m;
  const size_t mm = (size_t)m * m;
  bool same_R = true;
  for (int64_t k = 1; k < count; k++) {
    const rbis_indexed_measurement_t& g = msgs[k];
    if (g.measured_dim != m || g.measured_cov_dim != m * m)
      return rbis_set_error(RBIS_ERR_INVALID, "message %lld: measured_dim %d / measured_cov_dim %d differ from message 0", (long long)k,
                            g.measured_dim, g.measured_cov_dim);
    for (int a = 0; a < m; a++)
      if (g.z_indices[a] != out->idx[a]) return rbis_set_error(RBIS_ERR_INVALID, "message %lld: index set differs from message 0", (long long)k);
    std::memcpy(R_out + (size_t)k * mm, g.R_effective, sizeof(double) * mm);
    same_R = same_R && std::memcmp(g.R_effective, msgs[0].R_effective, sizeof(double) * mm) == 0;
  }
  out->r_mode = same_R ? RBIS_R_SHARED_FULL : RBIS_R_PER_ROW_FULL;
  out->rows = count;
  return 0;
}

// ---- KVH raw IMU batches ----
int rbis_kvh_stream_create(rbis_kvh_stream_t** out) {
  if (!out) return rbis_set_error(RBIS_ERR_INVALID, "out is NULL");
  *out = new (std::nothrow) rbis_kvh_stream();
  return *out ? 0 : rbis_set_error(RBIS_ERR_ALLOC, "host allocation failed");
}
int rbis_kvh_stream_destroy(rbis_kvh_stream_t* s) { delete s; return 0; }

// IMUStream::convertFromLCMBatch, imu_stream.cpp:62-97
int rbis_kvh_decode_batch(rbis_kvh_stream_t* s, int64_t batch_utime, int32_t num_packets, const rbis_kvh_packet_t* raw,
                          rbis_imu_packet_t* out_new, int32_t* n_new, rbis_imu_packet_t* out_old, int32_t* n_old) {
  if (!s || !raw || !out_new || !n_new || num_packets < 1) return rbis_set_error(RBIS_ERR_INVALID, "bad arguments");
  if (raw[0].packet_count < s->last_packet) {  // "Detected time skip, resetting IMUStream", :63-68
    s->last_packet = -1; s->last_packet_utime = 0; s->counter = 0;
  }
  int32_t nn = 0, no = 0;
  auto convert = [&](const rbis_kvh_packet_t& p, int64_t last_utime) {  // convertFromLCMPacket, :26-37
    rbis_imu_packet_t r;
    r.utime_raw = p.utime; r.utime_batch = batch_utime; r.utime_delta = p.utime - last_utime; r.utime = p.utime;
    r.packet_count = p.packet_count;
    for (int k = 0; k < 3; k++) { r.delta_rotation[k] = p.delta_rotation[k]; r.linear_acceleration[k] = p.linear_acceleration[k]; }
    return r;
  };
  for (int i = num_packets - 1; i >= 0; i--) {  // oldest first, :76
    if (raw[i].packet_count > s->last_packet) {
      out_new[nn++] = convert(raw[i], s->last_packet_utime);
      s->last_packet = raw[i].packet_count;
      s->last_packet_utime = raw[i].utime;
    } else if (out_old) {
      out_old[no++] = convert(raw[i], -raw[i].utime);  // "deliberately obfuscate the delta field", :88
    }
  }
  s->counter++;
  *n_new = nn;
  if (n_old) *n_old = no;
  return 0;
}

// q (w,x,y,z) applied to v: libbot bot_quat_rotate_to
static void quat_rotate(const double q[4], const double v[3], double out[3]) {
  const double w = q[0], x = q[1], y = q[2], z = q[3];
  const double ab = w * x, ac = w * y, ad = w * z, nbb = -x * x, bc = x * y, bd = x * z, ncc = -y * y, cd = y * z, ndd = -z * z;
  out[0] = 2 * ((ncc + ndd) * v[0] + (bc - ad) * v[1] + (ac + bd) * v[2]) + v[0];
  out[1] = 2 * ((ad + bc) * v[0] + (nbb + ndd) * v[1] + (cd - ab) * v[2]) + v[1];
  out[2] = 2 * ((bd - ac) * v[0] + (ab + cd) * v[1] + (nbb + ncc) * v[2]) + v[2];
}

// InsHandler::processMessageAtlas after the decode (sensor_handlers.cpp:186-251): the newest new packet of a batch ->
// the arguments of one RBISIMUProcessStep.  prev_utime: in/out, 0 before the first message (:239-246).
int rbis_kvh_imu_step(const rbis_imu_packet_t* newest, int64_t batch_utime, const double ins_to_body_quat[4],
                      const double ins_to_body_trans[3], double default_dt, int64_t* prev_utime, double gyro[3], double accel[3],
                      double* dt) {
  if (!newest || !ins_to_body_quat || !ins_to_body_trans || !prev_utime || !gyro || !accel || !dt) return rbis_set_error(RBIS_ERR_INVALID, "null argument");
  const double raw_dt = newest->utime_delta * 1E-6;  // :193
  const double sensor_gyro[3] = {newest->delta_rotation[0] / raw_dt, newest->delta_rotation[1] / raw_dt, newest->delta_rotation[2] / raw_dt};  // :209-212
  // bot_trans_apply_vec(&ins_to_body, linear_acceleration, body_accel): rotation AND translation, as the reference does (:227)
  quat_rotate(ins_to_body_quat, newest->linear_acceleration, accel);
  for (int k = 0; k < 3; k++) accel[k] += ins_to_body_trans[k];
  quat_rotate(ins_to_body_quat, sensor_gyro, gyro);  // bot_quat_rotate_to: rotation only (:234)
  *dt = (*prev_utime == 0) ? default_dt : (batch_utime - *prev_utime) * 1E-6;  // :239-244
  *prev_utime = batch_utime;
  return 0;
}

}  // extern "C"
