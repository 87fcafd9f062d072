// rbis_batch.cu -- host side of librbis_b200.so: the extern "C" batch API of include/rbis_batch.h
// over the sm_100a kernels in rbis_kernels.cuh / rbis_stats.cuh.  No CPU compute path exists here:
// every entry point that updates filters launches a CUDA kernel or fails.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/rbis_batch.h"
#include "rbis_kernels.cuh"   // namespace rbisk: the kernel parameter block and the layout-conversion kernels
#include "rbis_stats.cuh"
#include "rbis_smooth.cuh"
#include "rbis_synth.cuh"
// The fused kernels live in translation units of their own (rbis_fused_*.cu over rbis_fused_tu.inc): the dense
// lane-per-filter kernels, the decoupled ones at 384 / 256 / 128 filters per CTA and the warp-group kernels of rbis_group.cuh.
#include "rbis_fused_tu.h"

namespace {

thread_local std::string g_last_error;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

#define CUDA_TRY(expr)                                                                          \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess)                                                                      \
      return fail(RBIS_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

struct DevBuf {  // grow-only device buffer
  double* p = nullptr;
  size_t cap = 0;  // doubles
  int ensure(size_t n) {
    if (n <= cap) return 0;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    if (cudaMalloc(&p, n * sizeof(double)) != cudaSuccess) {
      cudaGetLastError();
      return -1;
    }
    cap = n;
    return 0;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

struct StagingSlot {  // device copies of caller-host input arrays for one fused run
  DevBuf imu;
  DevBuf z[RBIS_MAX_STREAMS], quat[RBIS_MAX_STREAMS], rdiag[RBIS_MAX_STREAMS];
  DevBuf f32;  // RBIS_MEM_F32_ROWS: device copy of the host float rows of one call (all arrays back to back), widened into the above
  DevBuf rtab; // RBIS_R_PER_ROW_FULL: the per-row R tables of the call's streams, back to back
  cudaEvent_t copied = nullptr, consumed = nullptr;
  int ring = -1;  // grouped launches: ring slot whose group events mark the consumption of this staging slot
};

}  // namespace

// shared with rbis_planner.cpp
int rbis_set_error(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

struct rbis_batch {
  int64_t N = 0;
  rbis_batch_config_t cfg{};
  int64_t utime = 0;
  int64_t launches = 0;
  cudaStream_t stream = nullptr;       // compute
  cudaStream_t copy_stream = nullptr;  // host->device input staging
  double *vec = nullptr, *quat = nullptr, *P = nullptr, *loglik = nullptr;
  double* qparams = nullptr;  // [4][N]
  double* snap = nullptr;
  std::vector<char> snap_valid;
  // ---- decoupled-filter tracking (rbis_kernels.cuh, "decoupled filters"): are the omega / a couplings of every
  // filter's covariance exactly zero?  -1 unknown (checked on the device before the next eligible fused launch),
  // 0 no, 1 yes.  snap_dc[slot] is the same for the content of a snapshot slot (0 = no or unknown).
  int decoupled = -1;
  std::vector<char> snap_dc;
  int* d_flag = nullptr;
  // ---- accelerometer notch cascade (rbis_batch_notch_*) ----
  rbisk::NotchCoeffs notch{};
  double* d_notch_state = nullptr;  // [3][MAX_NOTCH][4][notch_cols]
  int64_t notch_cols = 0;
  DevBuf notch_stage;               // device copy of a host chunk
  int last_variant = -1;  // kernel variant of the last fused launch: bit 1 decoupled, bit 0 with meas_block, bit 2 SYN (rows drawn in the kernel), bit 3 REC (the program records), bits 4.. lanes per filter (0 = one)
  int mapping = 1;        // lanes per filter of the fused kernels: 1 = lane-per-filter kernels, 2/4/8/16 = warp-group kernels
  int lane_tpb = 384;     // filters per CTA of the decoupled lane-per-filter kernels (384, 256, 128)
  int n_sms = 148;
  long long last_part = -1;  // filters per launch-group range of the last grouped launch (ranges differ between kernel variants)
  DevBuf full_cov;      // [441][N] scratch for set/get_state
  DevBuf misc;          // small scratch
  DevBuf stats_async;   // scratch of rbis_batch_stats_enqueue
  DevBuf synth_small;   // device copies of the noise-free rows and counters of rbis_batch_synthesize
  DevBuf stats_table;   // device-resident [total_chunks][96] table + [96] totals of rbis_batch_stats_allreduce
  rbisk::Op* d_ops = nullptr;
  size_t d_ops_cap = 0;
  double* d_rshared = nullptr;  // [MAX_STREAMS][81]
  StagingSlot slots[2];
  int slot_toggle = 0;
  // ---- column maps: [0] = IMU, [1 + s] = measurement stream s (nullptr = identity, array has N columns)
  int* d_map[1 + RBIS_MAX_STREAMS] = {};
  int64_t map_cols[1 + RBIS_MAX_STREAMS] = {};
  // ---- launch groups: the ensemble's CTAs are split into n_groups contiguous ranges, each launched on its own
  // stream, so that consecutive fused launches overlap (group g of launch k+1 starts when group g of launch k
  // is done) and the partially filled last wave of a launch does not idle SMs.  n_groups == 1: plain path.
  static constexpr int kMaxGroups = 8, kRing = 8;
  int n_groups = 1;
  cudaStream_t gstream[kMaxGroups] = {};
  cudaStream_t upload_stream = nullptr;
  cudaEvent_t gdone[kRing][kMaxGroups] = {};  // completion of group g of the launch that used ring slot r
  bool gdone_valid[kRing] = {};
  cudaEvent_t uploaded[kRing] = {};
  cudaEvent_t pre_evt = nullptr;
  cudaEvent_t syn_evt = nullptr;
  // ---- pinned host ring for the small per-call uploads (op table, shared R matrices, per-row R tables, noise-free synth rows): a
  // cudaMemcpyAsync from PAGEABLE memory makes the host wait until the stream has drained to the copy, which would stop
  // the host from running ahead of the device; from pinned memory it is truly asynchronous.
  static constexpr int kPinSlots = 16;
  static constexpr size_t kPinBytes = 128 << 10;
  char* pin_base = nullptr;
  cudaEvent_t pin_evt[kPinSlots] = {};
  int pin_next = 0;
  DevBuf d_syn;                 // noise-free rows of a fused-synthesis launch (plain path)
  DevBuf d_syn_ring[kRing];     // ... and per ring slot (grouped launches)
  rbisk::Op* d_ops_ring[kRing] = {};
  size_t d_ops_ring_cap[kRing] = {};
  double* d_rshared_ring[kRing] = {};
  int64_t launch_seq = 0;
  int last_ring = -1;
  bool groups_dirty = false;  // group streams hold work the main stream has not joined
  bool stream_dirty = true;   // the main stream got work since the last grouped launch
  cudaEvent_t tickets[8] = {};
  int next_ticket = 0;
  // ---- records (rbis_batch_set_record): RBIS_OP_RECORD ops write into the caller's device buffer in place; for a pinned host
  // buffer the kernels write the call's record rows into a staging buffer (double buffered across calls) that one copy on
  // rec_stream moves out after the call's last launches.  Nothing but the reuse of a staging buffer waits for that copy.
  bool rec_set = false;
  rbis_record_t rec{};
  int rec_k = 0;                          // doubles per filter and row: popcount(rec.fields) + the covariance entries
  cudaStream_t rec_stream = nullptr;
  cudaEvent_t rec_launched = nullptr;     // ungrouped launch done (rec_stream waits for it)
  DevBuf rec_stage[2];
  cudaEvent_t rec_copied[2] = {};         // the copy out of rec_stage[b] has run
  bool rec_pending[2] = {};
  int rec_toggle = 0;
  bool rec_copies = false;                // rec_stream has been given work
  cudaEvent_t ticket_rec[8] = {};         // rec_stream's position when ticket t was recorded
  bool ticket_rec_valid[8] = {};
  // ---- statistics over a snapshot slot on a side stream (rbis_batch_stats_snapshot_enqueue): the fused launches that follow do
  // not wait for it; a launch that REWRITES the slot waits for the slot's last reader
  cudaStream_t stats_stream = nullptr;
  std::vector<cudaEvent_t> snap_read_evt;   // per slot, created on first use
  std::vector<char> snap_read_pending;
  std::vector<DevBuf> snap_stats_scratch;   // per slot: truth [25] + chunk partials
  // ---- statistics over record or innovation rows (rbis_batch_stats_records_enqueue, rbis_batch_stats_innovations_enqueue),
  // on the same side stream: per device buffer a pending pass reads, the event after that pass; a fused call whose RECORD or
  // MEAS ops write into the buffer waits for it
  struct RowReader {
    const double *lo, *hi;  // [lo, hi): the record or innovation buffer
    cudaEvent_t done;
    bool pending;
  };
  std::vector<RowReader> row_readers;
  DevBuf rec_stats_scratch;                 // [truth [rows][25]] + tables [rows][chunks][96] + totals [rows][96]
  cudaEvent_t rec_stats_done = nullptr;     // the last pass (scratch reuse)
  bool rec_stats_pending = false;
  // ---- innovation sets (rbis_batch_set_innovations), per stream slot: MEAS ops on the stream write rows of innov[s].out
  bool innov_set[RBIS_MAX_STREAMS] = {};
  rbis_innovation_t innov[RBIS_MAX_STREAMS] = {};
  int innov_k[RBIS_MAX_STREAMS] = {};       // doubles per filter and row: NIS + m y + m S_DIAG + APPLIED
  // ---- NIS gates (rbis_batch_set_nis_gate), per stream slot: MEAS ops on the stream reject rows whose prior NIS exceeds the gate
  bool gate_set[RBIS_MAX_STREAMS] = {};
  rbis_nis_gate_t gate[RBIS_MAX_STREAMS] = {};
};

namespace {

// per stream in the shared-R device buffer: R (m x m column-major, 81), then for its correlated blocks the rows of
// L_R^-1 ([9][9] row-major, absolute row numbers) and D_R ([9]) of R_block = L_R D_R L_R^T (rbisk::RS_W, RS_D)
constexpr int kRShared = rbisk::RS_STRIDE;

static_assert(rbisk::OP_IMU == RBIS_OP_IMU && rbisk::OP_MEAS == RBIS_OP_MEAS && rbisk::OP_SNAPSHOT == RBIS_OP_SNAPSHOT &&
              rbisk::OP_RECORD == RBIS_OP_RECORD, "op kinds of the kernels and of the C ABI differ");
static_assert(rbisk::INNOV_NIS == RBIS_INNOV_NIS && rbisk::INNOV_Y == RBIS_INNOV_Y && rbisk::INNOV_S_DIAG == RBIS_INNOV_S_DIAG &&
                  rbisk::INNOV_APPLIED == RBIS_INNOV_APPLIED,
              "innovation fields of the kernels and of the C ABI differ");

constexpr int kMaxSmemOptin = 232448;
const rbis_fused_tu_t* const kTus[] = {&rbis_fused_tu_dense, &rbis_fused_tu_dc384, &rbis_fused_tu_dc256, &rbis_fused_tu_dc128,
                                       &rbis_fused_tu_g2,    &rbis_fused_tu_g4,    &rbis_fused_tu_g8,    &rbis_fused_tu_g16};
const rbis_fused_tu_t* group_tu(int G) {
  for (const rbis_fused_tu_t* t : kTus)
    if (t->lanes_per_filter == G) return t;
  return nullptr;
}
// the decoupled lane-per-filter kernels at tpb filters per CTA
const rbis_fused_tu_t* lane_tu(int tpb) {
  for (const rbis_fused_tu_t* t : kTus)
    if (t != &rbis_fused_tu_dense && t->lanes_per_filter == 1 && t->threads == tpb) return t;
  return nullptr;
}

// Launch geometry of a fused launch.  variant: bit 1 = decoupled, bit 0 = the program has measurement chunks other than
// aligned triples (lane-per-filter kernels only: the instantiations with meas1 / meas_block); mapping = lanes per filter;
// lane_tpb = filters per CTA of the decoupled lane-per-filter kernels (384, 256 or 128; the dense ones are 256).
struct LaunchGeom {
  unsigned grid;        // CTAs for the whole ensemble
  int threads, smem;
  long long fpc;        // filters per CTA
  const rbis_fused_tu_t* tu;
};
LaunchGeom launch_geom(int variant, int mapping, int lane_tpb, long long N, int n_sms) {
  LaunchGeom g{};
  if (mapping <= 1) {
    g.tu = (variant & 2) ? lane_tu(lane_tpb) : &rbis_fused_tu_dense;
    g.threads = g.tu->threads;
    g.smem = g.tu->smem;
    g.fpc = g.threads;
  } else {
    // warps per CTA so that the ensemble spreads over all SMs in whole waves
    g.tu = group_tu(mapping);
    const int stride = (variant & 2) ? (g.tu->smem_doubles_per_filter & 0xffff) : (g.tu->smem_doubles_per_filter >> 16);
    const int fpw = g.tu->filters_per_warp;
    int maxw = g.tu->max_warps;
    while (maxw > 1 && (long long)maxw * fpw * stride * 8 > kMaxSmemOptin) maxw--;
    const long long warps = (N + fpw - 1) / fpw;
    const long long waves = (warps + (long long)n_sms * maxw - 1) / ((long long)n_sms * maxw);
    long long wpc = (warps + n_sms * waves - 1) / (n_sms * waves);
    if (wpc > maxw) wpc = maxw;
    if (wpc < 1) wpc = 1;
    g.threads = 32 * (int)wpc;
    g.smem = (int)(wpc * fpw * stride * 8);
    g.fpc = wpc * fpw;
  }
  g.grid = (unsigned)((N + g.fpc - 1) / g.fpc);
  return g;
}

// variant bit 3: the program records or writes innovation sets (REC instantiations); bit 9 (+512): a stream skips NaN rows (MASK
// instantiations); bit 10 (+1024): the REC instantiations with the innovation path (INNOV); bit 11 (+2048, always with +512):
// the MASK instantiations with the NIS gates (GATE)
constexpr int kVariantMask = 512, kVariantInnov = 1024, kVariantGate = 2048;
cudaError_t launch_variant(int variant, int syn, const LaunchGeom& g, unsigned blocks, cudaStream_t st, const rbisk::KParams& kp) {
  const int rec = (variant & kVariantInnov) ? 2 : (variant & 8) ? 1 : 0;
  const int mask = (variant & kVariantGate) ? 2 : (variant & kVariantMask) ? 1 : 0;
  return g.tu->launch(variant & 1, (variant & 2) ? 1 : 0, syn, rec, mask, blocks, g.threads, g.smem, st, &kp);
}

// Automatic choice of the mapping (rbis_batch_config_t::mapping == 0) from the ensemble size: cycles per filter step of one
// wave of CTAs, measured on a B200 with dev/kbench (config-3 program, decoupled kernels; DESIGN.md 4.7), times the number
// of waves.  All candidates compute the same bits, so this is a pure scheduling decision.
struct MappingChoice {
  int mapping, lane_tpb;
};
// The decoupled lane-per-filter kernels of least cost (filters per CTA), and that cost.  One CTA per SM; large ensembles
// overlap their waves through the launch groups, so beyond one wave the cost grows with the CTA count, not with whole waves.
int auto_lane_tpb(long long N, int n_sms, double* cost = nullptr) {
  const struct { int tpb; double cyc; } lane[] = {{384, 16200.0}, {256, 12500.0}, {128, 9300.0}};
  double best = 1e300;
  int pick = 384;
  for (const auto& k : lane) {
    const long long ctas = (N + k.tpb - 1) / k.tpb;
    const double w = ctas <= n_sms ? 1.0 : (k.tpb == 384 ? (double)ctas / n_sms : (double)((ctas + n_sms - 1) / n_sms));
    if (w * k.cyc < best) { best = w * k.cyc; pick = k.tpb; }
  }
  if (cost) *cost = best;
  return pick;
}
MappingChoice auto_mapping(long long N, int n_sms) {
  double best;
  MappingChoice pick{1, auto_lane_tpb(N, n_sms, &best)};
  // warp groups of 4 lanes: one wave holds n_sms * 8 warps * 8 filters; cost grows with the warps per CTA
  const long long warps = (N + 7) / 8;
  const long long wv = (warps + (long long)n_sms * 8 - 1) / ((long long)n_sms * 8);
  const double wpc = (double)((warps + n_sms * wv - 1) / (n_sms * wv));
  if ((double)wv * (4300.0 + 560.0 * wpc) < best) pick = {4, 384};
  return pick;
}

int use_device(const rbis_batch* h) {
  cudaError_t e = cudaSetDevice(h->cfg.device);
  if (e != cudaSuccess) return fail(RBIS_ERR_CUDA, "cudaSetDevice(%d): %s", h->cfg.device, cudaGetErrorString(e));
  return 0;
}

// Every entry point that enqueues work on the main stream calls this first: the main stream joins the group
// streams (so it sees the results of grouped launches), and the next grouped launch will wait for it.
int main_stream_work(rbis_batch* h) {
  if (h->groups_dirty) {
    for (int g = 0; g < h->n_groups; g++) CUDA_TRY(cudaStreamWaitEvent(h->stream, h->gdone[h->last_ring][g], 0));
    h->groups_dirty = false;
  }
  h->stream_dirty = true;
  return 0;
}

// Split the m rows of a measurement into consecutive chunks along which R is block diagonal (the finest such blocks).
// Three consecutive one-row blocks on an aligned index triple (3k, 3k+1, 3k+2) are merged into one chunk for the unrolled
// meas3<I0> path; every other one-row block is a chunk of its own for the scalar path meas1 (chunk_fast = 100 + index);
// blocks of two or more correlated rows that are not an aligned triple take the general path.
void mark_fast_chunks(rbisk::StreamDesc& d, bool* needs_general) {
  for (int c = 0; c < d.n_chunks; c++) {
    const int a0 = d.chunk_start[c];
    const bool triple = d.chunk_len[c] == 3 && d.idx[a0] % 3 == 0 && d.idx[a0 + 1] == d.idx[a0] + 1 && d.idx[a0 + 2] == d.idx[a0] + 2;
    if (triple) d.chunk_fast[c] = d.idx[a0];
    else {
      d.chunk_fast[c] = d.chunk_len[c] == 1 ? 100 + d.idx[a0]   // one row: meas1
                                            : -1;               // correlated rows: meas_block on the decorrelated rows
      *needs_general = true;  // either lives in the BLOCKS kernel instantiations only
    }
  }
}

// R_block = L D L^T (unit lower L) of rows/columns a0..a0+len-1 of the m x m column-major R; writes the rows of L^-1 into
// W[(a0+a)*9 + (a0+b)] and D into Dg[a0+a].  With z' = L^-1 z the block becomes `len` scalar measurements with
// uncorrelated noise D, which the device applies one after the other (meas_block).
int decorrelate_block(const double* R, int m, int a0, int len, double* W, double* Dg) {
  double L[RBIS_MAX_MEAS][RBIS_MAX_MEAS] = {}, D[RBIS_MAX_MEAS] = {};
  for (int k = 0; k < len; k++) {
    double d = R[(a0 + k) + (size_t)m * (a0 + k)];
    for (int p = 0; p < k; p++) d -= L[k][p] * L[k][p] * D[p];
    if (!(d > 0)) return fail(RBIS_ERR_INVALID, "measurement covariance block at row %d is not positive definite", a0);
    D[k] = d;
    L[k][k] = 1.0;
    for (int i = k + 1; i < len; i++) {
      double v = R[(a0 + i) + (size_t)m * (a0 + k)];
      for (int p = 0; p < k; p++) v -= L[i][p] * L[k][p] * D[p];
      L[i][k] = v / d;
    }
  }
  // invert the unit lower triangle by forward substitution, column by column
  for (int c = 0; c < len; c++) {
    double x[RBIS_MAX_MEAS] = {};
    for (int i = c; i < len; i++) {
      double v = (i == c) ? 1.0 : 0.0;
      for (int k = c; k < i; k++) v -= L[i][k] * x[k];
      x[i] = v;
    }
    for (int i = c; i < len; i++) W[(a0 + i) * RBIS_MAX_MEAS + (a0 + c)] = x[i];
  }
  for (int k = 0; k < len; k++) Dg[a0 + k] = D[k];
  return 0;
}

// R_host: the m x m matrix whose off-diagonal zero pattern decides the cuts (for RBIS_R_PER_ROW_FULL, the union over the
// rows of the call: every row of the stream then runs the same chunk plan)
void plan_chunks(int m, int r_mode, const double* R_host, rbisk::StreamDesc& d) {
  std::vector<int> cut;  // start indices of the finest blocks
  cut.push_back(0);
  for (int k = 1; k < m; k++) {
    bool sep = true;
    if (r_mode != RBIS_R_PER_FILTER_DIAG) {
      for (int a = 0; a < k && sep; a++)
        for (int b = k; b < m; b++)
          if (R_host[a + m * b] != 0.0 || R_host[b + m * a] != 0.0) { sep = false; break; }
    }
    if (sep) cut.push_back(k);
  }
  cut.push_back(m);
  d.n_chunks = 0;
  auto aligned_triple = [&](int a) {
    return d.idx[a] % 3 == 0 && d.idx[a + 1] == d.idx[a] + 1 && d.idx[a + 2] == d.idx[a] + 2;
  };
  for (size_t i = 0; i + 1 < cut.size();) {
    const int a = cut[i], blen = cut[i + 1] - cut[i];
    // three one-row blocks in a row on an aligned index triple -> one chunk
    if (blen == 1 && i + 3 < cut.size() && cut[i + 2] - cut[i + 1] == 1 && cut[i + 3] - cut[i + 2] == 1 && aligned_triple(a)) {
      d.chunk_start[d.n_chunks] = a;
      d.chunk_len[d.n_chunks++] = 3;
      i += 3;
      continue;
    }
    d.chunk_start[d.n_chunks] = a;
    d.chunk_len[d.n_chunks++] = blen;
    i += 1;
  }
}

// cudaMemcpyAsync of a small host block through the handle's pinned ring (falls back to the pageable copy when it does not fit)
int upload_small(rbis_batch* h, void* dst, const void* src, size_t bytes, cudaStream_t st) {
  if (bytes == 0) return 0;
  if (!h->pin_base || bytes > rbis_batch::kPinBytes) {
    CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
    return 0;
  }
  const int k = h->pin_next;
  h->pin_next = (k + 1) % rbis_batch::kPinSlots;
  CUDA_TRY(cudaEventSynchronize(h->pin_evt[k]));  // the copy that last used this slot (16 uploads ago) has run
  char* p = h->pin_base + (size_t)k * rbis_batch::kPinBytes;
  std::memcpy(p, src, bytes);
  CUDA_TRY(cudaMemcpyAsync(dst, p, bytes, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaEventRecord(h->pin_evt[k], st));
  return 0;
}

int copy_in(rbis_batch* h, DevBuf& buf, const double* src, size_t count, int mem, cudaStream_t st,
            const double** out) {
  if (mem == RBIS_MEM_DEVICE) {
    *out = src;
    return 0;
  }
  if (buf.ensure(count)) return fail(RBIS_ERR_ALLOC, "device staging allocation of %zu doubles failed", count);
  CUDA_TRY(cudaMemcpyAsync(buf.p, src, count * sizeof(double), cudaMemcpyHostToDevice, st));
  *out = buf.p;
  (void)h;
  return 0;
}

// RBIS_MEM_F32_ROWS: float rows -> the double staging array (exact), on the copy stream
__global__ void widen_rows_kernel(const float* __restrict__ in, double* __restrict__ out, size_t n) {
  const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i + 3 < n && (reinterpret_cast<uintptr_t>(in) & 15) == 0) {
    const float4 v = *reinterpret_cast<const float4*>(in + i);
    reinterpret_cast<double2*>(out + i)[0] = make_double2((double)v.x, (double)v.y);
    reinterpret_cast<double2*>(out + i)[1] = make_double2((double)v.z, (double)v.w);
  } else {
    for (size_t k = i; k < n; k++) out[k] = (double)in[k];
  }
}
// f32_base / f32_off: the call's float scratch (device) and the running offset in floats (kept a multiple of 4)
int copy_in_f32(rbis_batch* h, DevBuf& buf, const void* src, size_t count, int mem, cudaStream_t st, float* f32_base, size_t* f32_off,
                const double** out) {
  if (buf.ensure(count)) return fail(RBIS_ERR_ALLOC, "device staging allocation of %zu doubles failed", count);
  const float* dsrc = static_cast<const float*>(src);
  if (mem == RBIS_MEM_HOST) {
    float* d = f32_base + *f32_off;
    CUDA_TRY(cudaMemcpyAsync(d, src, count * sizeof(float), cudaMemcpyHostToDevice, st));
    *f32_off += (count + 3) & ~(size_t)3;
    dsrc = d;
  }
  widen_rows_kernel<<<(unsigned)((count + 1023) / 1024), 256, 0, st>>>(dsrc, buf.p, count);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  *out = buf.p;
  return 0;
}

int validate_stream(int s, const rbis_stream_t& in) {
  if (in.m < 1 || in.m > RBIS_MAX_MEAS) return fail(RBIS_ERR_INVALID, "stream %d: m=%d out of range", s, in.m);
  for (int a = 0; a < in.m; a++)
    if (in.idx[a] < 0 || in.idx[a] >= RBIS_NUM_STATES) return fail(RBIS_ERR_INVALID, "stream %d: index %d out of range", s, in.idx[a]);
  if (in.rows < 0) return fail(RBIS_ERR_INVALID, "stream %d: negative rows", s);
  if (in.rows > 0 && (!in.z || !in.R)) return fail(RBIS_ERR_INVALID, "stream %d: z and R are required", s);
  if (in.has_orientation && in.rows > 0 && !in.quat) return fail(RBIS_ERR_INVALID, "stream %d: has_orientation but quat is NULL", s);
  if (in.r_mode != RBIS_R_SHARED_FULL && in.r_mode != RBIS_R_PER_FILTER_DIAG && in.r_mode != RBIS_R_PER_ROW_FULL)
    return fail(RBIS_ERR_INVALID, "stream %d: bad r_mode", s);
  if (in.flags & ~RBIS_STREAM_SKIP_NAN_ROWS) return fail(RBIS_ERR_INVALID, "stream %d: unknown flags 0x%x", s, (unsigned)in.flags);
  return 0;
}

// The device table of one R (layout of rbisk::RS_STRIDE): the m x m matrix, then for the correlated chunks the rows of
// L^-1 and D (decorrelate_block).  Without correlated chunks only the matrix is read, so a per-row stream stores m * m.
int r_table(const double* R, const rbisk::StreamDesc& d, double* out) {
  std::memcpy(out, R, sizeof(double) * d.m * d.m);
  for (int c = 0; c < d.n_chunks; c++)
    if (d.chunk_fast[c] == -1)
      if (int rc = decorrelate_block(R, d.m, d.chunk_start[c], d.chunk_len[c], out + rbisk::RS_W, out + rbisk::RS_D)) return rc;
  return 0;
}

}  // namespace
extern "C" int synthesize_into(rbis_batch_t* h, const rbis_synth_t* syn, double* imu_out, double* const* z_out, double* const* quat_out, cudaStream_t stream);
namespace {

// Pending side-stream passes that read [lo, hi): their events go to `waits` and they stop being pending.
void take_readers(rbis_batch* h, const double* lo, const double* hi, std::vector<cudaEvent_t>& waits) {
  for (auto& r : h->row_readers)
    if (r.pending && r.lo < hi && lo < r.hi) {
      waits.push_back(r.done);
      r.pending = false;
    }
}

// The side-stream pass of rbis_batch_stats_records_enqueue / rbis_batch_stats_innovations_enqueue over n_rows rows of the
// device buffer [lo, hi): the reader entry of the buffer, the scratch ([pre] + tables [n_rows][nch][96] + totals
// [n_rows][96]), ordering after the launches that wrote the rows, `pre` uploaded, launch(ss, d_pre, d_tables, r0, ny, nch)
// for the tables of rows r0..r0+ny-1 (at most 65535 rows, the gridDim.y limit), the tables and optional totals copied out,
// the reader event and a ticket.
template <class Launch>
int row_stats_pass(rbis_batch* h, const double* lo, const double* hi, int64_t n_rows, int chunk, const std::vector<double>& pre,
                   double* out_chunks, double* out_totals, int64_t* n_chunks, int32_t* ticket, Launch&& launch) {
  if (int rc = use_device(h)) return rc;
  if (!h->stats_stream) {
    CUDA_TRY(cudaStreamCreateWithFlags(&h->stats_stream, cudaStreamNonBlocking));
    h->snap_read_evt.assign((size_t)h->cfg.snapshot_slots, nullptr);
    h->snap_read_pending.assign((size_t)h->cfg.snapshot_slots, 0);
    h->snap_stats_scratch.resize((size_t)h->cfg.snapshot_slots);
  }
  if (!h->rec_stats_done) CUDA_TRY(cudaEventCreateWithFlags(&h->rec_stats_done, cudaEventDisableTiming));
  // the reader entry of this buffer (buffers no pass reads any more are dropped)
  rbis_batch::RowReader* rd = nullptr;
  for (auto& r : h->row_readers)
    if (r.lo == lo && r.hi == hi) rd = &r;
  if (!rd) {
    for (size_t i = 0; i < h->row_readers.size();)
      if (!h->row_readers[i].pending) {
        cudaEventDestroy(h->row_readers[i].done);
        h->row_readers.erase(h->row_readers.begin() + (long)i);
      } else {
        i++;
      }
    cudaEvent_t e;
    CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    h->row_readers.push_back({lo, hi, e, false});
    rd = &h->row_readers.back();
  }
  const size_t N = (size_t)h->N;
  const int64_t nch = (int64_t)((N + chunk - 1) / chunk);
  const size_t n_table = (size_t)nch * RBIS_NUM_STATS;
  const size_t need = pre.size() + (size_t)n_rows * (n_table + RBIS_NUM_STATS);
  DevBuf& scratch = h->rec_stats_scratch;
  if (scratch.cap < need) {
    if (h->rec_stats_pending) CUDA_TRY(cudaEventSynchronize(h->rec_stats_done));  // the last pass still reads the old scratch
    if (scratch.ensure(need)) return fail(RBIS_ERR_ALLOC, "scratch allocation failed");
  }
  cudaStream_t ss = h->stats_stream;
  // after the launches that wrote the rows: the group streams of the last fused call, or the main stream; the main stream is
  // NOT made to join anything (as rbis_batch_stats_snapshot_enqueue)
  if (h->groups_dirty) {
    for (int g = 0; g < h->n_groups; g++) CUDA_TRY(cudaStreamWaitEvent(ss, h->gdone[h->last_ring][g], 0));
  }
  if (!h->syn_evt) CUDA_TRY(cudaEventCreateWithFlags(&h->syn_evt, cudaEventDisableTiming));
  CUDA_TRY(cudaEventRecord(h->syn_evt, h->stream));
  CUDA_TRY(cudaStreamWaitEvent(ss, h->syn_evt, 0));
  double* d_pre = scratch.p;
  double* d_tables = d_pre + pre.size();
  double* d_totals = d_tables + (size_t)n_rows * n_table;
  if (!pre.empty())
    if (int rc = upload_small(h, d_pre, pre.data(), pre.size() * sizeof(double), ss)) return rc;
  constexpr int64_t kMaxY = 65535;  // gridDim.y limit
  for (int64_t r0 = 0; r0 < n_rows; r0 += kMaxY) {
    const int64_t ny = std::min<int64_t>(kMaxY, n_rows - r0);
    launch(ss, d_pre, d_tables + (size_t)r0 * n_table, r0, ny, nch);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
  }
  CUDA_TRY(cudaMemcpyAsync(out_chunks, d_tables, (size_t)n_rows * n_table * sizeof(double), cudaMemcpyDeviceToHost, ss));
  if (out_totals) {
    rbisk::reduce_chunk_table_kernel<<<(unsigned)n_rows, 128, 0, ss>>>(d_tables, (long long)nch, d_totals);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    CUDA_TRY(cudaMemcpyAsync(out_totals, d_totals, (size_t)n_rows * RBIS_NUM_STATS * sizeof(double), cudaMemcpyDeviceToHost, ss));
  }
  CUDA_TRY(cudaEventRecord(rd->done, ss));
  rd->pending = true;
  CUDA_TRY(cudaEventRecord(h->rec_stats_done, ss));
  h->rec_stats_pending = true;
  const int t = h->next_ticket;
  h->next_ticket = (t + 1) % 8;
  CUDA_TRY(cudaEventRecord(h->tickets[t], ss));
  *ticket = t;
  if (n_chunks) *n_chunks = nch;
  return 0;
}

// syn != nullptr: the input rows are synthesised on the device into the staging slot (rbis_batch_run_fused_synth) instead of
// being copied from the host; everything else -- double buffering, overlap with the previous launch -- is the host path's.
// use_innov = false: the single-update entry points, which ignore innovation sets and NIS gates
int launch_fused(rbis_batch* h, int64_t n_ops, const rbis_op_t* ops, const double* imu, int64_t imu_rows,
                 int n_streams, const rbis_stream_t* streams_in, int mem, bool use_maps = true,
                 const rbis_synth_t* syn = nullptr, bool use_innov = true) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (n_ops < 0 || (n_ops > 0 && !ops)) return fail(RBIS_ERR_INVALID, "bad op list");
  if (n_streams < 0 || n_streams > RBIS_MAX_STREAMS) return fail(RBIS_ERR_INVALID, "n_streams out of range");
  const bool f32_rows = (mem & RBIS_MEM_F32_ROWS) != 0;
  mem &= ~RBIS_MEM_F32_ROWS;
  if (mem != RBIS_MEM_HOST && mem != RBIS_MEM_DEVICE) return fail(RBIS_ERR_INVALID, "bad mem");
  if (f32_rows && syn) return fail(RBIS_ERR_INVALID, "RBIS_MEM_F32_ROWS does not apply to synthesised inputs");
  if (n_ops == 0) return 0;
  if (int rc = use_device(h)) return rc;
  const int64_t N = h->N;
  std::vector<rbis_stream_t> stream_copy;
  const rbis_stream_t* streams = streams_in;
  if (syn) {
    // rows come from the synth description; z / quat pointers are filled in below once the staging buffers exist
    if (n_streams != syn->n_streams) return fail(RBIS_ERR_INVALID, "n_streams differs from syn->n_streams");
    stream_copy.assign(streams_in, streams_in + n_streams);
    for (int s = 0; s < n_streams; s++) {
      const rbis_synth_stream_t& ss = syn->streams[s];
      if (ss.m != stream_copy[s].m || (ss.has_orientation != 0) != (stream_copy[s].has_orientation != 0))
        return fail(RBIS_ERR_INVALID, "stream %d: synth description does not match the stream", s);
      stream_copy[s].rows = ss.rows;
      stream_copy[s].z = reinterpret_cast<const double*>(8);     // placeholders for validation; replaced below
      stream_copy[s].quat = ss.has_orientation ? reinterpret_cast<const double*>(8) : nullptr;
    }
    streams = stream_copy.data();
    imu = syn->imu_rows > 0 ? reinterpret_cast<const double*>(8) : nullptr;
    imu_rows = syn->imu_rows;
    mem = RBIS_MEM_DEVICE;  // per-filter R arrays are device arrays on this path
  }

  // ---- validate ops and translate ----
  std::vector<rbisk::Op> kops((size_t)n_ops);
  std::vector<char> snap_valid = h->snap_valid;
  // decoupled-kernel eligibility of the program: every RESTORE must read a slot whose content is decoupled (written
  // by a decoupled launch, or by an earlier SNAPSHOT of this program)
  std::vector<char> snap_dc = h->snap_dc;
  bool restores_ok = true, any_snapshot = false;
  bool any_record = false;
  std::vector<int64_t> rec_rows;  // record rows of the call, in op order
  bool innov_used[RBIS_MAX_STREAMS] = {};  // streams whose innovation set a MEAS op of the call writes
  bool meas_on[RBIS_MAX_STREAMS] = {};     // streams a MEAS op of the call updates on
  int64_t last_utime = h->utime;
  for (int64_t i = 0; i < n_ops; i++) {
    const rbis_op_t& o = ops[i];
    rbisk::Op& k = kops[(size_t)i];
    k.kind = o.kind; k.stream = o.stream; k.row = o.row; k.dt = o.dt;
    switch (o.kind) {
      case RBIS_OP_IMU:
        if (!imu) return fail(RBIS_ERR_INVALID, "op %lld is an IMU op but imu is NULL", (long long)i);
        if (o.row < 0 || o.row >= imu_rows) return fail(RBIS_ERR_INVALID, "op %lld: imu row %lld out of range", (long long)i, (long long)o.row);
        if (!(o.dt > 0)) return fail(RBIS_ERR_INVALID, "op %lld: dt must be positive", (long long)i);
        last_utime = o.utime;
        break;
      case RBIS_OP_MEAS:
        if (o.stream < 0 || o.stream >= n_streams) return fail(RBIS_ERR_INVALID, "op %lld: stream %d out of range", (long long)i, o.stream);
        if (o.row < 0 || o.row >= streams[o.stream].rows) return fail(RBIS_ERR_INVALID, "op %lld: row %lld out of range for stream %d", (long long)i, (long long)o.row, o.stream);
        if (use_innov && h->innov_set[o.stream]) {
          if (o.row >= h->innov[o.stream].rows)
            return fail(RBIS_ERR_INVALID, "op %lld: row %lld out of range for the innovation set of stream %d (%lld rows)", (long long)i,
                        (long long)o.row, o.stream, (long long)h->innov[o.stream].rows);
          innov_used[o.stream] = true;
        }
        meas_on[o.stream] = true;
        last_utime = o.utime;
        break;
      case RBIS_OP_SNAPSHOT:
        if (o.row < 0 || o.row >= h->cfg.snapshot_slots) return fail(RBIS_ERR_INVALID, "op %lld: snapshot slot %lld out of range (%d slots)", (long long)i, (long long)o.row, h->cfg.snapshot_slots);
        snap_valid[(size_t)o.row] = 1;
        snap_dc[(size_t)o.row] = 2;  // "as this launch": resolved once the variant is known
        any_snapshot = true;
        break;
      case RBIS_OP_RESTORE:
        if (o.row < 0 || o.row >= h->cfg.snapshot_slots) return fail(RBIS_ERR_INVALID, "op %lld: snapshot slot %lld out of range (%d slots)", (long long)i, (long long)o.row, h->cfg.snapshot_slots);
        if (!snap_valid[(size_t)o.row]) return fail(RBIS_ERR_STATE, "op %lld: restore of empty snapshot slot %lld", (long long)i, (long long)o.row);
        if (!snap_dc[(size_t)o.row]) restores_ok = false;
        last_utime = o.utime;
        break;
      case RBIS_OP_RECORD:  // changes neither the filters nor the ensemble's utime
        if (!h->rec_set) return fail(RBIS_ERR_STATE, "op %lld: RBIS_OP_RECORD but no record set (rbis_batch_set_record)", (long long)i);
        if (o.row < 0 || o.row >= h->rec.rows) return fail(RBIS_ERR_INVALID, "op %lld: record row %lld out of range (%lld rows)", (long long)i, (long long)o.row, (long long)h->rec.rows);
        rec_rows.push_back(o.row);
        any_record = true;
        break;
      default:
        return fail(RBIS_ERR_INVALID, "op %lld: unknown kind %d", (long long)i, o.kind);
    }
  }

  rbisk::KParams kp;
  std::memset(&kp, 0, sizeof(kp));
  kp.N = N;
  kp.vec = h->vec; kp.quat = h->quat; kp.P = h->P; kp.loglik = h->loglik;
  kp.q_gyro = h->qparams; kp.q_accel = h->qparams + N; kp.q_gyro_bias = h->qparams + 2 * N;
  kp.q_accel_bias = h->qparams + 3 * N;
  kp.snap = h->snap;
  kp.n_snap = h->cfg.snapshot_slots;
  kp.n_ops = n_ops;
  kp.g_val = h->cfg.g_val; kp.chi_tol = h->cfg.chi_tol;
  kp.ctor_folds_chi = h->cfg.ctor_folds_chi; kp.renorm = h->cfg.renormalize_quat;

  // ---- measurement streams: index sets, chunks, kernel variant (no data movement yet) ----
  kp.imu_map = use_maps ? h->d_map[0] : nullptr;
  kp.imu_cols = kp.imu_map ? h->map_cols[0] : N;
  std::vector<double> rshared((size_t)RBIS_MAX_STREAMS * kRShared, 0.0);
  bool any_shared = false;
  bool shared_r[RBIS_MAX_STREAMS] = {};
  std::vector<double> rtab_host;                  // RBIS_R_PER_ROW_FULL tables of all streams, staged like z
  size_t rtab_off[RBIS_MAX_STREAMS] = {};
  bool needs_general = false;  // some chunk is not an aligned triple -> the kernel instantiations that contain meas1 / meas_block
  bool passive_index = false;  // some stream measures omega or a directly -> couplings become non-zero
  for (int s = 0; s < n_streams; s++) {
    const rbis_stream_t& in = streams[s];
    rbisk::StreamDesc& d = kp.streams[s];
    if (int rc = validate_stream(s, in)) return rc;
    if (use_innov && h->innov_set[s] && h->innov[s].m != in.m)
      return fail(RBIS_ERR_INVALID, "stream %d has m = %d, its innovation set m = %d", s, in.m, h->innov[s].m);
    if (in.flags & RBIS_STREAM_SKIP_NAN_ROWS) {
      if (syn) return fail(RBIS_ERR_INVALID, "stream %d: RBIS_STREAM_SKIP_NAN_ROWS does not apply to synthesised inputs (z is drawn, not read)", s);
      kp.skip_nan_streams |= 1u << s;
    }
    d.m = in.m; d.has_orient = in.has_orientation ? 1 : 0; d.r_mode = in.r_mode;
    for (int a = 0; a < in.m; a++) d.idx[a] = in.idx[a];
    d.map = use_maps ? h->d_map[1 + s] : nullptr;
    d.cols = d.map ? h->map_cols[1 + s] : N;
    if (in.rows == 0) { d.n_chunks = 0; continue; }
    const size_t mm = (size_t)in.m * in.m;
    if (in.r_mode == RBIS_R_PER_ROW_FULL) {
      // off-diagonal non-zeros of any row cut the chunks of every row; rows that all share one R plan as that R does
      std::vector<double> pattern(mm, 0.0);
      for (int64_t r = 0; r < in.rows; r++)
        for (size_t k = 0; k < mm; k++)
          if (in.R[(size_t)r * mm + k] != 0.0) pattern[k] = 1.0;
      plan_chunks(in.m, in.r_mode, pattern.data(), d);
    } else {
      plan_chunks(in.m, in.r_mode, in.r_mode == RBIS_R_SHARED_FULL ? in.R : nullptr, d);
    }
    mark_fast_chunks(d, &needs_general);
    for (int a = 0; a < in.m; a++)
      if (!rbisk::is_act(in.idx[a])) passive_index = true;
    if (in.r_mode == RBIS_R_SHARED_FULL) {
      if (int rc = r_table(in.R, d, &rshared[(size_t)s * kRShared])) return rc;
      d.R = h->d_rshared + (size_t)s * kRShared;  // grouped launches: re-pointed into the piece's ring slot below
      shared_r[s] = true;
      any_shared = true;
    } else if (in.r_mode == RBIS_R_PER_ROW_FULL) {
      bool blocks = false;
      for (int c = 0; c < d.n_chunks; c++) blocks = blocks || d.chunk_fast[c] == -1;
      d.r_stride = blocks ? kRShared : (long long)mm;
      rtab_off[s] = rtab_host.size();
      rtab_host.resize(rtab_host.size() + (size_t)in.rows * (size_t)d.r_stride, 0.0);
      for (int64_t r = 0; r < in.rows; r++)
        if (r_table(in.R + (size_t)r * mm, d, &rtab_host[rtab_off[s] + (size_t)r * (size_t)d.r_stride])) {
          const std::string why = g_last_error;
          return fail(RBIS_ERR_INVALID, "stream %d, stream row %lld: %s", s, (long long)r, why.c_str());
        }
    }
  }
  // NIS gates of the streams the program updates on; an innovation set that asks for INNOV_APPLIED needs the GATE
  // instantiations too (gated or not, they are the ones that write the entry)
  bool gate_kernels = false;
  for (int s = 0; s < n_streams; s++) {
    if (use_innov && h->gate_set[s] && meas_on[s]) {
      kp.gate_streams |= 1u << s;
      kp.gate_nis[s] = h->gate[s].nis_max;
      kp.gate_nis_filter[s] = h->gate[s].nis_max_per_filter;
      gate_kernels = true;
    }
    if (innov_used[s] && (h->innov[s].fields & RBIS_INNOV_APPLIED)) gate_kernels = true;
  }
  // ---- kernel variant ----
  // skipping or rejecting a row changes no coupling, so decoupled eligibility does not depend on the MASK / GATE instantiations
  int variant = (needs_general ? 1 : 0) | (kp.skip_nan_streams ? kVariantMask : 0) | (gate_kernels ? kVariantMask | kVariantGate : 0);
  const bool dc_eligible = !h->cfg.dense_only && !passive_index && restores_ok;
  if (dc_eligible && h->decoupled < 0) {
    // one device pass over the couplings, then a host read: happens once after set_state / set_filter, not per launch
    if (int rc = main_stream_work(h)) return rc;
    CUDA_TRY(cudaMemsetAsync(h->d_flag, 0, sizeof(int), h->stream));
    rbisk::coupling_check_kernel<<<(unsigned)((N + 255) / 256), 256, 0, h->stream>>>(h->P, (long long)N, h->d_flag);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    int flag = 0;
    CUDA_TRY(cudaMemcpyAsync(&flag, h->d_flag, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    h->decoupled = flag ? 0 : 1;
  }
  if (dc_eligible && h->decoupled == 1) variant |= 2;
  // Synthesised inputs: the decoupled kernels have SYN instantiations that draw the rows themselves (mode 1), so nothing is
  // materialised and the launch reads no per-filter input; otherwise the rows are generated into the staging slot first.  The
  // GATE instantiations read their rows from HBM: a gated program materialises them.
  const bool fuse_syn = syn != nullptr && syn->mode == 1 && !h->cfg.synth_materialize && (variant & 2) != 0 &&
                        (h->mapping > 1 || !(variant & 1)) && !gate_kernels;
  if (syn) {
    if (kp.imu_map) return fail(RBIS_ERR_STATE, "synthesised inputs draw one column per filter: clear the column maps first");
    for (int s = 0; s < n_streams; s++)
      if (use_maps && h->d_map[1 + s]) return fail(RBIS_ERR_STATE, "synthesised inputs draw one column per filter: clear the column maps first");
    if ((syn->sigma_gyro < 0 || syn->sigma_accel < 0) && !(syn->dt > 0)) return fail(RBIS_ERR_INVALID, "per-filter IMU noise needs dt > 0");
  }
  // the noise-free rows of a fused-synthesis launch as one host block: [imu_mean | imu_step | per stream: mean, mean_quat, step]
  std::vector<double> syn_host;
  size_t syn_o_imu = 0, syn_o_istep = 0, syn_o_mean[RBIS_MAX_STREAMS] = {}, syn_o_q[RBIS_MAX_STREAMS] = {}, syn_o_step[RBIS_MAX_STREAMS] = {};
  if (fuse_syn) {
    if (syn->imu_rows > 0 && (!syn->imu_mean || !syn->imu_step)) return fail(RBIS_ERR_INVALID, "bad synth IMU description");
    size_t words = (size_t)syn->imu_rows * 7;
    for (int s = 0; s < n_streams; s++) {
      const rbis_synth_stream_t& ss = syn->streams[s];
      if (ss.rows > 0 && (!ss.mean || !ss.step)) return fail(RBIS_ERR_INVALID, "synth stream %d: mean and step are required", s);
      if (ss.has_orientation && ss.rows > 0 && !ss.mean_quat) return fail(RBIS_ERR_INVALID, "synth stream %d: mean_quat is required", s);
      words += (size_t)ss.rows * (ss.m + 1 + (ss.has_orientation ? 4 : 0));
    }
    syn_host.resize(words + 1);
    size_t off = 0;
    auto put = [&](const void* src, size_t n_words) { if (n_words) std::memcpy(syn_host.data() + off, src, n_words * 8); off += n_words; return off - n_words; };
    syn_o_imu = put(syn->imu_mean, (size_t)syn->imu_rows * 6);
    syn_o_istep = put(syn->imu_step, (size_t)syn->imu_rows);
    for (int s = 0; s < n_streams; s++) {
      const rbis_synth_stream_t& ss = syn->streams[s];
      syn_o_mean[s] = put(ss.mean, (size_t)ss.rows * ss.m);
      if (ss.has_orientation) syn_o_q[s] = put(ss.mean_quat, (size_t)ss.rows * 4);
      syn_o_step[s] = put(ss.step, (size_t)ss.rows);
    }
    kp.syn.seed = syn->seed; kp.syn.first_filter = syn->first_filter;
    kp.syn.sigma_gyro = syn->sigma_gyro; kp.syn.sigma_accel = syn->sigma_accel; kp.syn.dt = syn->dt;
    for (int s = 0; s < n_streams; s++) {
      const rbis_synth_stream_t& ss = syn->streams[s];
      rbisk::SynStreamK& k = kp.syn.st[s];
      for (int a = 0; a < ss.m; a++) k.sigma[a] = ss.sigma[a];
      for (int a = 0; a < 3; a++) k.sigma_rot[a] = ss.sigma_rot[a];
      k.channel = ss.channel; k.channel_rot = ss.channel_rot;
    }
  }
  // device addresses of that block once it has a home (d = base of the uploaded copy)
  auto point_syn = [&](const double* d) {
    kp.syn.imu_mean = d + syn_o_imu;
    kp.syn.imu_step = reinterpret_cast<const long long*>(d + syn_o_istep);
    for (int s = 0; s < n_streams; s++) {
      rbisk::SynStreamK& k = kp.syn.st[s];
      k.mean = d + syn_o_mean[s];
      k.mean_quat = syn->streams[s].has_orientation ? d + syn_o_q[s] : nullptr;
      k.step = reinterpret_cast<const long long*>(d + syn_o_step[s]);
    }
  };

  // records: the REC instantiations.  A host output goes through staging buffer rec_b, which holds only the DISTINCT rows the
  // call records, in ascending order: the RECORD ops are renumbered into it, and each run of consecutive rows is copied out on
  // its own, so rows the call does not record stay untouched in the caller's buffer.
  const bool rec_host = any_record && h->rec.mem == RBIS_MEM_HOST;
  const int rec_b = h->rec_toggle;
  std::vector<int64_t> rec_distinct;
  if (any_record) {
    variant |= 8;
    kp.rec.fields = h->rec.fields;
    kp.rec.k = h->rec_k;
    kp.rec.out = h->rec.out;
    kp.rec_cov_blocks = (unsigned)h->rec.cov_blocks;
    if (rec_host) {
      rec_distinct = rec_rows;
      std::sort(rec_distinct.begin(), rec_distinct.end());
      rec_distinct.erase(std::unique(rec_distinct.begin(), rec_distinct.end()), rec_distinct.end());
      for (rbisk::Op& k : kops)
        if (k.kind == RBIS_OP_RECORD) k.row = std::lower_bound(rec_distinct.begin(), rec_distinct.end(), k.row) - rec_distinct.begin();
      const size_t rec_count = rec_distinct.size() * (size_t)h->rec_k * (size_t)N;
      DevBuf& sb = h->rec_stage[rec_b];
      if (sb.cap < rec_count) {
        if (h->rec_pending[rec_b]) CUDA_TRY(cudaEventSynchronize(h->rec_copied[rec_b]));  // its last copy (and launches) are done
        if (sb.ensure(rec_count)) return fail(RBIS_ERR_ALLOC, "record staging allocation of %zu doubles failed", rec_count);
      }
      h->rec_toggle ^= 1;
      kp.rec.out = sb.p;
    }
  }
  // innovation sets: the REC instantiations with the innovation path
  for (int s = 0; s < n_streams; s++)
    if (innov_used[s]) {
      variant |= 8 | kVariantInnov;
      kp.innov[s].out = h->innov[s].out;
      kp.innov[s].rows = h->innov[s].rows;
      kp.innov[s].k = h->innov_k[s];
      kp.innov[s].fields = (int)h->innov[s].fields;
    }
  // ---- inputs: stage host arrays on the copy stream (double buffered), or use device arrays in place ----
  StagingSlot& slot = h->slots[h->slot_toggle];
  cudaStream_t cst = h->copy_stream;
  // per-row R tables are per-call input like z: always staged, so that no launch reads a table a later call overwrote
  const bool staging = (((mem == RBIS_MEM_HOST) || syn != nullptr || f32_rows) && !fuse_syn) || !rtab_host.empty();
  const bool grouped = h->n_groups > 1;
  if (staging) {
    h->slot_toggle ^= 1;
    if (grouped && slot.ring >= 0) {
      for (int g = 0; g < h->n_groups; g++) CUDA_TRY(cudaStreamWaitEvent(cst, h->gdone[slot.ring][g], 0));
    } else {
      CUDA_TRY(cudaStreamWaitEvent(cst, slot.consumed, 0));
    }
  }
  if (syn && !fuse_syn) {
    // synthesise this call's rows into the staging slot, on the copy stream (ordered after everything the main stream has
    // enqueued so far: the process-noise arrays the IMU synthesis may read)
    double* z_out[RBIS_MAX_STREAMS] = {};
    double* q_out[RBIS_MAX_STREAMS] = {};
    if (imu_rows > 0 && slot.imu.ensure((size_t)imu_rows * 6 * (size_t)N)) return fail(RBIS_ERR_ALLOC, "synth IMU buffer allocation failed");
    for (int s = 0; s < n_streams; s++) {
      const rbis_synth_stream_t& ss = syn->streams[s];
      if (ss.rows == 0) continue;
      if (slot.z[s].ensure((size_t)ss.rows * ss.m * (size_t)N)) return fail(RBIS_ERR_ALLOC, "synth buffer allocation failed");
      z_out[s] = slot.z[s].p;
      stream_copy[s].z = z_out[s];
      if (ss.has_orientation) {
        if (slot.quat[s].ensure((size_t)ss.rows * 4 * (size_t)N)) return fail(RBIS_ERR_ALLOC, "synth buffer allocation failed");
        q_out[s] = slot.quat[s].p;
        stream_copy[s].quat = q_out[s];
      }
    }
    if (!h->syn_evt) CUDA_TRY(cudaEventCreateWithFlags(&h->syn_evt, cudaEventDisableTiming));
    CUDA_TRY(cudaEventRecord(h->syn_evt, h->stream));
    CUDA_TRY(cudaStreamWaitEvent(cst, h->syn_evt, 0));
    if (int rc = synthesize_into(h, syn, slot.imu.p, z_out, q_out, cst)) return rc;
    imu = slot.imu.p;
  }
  // RBIS_MEM_F32_ROWS with host rows: one float scratch for all arrays of the call
  size_t f32_off = 0;
  if (f32_rows && mem == RBIS_MEM_HOST) {
    size_t total = imu ? (((size_t)imu_rows * 6 * (size_t)kp.imu_cols + 3) & ~(size_t)3) : 0;
    for (int s = 0; s < n_streams; s++) {
      const size_t cols = (size_t)kp.streams[s].cols;
      total += ((size_t)streams[s].rows * streams[s].m * cols + 3) & ~(size_t)3;
      if (streams[s].has_orientation) total += ((size_t)streams[s].rows * 4 * cols + 3) & ~(size_t)3;
    }
    if (slot.f32.ensure((total + 1) / 2)) return fail(RBIS_ERR_ALLOC, "device staging allocation failed");
  }
  float* const f32_base = reinterpret_cast<float*>(slot.f32.p);
  if (imu && !fuse_syn) {
    const size_t cnt = (size_t)imu_rows * 6 * (size_t)kp.imu_cols;
    if (f32_rows) { if (int rc = copy_in_f32(h, slot.imu, imu, cnt, mem, cst, f32_base, &f32_off, &kp.imu)) return rc; }
    else if (int rc = copy_in(h, slot.imu, imu, cnt, mem, cst, &kp.imu)) return rc;
  }
  for (int s = 0; s < n_streams; s++) {
    const rbis_stream_t& in = streams[s];
    rbisk::StreamDesc& d = kp.streams[s];
    if (in.rows == 0) continue;
    if (!fuse_syn && f32_rows) {
      if (int rc = copy_in_f32(h, slot.z[s], in.z, (size_t)in.rows * in.m * (size_t)d.cols, mem, cst, f32_base, &f32_off, &d.z)) return rc;
      if (in.has_orientation)
        if (int rc = copy_in_f32(h, slot.quat[s], in.quat, (size_t)in.rows * 4 * (size_t)d.cols, mem, cst, f32_base, &f32_off, &d.quat)) return rc;
    } else if (!fuse_syn) {
      if (int rc = copy_in(h, slot.z[s], in.z, (size_t)in.rows * in.m * (size_t)d.cols, mem, cst, &d.z)) return rc;
      if (in.has_orientation)
        if (int rc = copy_in(h, slot.quat[s], in.quat, (size_t)in.rows * 4 * (size_t)d.cols, mem, cst, &d.quat)) return rc;
    }
    if (in.r_mode == RBIS_R_PER_FILTER_DIAG) {
      if (int rc = copy_in(h, slot.rdiag[s], in.R, (size_t)in.m * N, mem, cst, &d.R)) return rc;
    }
  }
  if (!rtab_host.empty()) {
    if (slot.rtab.ensure(rtab_host.size())) return fail(RBIS_ERR_ALLOC, "device staging allocation of %zu doubles failed", rtab_host.size());
    if (int rc = upload_small(h, slot.rtab.p, rtab_host.data(), rtab_host.size() * sizeof(double), cst)) return rc;
    for (int s = 0; s < n_streams; s++)
      if (streams[s].r_mode == RBIS_R_PER_ROW_FULL && streams[s].rows > 0) kp.streams[s].R = slot.rtab.p + rtab_off[s];
  }
  if (staging) CUDA_TRY(cudaEventRecord(slot.copied, cst));
  const LaunchGeom geom = launch_geom(variant, h->mapping, h->lane_tpb, N, h->n_sms);
  const unsigned grid = geom.grid;
  // slots this program overwrites that a side-stream statistics pass may still be reading
  std::vector<cudaEvent_t> slot_readers;
  if (any_snapshot && !h->snap_read_pending.empty()) {
    for (int64_t i = 0; i < n_ops; i++)
      if (ops[i].kind == RBIS_OP_SNAPSHOT && h->snap_read_pending[(size_t)ops[i].row]) {
        slot_readers.push_back(h->snap_read_evt[(size_t)ops[i].row]);
        h->snap_read_pending[(size_t)ops[i].row] = 0;
      }
  }
  // a device record or innovation buffer this program writes that a side-stream statistics pass may still be reading
  if (any_record && !rec_host) take_readers(h, h->rec.out, h->rec.out + (size_t)h->rec.rows * (size_t)h->rec_k * N, slot_readers);
  for (int s = 0; s < n_streams; s++)
    if (innov_used[s]) take_readers(h, h->innov[s].out, h->innov[s].out + (size_t)h->innov[s].rows * (size_t)h->innov_k[s] * N, slot_readers);
  if (!grouped) {
    if (int rc = main_stream_work(h)) return rc;
    for (cudaEvent_t e : slot_readers) CUDA_TRY(cudaStreamWaitEvent(h->stream, e, 0));
    if (staging) CUDA_TRY(cudaStreamWaitEvent(h->stream, slot.copied, 0));
    if (rec_host && h->rec_pending[rec_b]) CUDA_TRY(cudaStreamWaitEvent(h->stream, h->rec_copied[rec_b], 0));
    // ---- op table and shared R matrices (small, pageable source: staged synchronously by the runtime) ----
    if ((size_t)n_ops > h->d_ops_cap) {
      if (h->d_ops) {
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        cudaFree(h->d_ops);
        h->d_ops = nullptr;
        h->d_ops_cap = 0;
      }
      size_t cap = (size_t)n_ops * 2;
      if (cap < 1024) cap = 1024;
      CUDA_TRY(cudaMalloc(&h->d_ops, cap * sizeof(rbisk::Op)));
      h->d_ops_cap = cap;
    }
    if (int rc = upload_small(h, h->d_ops, kops.data(), (size_t)n_ops * sizeof(rbisk::Op), h->stream)) return rc;
    if (any_shared)
      if (int rc = upload_small(h, h->d_rshared, rshared.data(), rshared.size() * sizeof(double), h->stream)) return rc;
    if (fuse_syn) {
      if (h->d_syn.cap < syn_host.size()) {
        CUDA_TRY(cudaStreamSynchronize(h->stream));  // an earlier launch may still read the old block
        if (h->d_syn.ensure(syn_host.size() * 2)) return fail(RBIS_ERR_ALLOC, "synth row buffer allocation failed");
      }
      if (int rc = upload_small(h, h->d_syn.p, syn_host.data(), syn_host.size() * 8, h->stream)) return rc;
      point_syn(h->d_syn.p);
    }
    kp.ops = h->d_ops;
    kp.block_offset = 0;
    CUDA_TRY(launch_variant(variant, fuse_syn ? 1 : 0, geom, grid, h->stream, kp));
    h->launches++;
    if (staging) CUDA_TRY(cudaEventRecord(slot.consumed, h->stream));
    if (rec_host) {
      CUDA_TRY(cudaEventRecord(h->rec_launched, h->stream));
      CUDA_TRY(cudaStreamWaitEvent(h->rec_stream, h->rec_launched, 0));
    }
  } else {
    // ---- grouped launch: the program is cut into consecutive PIECES of ~piece_ops ops over the same (already staged)
    // inputs; every piece is one kernel per launch group, uploads on their own stream into the piece's ring slot.  Group g
    // of a piece starts when group g of the previous piece (or call) is done, so the partially filled last wave of CTAs of
    // one piece runs beside the next piece instead of idling most SMs; the state round trip through HBM per piece is
    // ~2 KB per filter, noise against a hundred ops of work.
    const int64_t piece_ops = h->cfg.piece_ops > 0 ? h->cfg.piece_ops : 256;
    const int64_t pieces = n_ops >= 2 * piece_ops ? (n_ops + piece_ops - 1) / piece_ops : 1;
    const unsigned per = (grid + (unsigned)h->n_groups - 1) / (unsigned)h->n_groups;
    // Group g of this launch may only run ahead of the other groups of the previous launch when both launches cut the
    // ensemble into the SAME filter ranges.  The ranges are per * (filters per CTA), and the filters per CTA differ between
    // kernel variants (256 dense, 384 decoupled, ...): after a change every group waits for ALL groups of the previous launch.
    const long long part = (long long)per * geom.fpc;
    for (int64_t pc = 0; pc < pieces; pc++) {
      const int64_t o0 = n_ops * pc / pieces, o1 = n_ops * (pc + 1) / pieces, np = o1 - o0;
      const int ring = (int)(h->launch_seq % rbis_batch::kRing);
      if (h->gdone_valid[ring])   // ring slot reuse: the piece that used it (kRing pieces ago) must be done
        for (int g = 0; g < h->n_groups; g++) CUDA_TRY(cudaEventSynchronize(h->gdone[ring][g]));
      if ((size_t)np > h->d_ops_ring_cap[ring]) {
        if (h->d_ops_ring[ring]) cudaFree(h->d_ops_ring[ring]);  // idle: its last user was synchronised above
        h->d_ops_ring[ring] = nullptr;
        h->d_ops_ring_cap[ring] = 0;
        size_t cap = (size_t)np * 2;
        if (cap < 1024) cap = 1024;
        CUDA_TRY(cudaMalloc(&h->d_ops_ring[ring], cap * sizeof(rbisk::Op)));
        h->d_ops_ring_cap[ring] = cap;
      }
      if (int rc = upload_small(h, h->d_ops_ring[ring], kops.data() + o0, (size_t)np * sizeof(rbisk::Op), h->upload_stream)) return rc;
      if (any_shared) {
        if (int rc = upload_small(h, h->d_rshared_ring[ring], rshared.data(), rshared.size() * sizeof(double), h->upload_stream)) return rc;
        for (int s2 = 0; s2 < n_streams; s2++)
          if (shared_r[s2]) kp.streams[s2].R = h->d_rshared_ring[ring] + (size_t)s2 * kRShared;
      }
      if (fuse_syn) {
        // every piece carries its own copy of the noise-free rows: a ring slot is reused as soon as ITS piece is done
        if (h->d_syn_ring[ring].cap < syn_host.size() && h->d_syn_ring[ring].ensure(syn_host.size() * 2))
          return fail(RBIS_ERR_ALLOC, "synth row buffer allocation failed");
        if (int rc = upload_small(h, h->d_syn_ring[ring].p, syn_host.data(), syn_host.size() * 8, h->upload_stream)) return rc;
        point_syn(h->d_syn_ring[ring].p);
      }
      CUDA_TRY(cudaEventRecord(h->uploaded[ring], h->upload_stream));
      kp.ops = h->d_ops_ring[ring];
      kp.n_ops = np;
      const bool wait_main = h->stream_dirty;
      if (wait_main) CUDA_TRY(cudaEventRecord(h->pre_evt, h->stream));
      const bool repartitioned = h->last_ring >= 0 && h->groups_dirty && h->last_part != part;
      for (int g = 0; g < h->n_groups; g++) {
        const unsigned b0 = (unsigned)g * per, b1 = b0 + per < grid ? b0 + per : grid;
        cudaStream_t gs = h->gstream[g];
        if (repartitioned)
          for (int g2 = 0; g2 < h->n_groups; g2++) CUDA_TRY(cudaStreamWaitEvent(gs, h->gdone[h->last_ring][g2], 0));
        if (wait_main) CUDA_TRY(cudaStreamWaitEvent(gs, h->pre_evt, 0));
        if (pc == 0)
          for (cudaEvent_t e : slot_readers) CUDA_TRY(cudaStreamWaitEvent(gs, e, 0));
        if (staging && pc == 0) CUDA_TRY(cudaStreamWaitEvent(gs, slot.copied, 0));
        if (rec_host && pc == 0 && h->rec_pending[rec_b]) CUDA_TRY(cudaStreamWaitEvent(gs, h->rec_copied[rec_b], 0));
        CUDA_TRY(cudaStreamWaitEvent(gs, h->uploaded[ring], 0));
        if (b1 > b0) {
          kp.block_offset = (int)b0;
          CUDA_TRY(launch_variant(variant, fuse_syn ? 1 : 0, geom, b1 - b0, gs, kp));
          h->launches++;
        }
        CUDA_TRY(cudaEventRecord(h->gdone[ring][g], gs));
      }
      h->gdone_valid[ring] = true;
      h->last_ring = ring;
      h->last_part = part;
      h->groups_dirty = true;
      h->stream_dirty = false;
      if (staging) slot.ring = ring;   // the LAST piece that reads the staging slot marks its consumption
      if (pc + 1 < pieces) h->launch_seq++;
    }
    if (rec_host)  // every group of the last piece: the groups of earlier pieces ran before them on the same streams
      for (int g = 0; g < h->n_groups; g++) CUDA_TRY(cudaStreamWaitEvent(h->rec_stream, h->gdone[h->last_ring][g], 0));
  }
  if (rec_host) {
    const size_t row_doubles = (size_t)h->rec_k * (size_t)N;
    for (size_t a = 0; a < rec_distinct.size();) {  // one copy per run of consecutive record rows
      size_t e = a + 1;
      while (e < rec_distinct.size() && rec_distinct[e] == rec_distinct[e - 1] + 1) e++;
      CUDA_TRY(cudaMemcpyAsync(h->rec.out + (size_t)rec_distinct[a] * row_doubles, h->rec_stage[rec_b].p + a * row_doubles,
                               (e - a) * row_doubles * sizeof(double), cudaMemcpyDeviceToHost, h->rec_stream));
      a = e;
    }
    CUDA_TRY(cudaEventRecord(h->rec_copied[rec_b], h->rec_stream));
    h->rec_pending[rec_b] = true;
    h->rec_copies = true;
  }
  h->launch_seq++;
  h->snap_valid = snap_valid;
  // ---- what the launch leaves behind ----
  // A dense launch keeps exact zeros exact unless it measured omega / a or restored a slot of unknown content.
  const int before = h->decoupled;
  if (!(variant & 2)) {
    if (passive_index) h->decoupled = 0;
    else if (!restores_ok) h->decoupled = -1;
  }
  if (any_snapshot) {
    const char as_launch = ((variant & 2) || (before == 1 && !passive_index && restores_ok)) ? 1 : 0;
    for (auto& f : snap_dc)
      if (f == 2) f = as_launch;
  }
  h->snap_dc = snap_dc;
  h->last_variant = variant | (fuse_syn ? 4 : 0) | (h->mapping > 1 ? (h->mapping << 4) : 0);
  h->utime = last_utime;
  return 0;
}

}  // namespace

extern "C" {

const char* rbis_last_error(void) { return g_last_error.c_str(); }

void rbis_default_config(rbis_batch_config_t* cfg) {
  if (!cfg) return;
  cfg->g_val = 9.8;
  cfg->chi_tol = 1e-6;
  cfg->ctor_folds_chi = 1;
  cfg->renormalize_quat = 0;
  cfg->snapshot_slots = 0;
  cfg->device = 0;
  cfg->launch_groups = 0;
  cfg->dense_only = 0;
  cfg->mapping = 0;
  cfg->lane_filters_per_cta = 0;
  cfg->piece_ops = 0;
  cfg->synth_materialize = 0;
}

int rbis_batch_create(rbis_batch_t** out, int64_t n_filters, const rbis_batch_config_t* cfg) {
  if (!out) return fail(RBIS_ERR_INVALID, "out is NULL");
  *out = nullptr;
  if (n_filters <= 0) return fail(RBIS_ERR_INVALID, "n_filters must be positive");
  rbis_batch_config_t c;
  if (cfg) c = *cfg; else rbis_default_config(&c);
  if (c.snapshot_slots < 0) return fail(RBIS_ERR_INVALID, "snapshot_slots must be >= 0");
  if (c.launch_groups < 0 || c.launch_groups > rbis_batch::kMaxGroups)
    return fail(RBIS_ERR_INVALID, "launch_groups must be in [0, %d]", rbis_batch::kMaxGroups);
  if (c.mapping != 0 && c.mapping != 1 && c.mapping != 2 && c.mapping != 4 && c.mapping != 8 && c.mapping != 16)
    return fail(RBIS_ERR_INVALID, "mapping must be 0 (automatic), 1, 2, 4, 8 or 16 lanes per filter");
  if (c.piece_ops < 0 || (c.piece_ops > 0 && c.piece_ops < 8)) return fail(RBIS_ERR_INVALID, "piece_ops must be 0 (automatic) or >= 8");
  if (c.lane_filters_per_cta != 0 && c.lane_filters_per_cta != 384 && c.lane_filters_per_cta != 256 && c.lane_filters_per_cta != 128)
    return fail(RBIS_ERR_INVALID, "lane_filters_per_cta must be 0 (automatic), 384, 256 or 128");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(RBIS_ERR_CUDA, "no CUDA device available (%s); this library has no CPU path", cudaGetErrorString(e));
  }
  if (c.device < 0 || c.device >= ndev) return fail(RBIS_ERR_INVALID, "device %d out of range (%d devices)", c.device, ndev);
  CUDA_TRY(cudaSetDevice(c.device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, c.device));
  if (prop.major != 10)
    return fail(RBIS_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", c.device, prop.major, prop.minor);
  if ((int)prop.sharedMemPerBlockOptin < rbis_fused_tu_dense.smem)
    return fail(RBIS_ERR_CUDA, "device offers %zu B shared memory per block, %d needed", prop.sharedMemPerBlockOptin, rbis_fused_tu_dense.smem);

  rbis_batch* h = new (std::nothrow) rbis_batch();
  if (!h) return fail(RBIS_ERR_ALLOC, "host allocation failed");
  h->N = n_filters;
  h->cfg = c;
  h->n_sms = prop.multiProcessorCount;
  {
    const MappingChoice mc = auto_mapping(n_filters, h->n_sms);
    h->mapping = c.mapping ? c.mapping : mc.mapping;
    h->lane_tpb = c.lane_filters_per_cta ? c.lane_filters_per_cta : (c.mapping == 1 ? auto_lane_tpb(n_filters, h->n_sms) : mc.lane_tpb);
    for (const rbis_fused_tu_t* t : kTus)
      if (t->kparams_bytes != sizeof(rbisk::KParams)) { fail(RBIS_ERR_CUDA, "kernel parameter block mismatch between translation units"); rbis_batch_destroy(h); return RBIS_ERR_CUDA; }
  }
  const size_t N = (size_t)n_filters;
  auto cleanup = [&](int code) { rbis_batch_destroy(h); return code; };
#define CREATE_TRY(expr)                                                                             \
  do {                                                                                               \
    cudaError_t _e = (expr);                                                                         \
    if (_e != cudaSuccess) {                                                                         \
      fail(_e == cudaErrorMemoryAllocation ? RBIS_ERR_ALLOC : RBIS_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(_e)); \
      cudaGetLastError();                                                                            \
      return cleanup(_e == cudaErrorMemoryAllocation ? RBIS_ERR_ALLOC : RBIS_ERR_CUDA);              \
    }                                                                                                \
  } while (0)
  CREATE_TRY(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  CREATE_TRY(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
  {
    // launch groups: explicit, or automatic = 6 when the CTAs do not fill a whole number of waves (measured: 2 groups 2.12, 3: 1.92, 4: 1.89, 6: 1.865, 8: 1.88 ms per launch)
    const int dense_tpb = rbis_fused_tu_dense.threads;
    const long long ctas = (long long)((n_filters + dense_tpb - 1) / dense_tpb), sms = prop.multiProcessorCount;
    const long long ctas_dc = (long long)((n_filters + h->lane_tpb - 1) / h->lane_tpb);
    int g = c.launch_groups;
    if (g == 0) g = (h->mapping == 1 && ((ctas > sms && ctas % sms != 0) || (!c.dense_only && ctas_dc > sms && ctas_dc % sms != 0))) ? 6 : 1;
    if ((long long)g > ctas_dc) g = (int)ctas_dc;
    if ((long long)g > ctas) g = (int)ctas;
    h->n_groups = g < 1 ? 1 : g;
  }
  if (h->n_groups > 1) {
    CREATE_TRY(cudaStreamCreateWithFlags(&h->upload_stream, cudaStreamNonBlocking));
    CREATE_TRY(cudaEventCreateWithFlags(&h->pre_evt, cudaEventDisableTiming));
    for (int g = 0; g < h->n_groups; g++) CREATE_TRY(cudaStreamCreateWithFlags(&h->gstream[g], cudaStreamNonBlocking));
    for (int r = 0; r < rbis_batch::kRing; r++) {
      CREATE_TRY(cudaEventCreateWithFlags(&h->uploaded[r], cudaEventDisableTiming));
      for (int g = 0; g < h->n_groups; g++) CREATE_TRY(cudaEventCreateWithFlags(&h->gdone[r][g], cudaEventDisableTiming));
      CREATE_TRY(cudaMalloc(&h->d_rshared_ring[r], (size_t)RBIS_MAX_STREAMS * kRShared * sizeof(double)));
    }
  }
  for (auto& s : h->slots) {
    CREATE_TRY(cudaEventCreateWithFlags(&s.copied, cudaEventDisableTiming));
    CREATE_TRY(cudaEventCreateWithFlags(&s.consumed, cudaEventDisableTiming));
  }
  for (auto& t : h->tickets) CREATE_TRY(cudaEventCreateWithFlags(&t, cudaEventDisableTiming));
  for (auto& t : h->ticket_rec) CREATE_TRY(cudaEventCreateWithFlags(&t, cudaEventDisableTiming));
  CREATE_TRY(cudaStreamCreateWithFlags(&h->rec_stream, cudaStreamNonBlocking));
  CREATE_TRY(cudaEventCreateWithFlags(&h->rec_launched, cudaEventDisableTiming));
  for (auto& e : h->rec_copied) CREATE_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  CREATE_TRY(cudaMallocHost(&h->pin_base, rbis_batch::kPinSlots * rbis_batch::kPinBytes));
  for (auto& e : h->pin_evt) CREATE_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  CREATE_TRY(cudaMalloc(&h->vec, N * 21 * sizeof(double)));
  CREATE_TRY(cudaMalloc(&h->quat, N * 4 * sizeof(double)));
  CREATE_TRY(cudaMalloc(&h->P, N * rbisk::NP * sizeof(double)));
  CREATE_TRY(cudaMalloc(&h->loglik, N * sizeof(double)));
  CREATE_TRY(cudaMalloc(&h->qparams, N * 4 * sizeof(double)));
  CREATE_TRY(cudaMalloc(&h->d_rshared, (size_t)RBIS_MAX_STREAMS * kRShared * sizeof(double)));
  if (c.snapshot_slots > 0) {
    CREATE_TRY(cudaMalloc(&h->snap, (size_t)c.snapshot_slots * rbisk::SNAP_ROWS * N * sizeof(double)));
    h->snap_valid.assign((size_t)c.snapshot_slots, 0);
    h->snap_dc.assign((size_t)c.snapshot_slots, 0);
  }
  CREATE_TRY(cudaMalloc(&h->d_flag, sizeof(int)));
  CREATE_TRY(cudaFuncSetAttribute(rbisk::rbis_smooth_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, rbisk::SMOOTH_SMEM_BYTES));
  for (const rbis_fused_tu_t* t : kTus) CREATE_TRY(t->prepare());
  // default state: zeros, identity quaternion, zero covariance, zero process noise
  CREATE_TRY(cudaMemsetAsync(h->vec, 0, N * 21 * sizeof(double), h->stream));
  CREATE_TRY(cudaMemsetAsync(h->quat, 0, N * 4 * sizeof(double), h->stream));
  rbisk::fill_kernel<<<(unsigned)((N + 255) / 256), 256, 0, h->stream>>>(h->quat, 1.0, (long long)N);
  CREATE_TRY(cudaGetLastError());
  CREATE_TRY(cudaMemsetAsync(h->P, 0, N * rbisk::NP * sizeof(double), h->stream));
  CREATE_TRY(cudaMemsetAsync(h->loglik, 0, N * sizeof(double), h->stream));
  CREATE_TRY(cudaMemsetAsync(h->qparams, 0, N * 4 * sizeof(double), h->stream));
  CREATE_TRY(cudaStreamSynchronize(h->stream));
#undef CREATE_TRY
  *out = h;
  return 0;
}

int rbis_batch_destroy(rbis_batch_t* h) {
  if (!h) return 0;
  cudaSetDevice(h->cfg.device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->copy_stream) cudaStreamSynchronize(h->copy_stream);
  if (h->rec_stream) { cudaStreamSynchronize(h->rec_stream); cudaStreamDestroy(h->rec_stream); }
  if (h->rec_launched) cudaEventDestroy(h->rec_launched);
  for (auto& e : h->rec_copied)
    if (e) cudaEventDestroy(e);
  for (auto& e : h->ticket_rec)
    if (e) cudaEventDestroy(e);
  for (auto& b : h->rec_stage) b.release();
  if (h->upload_stream) { cudaStreamSynchronize(h->upload_stream); cudaStreamDestroy(h->upload_stream); }
  for (int g = 0; g < rbis_batch::kMaxGroups; g++)
    if (h->gstream[g]) { cudaStreamSynchronize(h->gstream[g]); cudaStreamDestroy(h->gstream[g]); }
  for (int r = 0; r < rbis_batch::kRing; r++) {
    if (h->uploaded[r]) cudaEventDestroy(h->uploaded[r]);
    for (int g = 0; g < rbis_batch::kMaxGroups; g++)
      if (h->gdone[r][g]) cudaEventDestroy(h->gdone[r][g]);
    cudaFree(h->d_ops_ring[r]);
    cudaFree(h->d_rshared_ring[r]);
  }
  if (h->pre_evt) cudaEventDestroy(h->pre_evt);
  if (h->syn_evt) cudaEventDestroy(h->syn_evt);
  for (auto& e : h->pin_evt)
    if (e) cudaEventDestroy(e);
  if (h->pin_base) cudaFreeHost(h->pin_base);
  cudaFree(h->vec); cudaFree(h->quat); cudaFree(h->P); cudaFree(h->loglik); cudaFree(h->qparams);
  cudaFree(h->snap); cudaFree(h->d_ops); cudaFree(h->d_rshared); cudaFree(h->d_flag); cudaFree(h->d_notch_state);
  h->notch_stage.release();
  for (auto& m : h->d_map) cudaFree(m);
  h->full_cov.release(); h->misc.release(); h->stats_async.release(); h->stats_table.release(); h->synth_small.release(); h->d_syn.release();
  for (auto& b : h->snap_stats_scratch) b.release();
  for (cudaEvent_t e : h->snap_read_evt) if (e) cudaEventDestroy(e);
  for (auto& r : h->row_readers) cudaEventDestroy(r.done);
  if (h->rec_stats_done) cudaEventDestroy(h->rec_stats_done);
  h->rec_stats_scratch.release();
  if (h->stats_stream) cudaStreamDestroy(h->stats_stream);
  for (auto& b : h->d_syn_ring) b.release();
  for (auto& s : h->slots) {
    s.imu.release(); s.f32.release(); s.rtab.release();
    for (int i = 0; i < RBIS_MAX_STREAMS; i++) { s.z[i].release(); s.quat[i].release(); s.rdiag[i].release(); }
    if (s.copied) cudaEventDestroy(s.copied);
    if (s.consumed) cudaEventDestroy(s.consumed);
  }
  for (auto& t : h->tickets)
    if (t) cudaEventDestroy(t);
  if (h->stream) cudaStreamDestroy(h->stream);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  cudaGetLastError();
  delete h;
  return 0;
}

int rbis_batch_synchronize(rbis_batch_t* h) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  CUDA_TRY(cudaStreamSynchronize(h->copy_stream));
  if (h->upload_stream) CUDA_TRY(cudaStreamSynchronize(h->upload_stream));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  CUDA_TRY(cudaStreamSynchronize(h->rec_stream));  // record copies to host memory
  if (h->stats_stream) {  // side-stream statistics (rbis_batch_stats_snapshot_enqueue): done too, their slots are free again
    CUDA_TRY(cudaStreamSynchronize(h->stats_stream));
    std::fill(h->snap_read_pending.begin(), h->snap_read_pending.end(), 0);
    for (auto& r : h->row_readers) r.pending = false;
    h->rec_stats_pending = false;
  }
  return 0;
}

int64_t rbis_batch_num_filters(const rbis_batch_t* h) { return h ? h->N : 0; }
void* rbis_batch_stream(rbis_batch_t* h) { return h ? (void*)h->stream : nullptr; }
int64_t rbis_batch_launch_count(const rbis_batch_t* h) { return h ? h->launches : 0; }
int rbis_batch_last_kernel_variant(const rbis_batch_t* h) { return h ? h->last_variant : -1; }

int rbis_batch_set_state(rbis_batch_t* h, const double* vec, const double* quat, const double* cov,
                         const double* loglik, int64_t utime, int mem) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (!vec || !quat) return fail(RBIS_ERR_INVALID, "vec and quat are required");
  if (mem != RBIS_MEM_HOST && mem != RBIS_MEM_DEVICE) return fail(RBIS_ERR_INVALID, "bad mem");
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  const size_t N = (size_t)h->N;
  const cudaMemcpyKind kind = mem == RBIS_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
  CUDA_TRY(cudaMemcpyAsync(h->vec, vec, N * 21 * sizeof(double), kind, h->stream));
  CUDA_TRY(cudaMemcpyAsync(h->quat, quat, N * 4 * sizeof(double), kind, h->stream));
  if (cov) {
    const double* src = cov;
    if (mem == RBIS_MEM_HOST) {
      if (h->full_cov.ensure(N * 441)) return fail(RBIS_ERR_ALLOC, "covariance scratch allocation failed");
      CUDA_TRY(cudaMemcpyAsync(h->full_cov.p, cov, N * 441 * sizeof(double), kind, h->stream));
      src = h->full_cov.p;
    }
    rbisk::pack_cov_kernel<<<(unsigned)((N + 127) / 128), 128, 0, h->stream>>>(src, h->P, (long long)N);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    h->decoupled = -1;
  }
  if (loglik) CUDA_TRY(cudaMemcpyAsync(h->loglik, loglik, N * sizeof(double), kind, h->stream));
  else CUDA_TRY(cudaMemsetAsync(h->loglik, 0, N * sizeof(double), h->stream));
  if (mem == RBIS_MEM_HOST) CUDA_TRY(cudaStreamSynchronize(h->stream));  // caller may reuse its buffers
  h->utime = utime;
  return 0;
}

int rbis_batch_get_state(rbis_batch_t* h, double* vec, double* quat, double* cov, double* loglik, int64_t* utime,
                         int mem) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (mem != RBIS_MEM_HOST && mem != RBIS_MEM_DEVICE) return fail(RBIS_ERR_INVALID, "bad mem");
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  const size_t N = (size_t)h->N;
  const cudaMemcpyKind kind = mem == RBIS_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  if (vec) CUDA_TRY(cudaMemcpyAsync(vec, h->vec, N * 21 * sizeof(double), kind, h->stream));
  if (quat) CUDA_TRY(cudaMemcpyAsync(quat, h->quat, N * 4 * sizeof(double), kind, h->stream));
  if (loglik) CUDA_TRY(cudaMemcpyAsync(loglik, h->loglik, N * sizeof(double), kind, h->stream));
  if (cov) {
    double* dst = cov;
    if (mem == RBIS_MEM_HOST) {
      if (h->full_cov.ensure(N * 441)) return fail(RBIS_ERR_ALLOC, "covariance scratch allocation failed");
      dst = h->full_cov.p;
    }
    rbisk::unpack_cov_kernel<<<(unsigned)((N + 127) / 128), 128, 0, h->stream>>>(h->P, dst, (long long)N);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    if (mem == RBIS_MEM_HOST) CUDA_TRY(cudaMemcpyAsync(cov, dst, N * 441 * sizeof(double), kind, h->stream));
  }
  if (utime) *utime = h->utime;
  if (mem == RBIS_MEM_HOST) CUDA_TRY(cudaStreamSynchronize(h->stream));
  return 0;
}

int rbis_batch_set_filter(rbis_batch_t* h, int64_t n, const double* vec, const double* quat, const double* cov,
                          double loglik) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (n < 0 || n >= h->N) return fail(RBIS_ERR_INVALID, "filter index out of range");
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  const size_t pitch = (size_t)h->N * sizeof(double);
  if (vec) CUDA_TRY(cudaMemcpy2DAsync(h->vec + n, pitch, vec, sizeof(double), sizeof(double), 21, cudaMemcpyHostToDevice, h->stream));
  if (quat) CUDA_TRY(cudaMemcpy2DAsync(h->quat + n, pitch, quat, sizeof(double), sizeof(double), 4, cudaMemcpyHostToDevice, h->stream));
  double packed[rbisk::NP];
  if (cov) {
    for (int j = 0; j < 21; j++)
      for (int i = 0; i <= j; i++) packed[rbisk::slot(i, j)] = cov[i + 21 * j];
    CUDA_TRY(cudaMemcpy2DAsync(h->P + n, pitch, packed, sizeof(double), sizeof(double), rbisk::NP, cudaMemcpyHostToDevice, h->stream));
    if (h->decoupled == 1) {
      // stays decoupled when the new covariance is: checked on the host, no device pass needed
      for (int j = 0; j < 21 && h->decoupled == 1; j++)
        for (int i = 0; i <= j; i++) {
          const bool blk = (j < 3) || (i >= 12 && j < 15);
          if (!(rbisk::is_act(i) && rbisk::is_act(j)) && !blk && !(packed[rbisk::slot(i, j)] == 0.0)) { h->decoupled = 0; break; }
        }
    }
  }
  CUDA_TRY(cudaMemcpyAsync(h->loglik + n, &loglik, sizeof(double), cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  return 0;
}

int rbis_batch_get_filter(rbis_batch_t* h, int64_t n, double* vec, double* quat, double* cov, double* loglik) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (n < 0 || n >= h->N) return fail(RBIS_ERR_INVALID, "filter index out of range");
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  const size_t pitch = (size_t)h->N * sizeof(double);
  double packed[rbisk::NP];
  if (vec) CUDA_TRY(cudaMemcpy2DAsync(vec, sizeof(double), h->vec + n, pitch, sizeof(double), 21, cudaMemcpyDeviceToHost, h->stream));
  if (quat) CUDA_TRY(cudaMemcpy2DAsync(quat, sizeof(double), h->quat + n, pitch, sizeof(double), 4, cudaMemcpyDeviceToHost, h->stream));
  if (cov) CUDA_TRY(cudaMemcpy2DAsync(packed, sizeof(double), h->P + n, pitch, sizeof(double), rbisk::NP, cudaMemcpyDeviceToHost, h->stream));
  if (loglik) CUDA_TRY(cudaMemcpyAsync(loglik, h->loglik + n, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  if (cov)
    for (int j = 0; j < 21; j++)
      for (int i = 0; i < 21; i++) cov[i + 21 * j] = packed[rbisk::slot(i, j)];
  return 0;
}

int rbis_batch_set_process_noise(rbis_batch_t* h, double q_gyro, double q_accel, double q_gyro_bias,
                                 double q_accel_bias) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  const long long N = h->N;
  const double q[4] = {q_gyro, q_accel, q_gyro_bias, q_accel_bias};
  for (int k = 0; k < 4; k++) {
    rbisk::fill_kernel<<<(unsigned)((N + 255) / 256), 256, 0, h->stream>>>(h->qparams + k * N, q[k], N);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
  }
  return 0;
}

int rbis_batch_set_process_noise_per_filter(rbis_batch_t* h, const double* q_gyro, const double* q_accel,
                                            const double* q_gyro_bias, const double* q_accel_bias, int mem) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (!q_gyro || !q_accel || !q_gyro_bias || !q_accel_bias) return fail(RBIS_ERR_INVALID, "all four arrays are required");
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  const size_t N = (size_t)h->N;
  const cudaMemcpyKind kind = mem == RBIS_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
  const double* src[4] = {q_gyro, q_accel, q_gyro_bias, q_accel_bias};
  for (int k = 0; k < 4; k++) CUDA_TRY(cudaMemcpyAsync(h->qparams + k * N, src[k], N * sizeof(double), kind, h->stream));
  if (mem == RBIS_MEM_HOST) CUDA_TRY(cudaStreamSynchronize(h->stream));
  return 0;
}

int rbis_batch_set_column_map(rbis_batch_t* h, int which, const int32_t* map, int64_t cols) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (which < -1 || which >= RBIS_MAX_STREAMS) return fail(RBIS_ERR_INVALID, "which must be -1 (IMU) or a stream number");
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  const int k = which + 1;
  CUDA_TRY(cudaStreamSynchronize(h->stream));  // no launch may still read the old map
  if (!map) {
    cudaFree(h->d_map[k]);
    h->d_map[k] = nullptr;
    h->map_cols[k] = 0;
    return 0;
  }
  if (cols <= 0) return fail(RBIS_ERR_INVALID, "cols must be positive");
  for (int64_t n = 0; n < h->N; n++)
    if (map[n] < 0 || map[n] >= cols) return fail(RBIS_ERR_INVALID, "map[%lld] = %d is outside [0, %lld)", (long long)n, map[n], (long long)cols);
  if (!h->d_map[k]) CUDA_TRY(cudaMalloc(&h->d_map[k], (size_t)h->N * sizeof(int)));
  CUDA_TRY(cudaMemcpy(h->d_map[k], map, (size_t)h->N * sizeof(int), cudaMemcpyHostToDevice));
  h->map_cols[k] = cols;
  return 0;
}

int rbis_batch_set_record(rbis_batch_t* h, const rbis_record_t* rec) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (!rec) {
    h->rec_set = false;
    return 0;
  }
  if ((rec->fields >> rbisk::REC_FIELDS) != 0)
    return fail(RBIS_ERR_INVALID, "record fields 0x%llx: bits 0..%d only", (unsigned long long)rec->fields, rbisk::REC_FIELDS - 1);
  if ((unsigned)rec->cov_blocks >> rbisk::REC_BLOCKS)
    return fail(RBIS_ERR_INVALID, "record cov_blocks 0x%x: bits 0..%d only", (unsigned)rec->cov_blocks, rbisk::REC_BLOCKS - 1);
  if (rec->fields == 0 && rec->cov_blocks == 0) return fail(RBIS_ERR_INVALID, "record set is empty: no fields and no covariance blocks");
  if (!rec->out) return fail(RBIS_ERR_INVALID, "record output is NULL");
  if (rec->rows <= 0) return fail(RBIS_ERR_INVALID, "record rows must be positive");
  if (rec->mem != RBIS_MEM_HOST && rec->mem != RBIS_MEM_DEVICE) return fail(RBIS_ERR_INVALID, "record mem must be RBIS_MEM_HOST or RBIS_MEM_DEVICE");
  if (int rc = use_device(h)) return rc;
  cudaPointerAttributes a;
  cudaError_t e = cudaPointerGetAttributes(&a, rec->out);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(RBIS_ERR_INVALID, "record output: cudaPointerGetAttributes failed: %s", cudaGetErrorString(e));
  }
  if (rec->mem == RBIS_MEM_HOST && a.type != cudaMemoryTypeHost)
    return fail(RBIS_ERR_INVALID, "a host record output must be pinned (page-locked) memory: a copy into pageable memory would synchronise");
  if (rec->mem == RBIS_MEM_DEVICE && ((a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != h->cfg.device))
    return fail(RBIS_ERR_INVALID, "record output is not memory of device %d", h->cfg.device);
  h->rec = *rec;
  const int nb = 3 * __builtin_popcount((unsigned)rec->cov_blocks);
  h->rec_k = __builtin_popcountll(rec->fields) + nb * (nb + 1) / 2;
  h->rec_set = true;
  return 0;
}

int rbis_batch_set_innovations(rbis_batch_t* h, int32_t stream, const rbis_innovation_t* spec) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (stream < 0 || stream >= RBIS_MAX_STREAMS) return fail(RBIS_ERR_INVALID, "stream slot %d outside 0..%d", stream, RBIS_MAX_STREAMS - 1);
  if (!spec) {
    h->innov_set[stream] = false;
    return 0;
  }
  constexpr uint32_t values = RBIS_INNOV_NIS | RBIS_INNOV_Y | RBIS_INNOV_S_DIAG;
  if (!(spec->fields & values) || (spec->fields & ~(values | RBIS_INNOV_APPLIED)))
    return fail(RBIS_ERR_INVALID, "innovation fields 0x%x: a non-empty set of RBIS_INNOV_NIS / _Y / _S_DIAG, optionally with RBIS_INNOV_APPLIED",
                spec->fields);
  if (spec->m < 1 || spec->m > RBIS_MAX_MEAS) return fail(RBIS_ERR_INVALID, "innovation m = %d outside 1..%d", spec->m, RBIS_MAX_MEAS);
  if (!spec->out) return fail(RBIS_ERR_INVALID, "innovation output is NULL");
  if (spec->rows <= 0) return fail(RBIS_ERR_INVALID, "innovation rows must be positive");
  if (int rc = use_device(h)) return rc;
  cudaPointerAttributes a;
  cudaError_t e = cudaPointerGetAttributes(&a, spec->out);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(RBIS_ERR_INVALID, "innovation output: cudaPointerGetAttributes failed: %s", cudaGetErrorString(e));
  }
  if ((a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != h->cfg.device)
    return fail(RBIS_ERR_INVALID, "innovation output is not memory of device %d", h->cfg.device);
  h->innov[stream] = *spec;
  h->innov_k[stream] = ((spec->fields & RBIS_INNOV_NIS) ? 1 : 0) + ((spec->fields & RBIS_INNOV_Y) ? spec->m : 0) +
                       ((spec->fields & RBIS_INNOV_S_DIAG) ? spec->m : 0) + ((spec->fields & RBIS_INNOV_APPLIED) ? 1 : 0);
  h->innov_set[stream] = true;
  return 0;
}

int rbis_batch_set_nis_gate(rbis_batch_t* h, int32_t stream, const rbis_nis_gate_t* gate) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (stream < 0 || stream >= RBIS_MAX_STREAMS) return fail(RBIS_ERR_INVALID, "stream slot %d outside 0..%d", stream, RBIS_MAX_STREAMS - 1);
  if (!gate) {
    h->gate_set[stream] = false;
    return 0;
  }
  if (!gate->nis_max_per_filter) {
    if (!(gate->nis_max > 0)) return fail(RBIS_ERR_INVALID, "NIS gate threshold %g: must be > 0 (+inf allowed)", gate->nis_max);
  } else {
    if (int rc = use_device(h)) return rc;
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, gate->nis_max_per_filter);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(RBIS_ERR_INVALID, "per-filter NIS thresholds: cudaPointerGetAttributes failed: %s", cudaGetErrorString(e));
    }
    if ((a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != h->cfg.device)
      return fail(RBIS_ERR_INVALID, "per-filter NIS thresholds are not memory of device %d", h->cfg.device);
  }
  h->gate[stream] = *gate;
  h->gate_set[stream] = true;
  return 0;
}

int rbis_batch_run_fused(rbis_batch_t* h, int64_t n_ops, const rbis_op_t* ops, const double* imu, int64_t imu_rows,
                         int n_streams, const rbis_stream_t* streams, int mem) {
  if (n_streams > 0 && !streams) return fail(RBIS_ERR_INVALID, "streams is NULL");
  return launch_fused(h, n_ops, ops, imu, imu_rows, n_streams, streams, mem);
}

// Enqueue the synthesis kernels on the main stream: imu_out [imu_rows][6][N], z_out[s] [rows][m][N], quat_out[s] [rows][4][N]
// are DEVICE arrays.
__attribute__((visibility("hidden"))) int synthesize_into(rbis_batch_t* h, const rbis_synth_t* syn, double* imu_out, double* const* z_out, double* const* quat_out, cudaStream_t stream) {
  if (!syn) return fail(RBIS_ERR_INVALID, "syn is NULL");
  if (syn->mode != 0 && syn->mode != 1) return fail(RBIS_ERR_INVALID, "synth mode must be 0 (exact) or 1 (fast)");
  if (syn->n_streams < 0 || syn->n_streams > RBIS_MAX_STREAMS || (syn->n_streams > 0 && !syn->streams)) return fail(RBIS_ERR_INVALID, "bad synth streams");
  if (syn->imu_rows < 0 || (syn->imu_rows > 0 && (!syn->imu_mean || !syn->imu_step || !imu_out))) return fail(RBIS_ERR_INVALID, "bad synth IMU description");
  if ((syn->sigma_gyro < 0 || syn->sigma_accel < 0) && !(syn->dt > 0)) return fail(RBIS_ERR_INVALID, "per-filter IMU noise needs dt > 0");
  const long long N = h->N;
  // one small host block -> device: [imu_mean | imu_step | per stream: mean, mean_quat, step]
  size_t words = (size_t)syn->imu_rows * 7;
  for (int s = 0; s < syn->n_streams; s++) {
    const rbis_synth_stream_t& st = syn->streams[s];
    if (st.m < 1 || st.m > RBIS_MAX_MEAS || st.rows < 0) return fail(RBIS_ERR_INVALID, "synth stream %d: bad m / rows", s);
    if (st.rows > 0 && (!st.mean || !st.step || !z_out || !z_out[s])) return fail(RBIS_ERR_INVALID, "synth stream %d: mean, step and an output array are required", s);
    if (st.has_orientation && st.rows > 0 && (!st.mean_quat || !quat_out || !quat_out[s])) return fail(RBIS_ERR_INVALID, "synth stream %d: mean_quat and a quaternion output are required", s);
    words += (size_t)st.rows * (st.m + 1 + (st.has_orientation ? 4 : 0));
  }
  if (words == 0) return 0;
  std::vector<double> host(words);
  size_t off = 0;
  auto put = [&](const void* src, size_t n_words) { std::memcpy(host.data() + off, src, n_words * 8); off += n_words; return off - n_words; };
  const size_t o_imu = put(syn->imu_mean, (size_t)syn->imu_rows * 6), o_istep = put(syn->imu_step, (size_t)syn->imu_rows);
  size_t o_mean[RBIS_MAX_STREAMS] = {}, o_q[RBIS_MAX_STREAMS] = {}, o_step[RBIS_MAX_STREAMS] = {};
  for (int s = 0; s < syn->n_streams; s++) {
    const rbis_synth_stream_t& st = syn->streams[s];
    o_mean[s] = put(st.mean, (size_t)st.rows * st.m);
    if (st.has_orientation) o_q[s] = put(st.mean_quat, (size_t)st.rows * 4);
    o_step[s] = put(st.step, (size_t)st.rows);
  }
  // the previous call's kernels may still read the small block: it is rewritten on the same stream, after them
  if (h->synth_small.cap < words) CUDA_TRY(cudaStreamSynchronize(stream));
  if (h->synth_small.ensure(words)) return fail(RBIS_ERR_ALLOC, "synth scratch allocation failed");
  double* d = h->synth_small.p;
  if (int rc = upload_small(h, d, host.data(), words * 8, stream)) return rc;
  const unsigned gx = (unsigned)((N + 255) / 256);
  if (syn->imu_rows > 0) {
    const dim3 grid(gx, (unsigned)syn->imu_rows);
    if (syn->mode == 0)
      rbisk::synth_imu_kernel<0><<<grid, 256, 0, stream>>>(imu_out, d + o_imu, reinterpret_cast<const long long*>(d + o_istep), syn->imu_rows, N, syn->seed,
                                                              syn->first_filter, syn->sigma_gyro, syn->sigma_accel, h->qparams, h->qparams + N, syn->dt);
    else
      rbisk::synth_imu_kernel<1><<<grid, 256, 0, stream>>>(imu_out, d + o_imu, reinterpret_cast<const long long*>(d + o_istep), syn->imu_rows, N, syn->seed,
                                                              syn->first_filter, syn->sigma_gyro, syn->sigma_accel, h->qparams, h->qparams + N, syn->dt);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
  }
  for (int s = 0; s < syn->n_streams; s++) {
    const rbis_synth_stream_t& st = syn->streams[s];
    if (st.rows == 0) continue;
    rbisk::SynStreamDev sd;
    std::memset(&sd, 0, sizeof(sd));
    sd.m = st.m; sd.has_orient = st.has_orientation ? 1 : 0; sd.channel = st.channel; sd.channel_rot = st.channel_rot;
    sd.mean = d + o_mean[s]; sd.mean_quat = st.has_orientation ? d + o_q[s] : nullptr;
    sd.step = reinterpret_cast<const long long*>(d + o_step[s]);
    for (int a = 0; a < st.m; a++) sd.sigma[a] = st.sigma[a];
    for (int a = 0; a < 3; a++) sd.sigma_rot[a] = st.sigma_rot[a];
    sd.z = z_out[s]; sd.quat = st.has_orientation ? quat_out[s] : nullptr; sd.rows = st.rows;
    const dim3 grid(gx, (unsigned)st.rows);
    if (syn->mode == 0) rbisk::synth_stream_kernel<0><<<grid, 256, 0, stream>>>(sd, N, syn->seed, syn->first_filter);
    else rbisk::synth_stream_kernel<1><<<grid, 256, 0, stream>>>(sd, N, syn->seed, syn->first_filter);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
  }
  return 0;
}

int rbis_batch_synthesize(rbis_batch_t* h, const rbis_synth_t* syn, double* imu_out, double* const* z_out, double* const* quat_out) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  return synthesize_into(h, syn, imu_out, z_out, quat_out, h->stream);
}

int rbis_batch_run_fused_synth(rbis_batch_t* h, int64_t n_ops, const rbis_op_t* ops, int n_streams, const rbis_stream_t* streams,
                               const rbis_synth_t* syn) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (!syn) return fail(RBIS_ERR_INVALID, "syn is NULL");
  if (n_streams > 0 && !streams) return fail(RBIS_ERR_INVALID, "streams is NULL");
  return launch_fused(h, n_ops, ops, nullptr, 0, n_streams, streams, RBIS_MEM_DEVICE, true, syn);
}

int rbis_batch_ins_step(rbis_batch_t* h, const double* gyro, const double* accel, double dt, int64_t utime, int mem) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (!gyro || !accel) return fail(RBIS_ERR_INVALID, "gyro and accel are required");
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  // assemble one [6][N] IMU row on the device
  const size_t N = (size_t)h->N;
  if (h->misc.ensure(6 * N)) return fail(RBIS_ERR_ALLOC, "scratch allocation failed");
  const cudaMemcpyKind kind = mem == RBIS_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
  CUDA_TRY(cudaMemcpyAsync(h->misc.p, gyro, 3 * N * sizeof(double), kind, h->stream));
  CUDA_TRY(cudaMemcpyAsync(h->misc.p + 3 * N, accel, 3 * N * sizeof(double), kind, h->stream));
  rbis_op_t op;
  op.kind = RBIS_OP_IMU; op.stream = 0; op.row = 0; op.utime = utime; op.dt = dt;
  return launch_fused(h, 1, &op, h->misc.p, 1, 0, nullptr, RBIS_MEM_DEVICE, /*use_maps=*/false);
}

static int single_meas(rbis_batch_t* h, int m, const int32_t* idx, const double* z, const double* quat,
                       const double* R, int r_mode, int64_t utime, int mem, int has_orient) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (m < 1 || m > RBIS_MAX_MEAS || !idx) return fail(RBIS_ERR_INVALID, "bad m / idx");
  if (r_mode == RBIS_R_PER_ROW_FULL)
    return fail(RBIS_ERR_INVALID, "RBIS_R_PER_ROW_FULL applies to fused programs only: one update has one R (RBIS_R_SHARED_FULL)");
  rbis_stream_t st;
  std::memset(&st, 0, sizeof(st));
  st.m = m; st.has_orientation = has_orient; st.r_mode = r_mode;
  for (int a = 0; a < m; a++) st.idx[a] = idx[a];
  st.z = z; st.quat = quat; st.R = R; st.rows = 1;
  rbis_op_t op;
  op.kind = RBIS_OP_MEAS; op.stream = 0; op.row = 0; op.utime = utime; op.dt = 0;
  return launch_fused(h, 1, &op, nullptr, 0, 1, &st, mem, /*use_maps=*/false, nullptr, /*use_innov=*/false);
}

int rbis_batch_indexed_update(rbis_batch_t* h, int m, const int32_t* idx, const double* z, const double* R,
                              int r_mode, int64_t utime, int mem) {
  return single_meas(h, m, idx, z, nullptr, R, r_mode, utime, mem, 0);
}

int rbis_batch_indexed_orient_update(rbis_batch_t* h, int m, const int32_t* idx, const double* z, const double* quat,
                                     const double* R, int r_mode, int64_t utime, int mem) {
  if (!quat) return fail(RBIS_ERR_INVALID, "quat is required");
  return single_meas(h, m, idx, z, quat, R, r_mode, utime, mem, 1);
}

int rbis_batch_stats(rbis_batch_t* h, const double* truth_vec, const double* truth_quat, int per_filter, int chunk,
                     double* out_chunks, int64_t* n_chunks, double* out_per_filter, int mem) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (!truth_vec || !truth_quat || !out_chunks) return fail(RBIS_ERR_INVALID, "truth and out_chunks are required");
  if (chunk < 32 || chunk > 1024 || (chunk & (chunk - 1))) return fail(RBIS_ERR_INVALID, "chunk must be a power of two in [32,1024]");
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  const size_t N = (size_t)h->N;
  const int64_t nch = (int64_t)((N + chunk - 1) / chunk);
  // scratch: truth (25 or 25N) + per-filter [23][N] + chunks [nch][96]
  const size_t truth_n = per_filter ? 25 * N : 25;
  if (h->misc.ensure(truth_n + 23 * N + (size_t)nch * RBIS_NUM_STATS)) return fail(RBIS_ERR_ALLOC, "scratch allocation failed");
  double* d_truth = h->misc.p;
  double* d_pf = d_truth + truth_n;
  double* d_chunks = d_pf + 23 * N;
  const double *tv = d_truth, *tq = d_truth + (per_filter ? 21 * N : 21);
  if (per_filter && mem == RBIS_MEM_DEVICE) {
    tv = truth_vec; tq = truth_quat;
  } else {
    const size_t nv = per_filter ? 21 * N : 21, nq = per_filter ? 4 * N : 4;
    CUDA_TRY(cudaMemcpyAsync(d_truth, truth_vec, nv * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(cudaMemcpyAsync(d_truth + nv, truth_quat, nq * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  }
  double* pf = d_pf;
  if (out_per_filter && mem == RBIS_MEM_DEVICE) pf = out_per_filter;
  rbisk::stats_kernel<<<(unsigned)nch, chunk, chunk * sizeof(double), h->stream>>>(
      rbisk::StatsArrays{h->vec, h->quat, h->P, h->loglik}, tv, tq, per_filter, (long long)N, pf, d_chunks);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  CUDA_TRY(cudaMemcpyAsync(out_chunks, d_chunks, (size_t)nch * RBIS_NUM_STATS * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (out_per_filter && mem == RBIS_MEM_HOST)
    CUDA_TRY(cudaMemcpyAsync(out_per_filter, d_pf, 23 * N * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  if (n_chunks) *n_chunks = nch;
  return 0;
}

int rbis_batch_stats_enqueue(rbis_batch_t* h, const double* truth_vec, const double* truth_quat, int chunk,
                             double* out_chunks, int64_t* n_chunks) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (!truth_vec || !truth_quat || !out_chunks) return fail(RBIS_ERR_INVALID, "truth and out_chunks are required");
  if (chunk < 32 || chunk > 1024 || (chunk & (chunk - 1))) return fail(RBIS_ERR_INVALID, "chunk must be a power of two in [32,1024]");
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  const size_t N = (size_t)h->N;
  const int64_t nch = (int64_t)((N + chunk - 1) / chunk);
  // separate scratch from rbis_batch_stats so that a pending enqueue is never disturbed by a resize
  if (h->stats_async.ensure(25 + (size_t)nch * RBIS_NUM_STATS)) return fail(RBIS_ERR_ALLOC, "scratch allocation failed");
  double* d_truth = h->stats_async.p;
  double* d_chunks = d_truth + 25;
  double tbuf[25];
  std::memcpy(tbuf, truth_vec, 21 * sizeof(double));
  std::memcpy(tbuf + 21, truth_quat, 4 * sizeof(double));
  if (int rc = upload_small(h, d_truth, tbuf, sizeof(tbuf), h->stream)) return rc;  // pinned ring: the host does not wait for the stream
  rbisk::stats_kernel<<<(unsigned)nch, chunk, chunk * sizeof(double), h->stream>>>(
      rbisk::StatsArrays{h->vec, h->quat, h->P, h->loglik}, d_truth, d_truth + 21, 0, (long long)N, nullptr, d_chunks);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  CUDA_TRY(cudaMemcpyAsync(out_chunks, d_chunks, (size_t)nch * RBIS_NUM_STATS * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (n_chunks) *n_chunks = nch;
  return 0;
}

int rbis_batch_stats_snapshot_enqueue(rbis_batch_t* h, int32_t slot, const double* truth_vec, const double* truth_quat, int chunk,
                                      double* out_chunks, int64_t* n_chunks, int32_t* ticket) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (!truth_vec || !truth_quat || !out_chunks || !ticket) return fail(RBIS_ERR_INVALID, "truth, out_chunks and ticket are required");
  if (chunk < 32 || chunk > 1024 || (chunk & (chunk - 1))) return fail(RBIS_ERR_INVALID, "chunk must be a power of two in [32,1024]");
  const int S = h->cfg.snapshot_slots;
  if (slot < 0 || slot >= S) return fail(RBIS_ERR_INVALID, "snapshot slot %d out of range (%d slots)", slot, S);
  if (!h->snap_valid[(size_t)slot]) return fail(RBIS_ERR_STATE, "snapshot slot %d is empty", slot);
  if (int rc = use_device(h)) return rc;
  if (!h->stats_stream) {
    CUDA_TRY(cudaStreamCreateWithFlags(&h->stats_stream, cudaStreamNonBlocking));
    h->snap_read_evt.assign((size_t)S, nullptr);
    h->snap_read_pending.assign((size_t)S, 0);
    h->snap_stats_scratch.resize((size_t)S);
  }
  if (!h->snap_read_evt[(size_t)slot]) CUDA_TRY(cudaEventCreateWithFlags(&h->snap_read_evt[(size_t)slot], cudaEventDisableTiming));
  const size_t N = (size_t)h->N;
  const int64_t nch = (int64_t)((N + chunk - 1) / chunk);
  cudaStream_t ss = h->stats_stream;
  // after whatever wrote the slot: the group streams of the last fused launch, or the main stream; the main stream is NOT
  // made to join anything, so the fused launches that follow keep overlapping the ones before
  if (h->groups_dirty) {
    for (int g = 0; g < h->n_groups; g++) CUDA_TRY(cudaStreamWaitEvent(ss, h->gdone[h->last_ring][g], 0));
  }
  if (!h->syn_evt) CUDA_TRY(cudaEventCreateWithFlags(&h->syn_evt, cudaEventDisableTiming));
  CUDA_TRY(cudaEventRecord(h->syn_evt, h->stream));
  CUDA_TRY(cudaStreamWaitEvent(ss, h->syn_evt, 0));
  DevBuf& scratch = h->snap_stats_scratch[(size_t)slot];
  if (scratch.cap < 25 + (size_t)nch * RBIS_NUM_STATS) {
    if (h->snap_read_pending[(size_t)slot]) CUDA_TRY(cudaEventSynchronize(h->snap_read_evt[(size_t)slot]));
    if (scratch.ensure(25 + (size_t)nch * RBIS_NUM_STATS)) return fail(RBIS_ERR_ALLOC, "scratch allocation failed");
  }
  double* d_truth = scratch.p;
  double* d_chunks = d_truth + 25;
  double tbuf[25];
  std::memcpy(tbuf, truth_vec, 21 * sizeof(double));
  std::memcpy(tbuf + 21, truth_quat, 4 * sizeof(double));
  if (int rc = upload_small(h, d_truth, tbuf, sizeof(tbuf), ss)) return rc;
  const double* d = h->snap + (size_t)slot * rbisk::SNAP_ROWS * N;  // [257][N]: vec 0..20, quat 21..24, loglik 25, packed covariance 26..
  rbisk::stats_kernel<<<(unsigned)nch, chunk, chunk * sizeof(double), ss>>>(rbisk::StatsArrays{d, d + 21 * N, d + 26 * N, d + 25 * N}, d_truth, d_truth + 21, 0,
                                                                            (long long)N, nullptr, d_chunks);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  CUDA_TRY(cudaMemcpyAsync(out_chunks, d_chunks, (size_t)nch * RBIS_NUM_STATS * sizeof(double), cudaMemcpyDeviceToHost, ss));
  CUDA_TRY(cudaEventRecord(h->snap_read_evt[(size_t)slot], ss));
  h->snap_read_pending[(size_t)slot] = 1;
  const int t = h->next_ticket;
  h->next_ticket = (t + 1) % 8;
  CUDA_TRY(cudaEventRecord(h->tickets[t], ss));
  *ticket = t;
  if (n_chunks) *n_chunks = nch;
  return 0;
}

int rbis_batch_stats_records_enqueue(rbis_batch_t* h, int64_t first_row, int64_t n_rows, const double* truth_vec,
                                     const double* truth_quat, int chunk, double* out_chunks, double* out_totals, int64_t* n_chunks,
                                     int32_t* ticket) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (!truth_vec || !truth_quat || !out_chunks || !ticket) return fail(RBIS_ERR_INVALID, "truth, out_chunks and ticket are required");
  if (chunk < 32 || chunk > 1024 || (chunk & (chunk - 1))) return fail(RBIS_ERR_INVALID, "chunk must be a power of two in [32,1024]");
  if (!h->rec_set) return fail(RBIS_ERR_STATE, "no record set (rbis_batch_set_record)");
  const rbis_record_t& rec = h->rec;
  if (rec.mem != RBIS_MEM_DEVICE) return fail(RBIS_ERR_INVALID, "statistics of record rows need a record set in device memory");
  if ((rec.fields & 0x3FFFFFFull) != 0x3FFFFFFull) return fail(RBIS_ERR_INVALID, "statistics of record rows need record fields 0..25 (vec, quat, loglik)");
  if ((rec.cov_blocks & 0xE) != 0xE) return fail(RBIS_ERR_INVALID, "statistics of record rows need covariance blocks 1, 2 and 3 (v, chi, p)");
  if (n_rows < 1 || first_row < 0 || first_row + n_rows > rec.rows)
    return fail(RBIS_ERR_INVALID, "record rows %lld..%lld outside [0, %lld)", (long long)first_row, (long long)(first_row + n_rows), (long long)rec.rows);
  const size_t N = (size_t)h->N, k = (size_t)h->rec_k;
  // uploaded first: truth vec [n_rows][21] | truth quat [n_rows][4]
  std::vector<double> tbuf((size_t)n_rows * 25);
  std::memcpy(tbuf.data(), truth_vec, (size_t)n_rows * 21 * sizeof(double));
  std::memcpy(tbuf.data() + (size_t)n_rows * 21, truth_quat, (size_t)n_rows * 4 * sizeof(double));
  rbisk::StatsRecords src{};
  src.k = (long long)k;
  src.kf = __builtin_popcountll(rec.fields);
  src.base = (rec.cov_blocks & 1) ? 3 : 0;
  return row_stats_pass(h, rec.out, rec.out + (size_t)rec.rows * k * N, n_rows, chunk, tbuf, out_chunks, out_totals, n_chunks, ticket,
                        [&](cudaStream_t ss, const double* d_pre, double* d_tables, int64_t r0, int64_t ny, int64_t nch) {
                          const double* d_tvec = d_pre;
                          const double* d_tquat = d_pre + (size_t)n_rows * 21;
                          src.rows = rec.out + (size_t)(first_row + r0) * k * N;
                          rbisk::stats_kernel<<<dim3((unsigned)nch, (unsigned)ny), chunk, chunk * sizeof(double), ss>>>(
                              src, d_tvec + r0 * 21, d_tquat + r0 * 4, 0, (long long)N, nullptr, d_tables);
                        });
}

int rbis_batch_stats_innovations_enqueue(rbis_batch_t* h, int32_t stream, int64_t first_row, int64_t n_rows, int chunk,
                                         double* out_chunks, double* out_totals, int64_t* n_chunks, int32_t* ticket) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (!out_chunks || !ticket) return fail(RBIS_ERR_INVALID, "out_chunks and ticket are required");
  if (chunk < 32 || chunk > 1024 || (chunk & (chunk - 1))) return fail(RBIS_ERR_INVALID, "chunk must be a power of two in [32,1024]");
  if (stream < 0 || stream >= RBIS_MAX_STREAMS) return fail(RBIS_ERR_INVALID, "stream slot %d outside 0..%d", stream, RBIS_MAX_STREAMS - 1);
  if (!h->innov_set[stream]) return fail(RBIS_ERR_STATE, "no innovation set on stream slot %d (rbis_batch_set_innovations)", stream);
  const rbis_innovation_t& iv = h->innov[stream];
  if (!(iv.fields & RBIS_INNOV_NIS)) return fail(RBIS_ERR_INVALID, "statistics of innovation rows need the RBIS_INNOV_NIS field");
  if (n_rows < 1 || first_row < 0 || first_row + n_rows > iv.rows)
    return fail(RBIS_ERR_INVALID, "innovation rows %lld..%lld outside [0, %lld)", (long long)first_row, (long long)(first_row + n_rows), (long long)iv.rows);
  const size_t N = (size_t)h->N, k = (size_t)h->innov_k[stream];
  return row_stats_pass(h, iv.out, iv.out + (size_t)iv.rows * k * N, n_rows, chunk, std::vector<double>(), out_chunks, out_totals, n_chunks,
                        ticket, [&](cudaStream_t ss, const double*, double* d_tables, int64_t r0, int64_t ny, int64_t nch) {
                          rbisk::innov_stats_kernel<<<dim3((unsigned)nch, (unsigned)ny), chunk, chunk * sizeof(double), ss>>>(
                              iv.out + (size_t)(first_row + r0) * k * N, (long long)k, iv.m, (int)iv.fields, (long long)N, d_tables);
                        });
}

// NCCL is taken from the calling process at run time (dlsym): a host that passes an ncclComm_t has NCCL loaded already, and the
// communicator must belong to that very library; librbis_b200.so itself carries no NCCL dependency.
typedef int (*nccl_allreduce_fn)(const void*, void*, size_t, int /*ncclDataType_t*/, int /*ncclRedOp_t*/, void* /*ncclComm_t*/, cudaStream_t);
static nccl_allreduce_fn resolve_nccl_allreduce() {
  static nccl_allreduce_fn fn = nullptr;
  if (fn) return fn;
  void* sym = dlsym(RTLD_DEFAULT, "ncclAllReduce");
  if (!sym) {
    for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
      if (void* lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL | RTLD_NOLOAD)) { sym = dlsym(lib, "ncclAllReduce"); if (sym) break; }
    }
  }
  fn = reinterpret_cast<nccl_allreduce_fn>(sym);
  return fn;
}

int rbis_batch_stats_allreduce(rbis_batch_t* h, void* nccl_comm, const double* truth_vec, const double* truth_quat, int chunk,
                               int64_t first_chunk, int64_t total_chunks, double* out_totals, double* out_table) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (!truth_vec || !truth_quat || !out_totals) return fail(RBIS_ERR_INVALID, "truth and out_totals are required");
  if (chunk < 32 || chunk > 1024 || (chunk & (chunk - 1))) return fail(RBIS_ERR_INVALID, "chunk must be a power of two in [32,1024]");
  const size_t N = (size_t)h->N;
  const int64_t nch = (int64_t)((N + chunk - 1) / chunk);
  if (first_chunk < 0 || total_chunks < 1 || first_chunk + nch > total_chunks)
    return fail(RBIS_ERR_INVALID, "chunks %lld..%lld of this shard do not fit a table of %lld chunks", (long long)first_chunk,
                (long long)(first_chunk + nch), (long long)total_chunks);
  nccl_allreduce_fn allreduce = nullptr;
  if (nccl_comm) {
    allreduce = resolve_nccl_allreduce();
    if (!allreduce) return fail(RBIS_ERR_STATE, "an NCCL communicator was passed but no NCCL library is loaded in this process (ncclAllReduce not found)");
  }
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  // device-resident: truth [25] | table [total_chunks][96] | totals [96]
  const size_t n_table = (size_t)total_chunks * RBIS_NUM_STATS;
  if (h->stats_table.ensure(32 + n_table + RBIS_NUM_STATS)) return fail(RBIS_ERR_ALLOC, "statistics table allocation failed");
  double* d_truth = h->stats_table.p;
  double* d_table = d_truth + 32;
  double* d_totals = d_table + n_table;
  double tbuf[25];
  std::memcpy(tbuf, truth_vec, 21 * sizeof(double));
  std::memcpy(tbuf + 21, truth_quat, 4 * sizeof(double));
  if (int rc = upload_small(h, d_truth, tbuf, sizeof(tbuf), h->stream)) return rc;
  // every slot of the table has exactly one non-zero contributor (the rank that owns the chunk): the SUM all-reduce is
  // exact in any order (x + 0 = x), SURVEY.md 8e
  CUDA_TRY(cudaMemsetAsync(d_table, 0, n_table * sizeof(double), h->stream));
  rbisk::stats_kernel<<<(unsigned)nch, chunk, chunk * sizeof(double), h->stream>>>(
      rbisk::StatsArrays{h->vec, h->quat, h->P, h->loglik}, d_truth, d_truth + 21, 0, (long long)N, nullptr, d_table + (size_t)first_chunk * RBIS_NUM_STATS);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  if (allreduce) {
    const int rc = allreduce(d_table, d_table, n_table, /*ncclDouble*/ 8, /*ncclSum*/ 0, nccl_comm, h->stream);
    if (rc != 0) return fail(RBIS_ERR_CUDA, "ncclAllReduce failed with ncclResult_t %d", rc);
  }
  rbisk::reduce_chunk_table_kernel<<<1, 128, 0, h->stream>>>(d_table, (long long)total_chunks, d_totals);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  CUDA_TRY(cudaMemcpyAsync(out_totals, d_totals, RBIS_NUM_STATS * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (out_table) CUDA_TRY(cudaMemcpyAsync(out_table, d_table, n_table * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  return 0;
}

int rbis_batch_window_neg_loglik(rbis_batch_t* h, const double* truth_vec, const double* truth_quat, const double* base_cov,
                                 const int32_t* base_map, int64_t base_cols, int n_active, const int32_t* active_idx,
                                 double* out, int mem) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (!truth_vec || !truth_quat || !base_cov || !active_idx || !out) return fail(RBIS_ERR_INVALID, "null argument");
  if (mem != RBIS_MEM_HOST && mem != RBIS_MEM_DEVICE) return fail(RBIS_ERR_INVALID, "bad mem");
  if (n_active < 1 || n_active > RBIS_NUM_STATES) return fail(RBIS_ERR_INVALID, "n_active out of range");
  for (int a = 0; a < n_active; a++)
    if (active_idx[a] < 0 || active_idx[a] >= RBIS_NUM_STATES) return fail(RBIS_ERR_INVALID, "active index out of range");
  const size_t N = (size_t)h->N;
  if (!base_map) base_cols = (int64_t)N;
  if (base_cols <= 0) return fail(RBIS_ERR_INVALID, "base_cols must be positive");
  if (base_map)
    for (size_t n = 0; n < N; n++)
      if (base_map[n] < 0 || base_map[n] >= base_cols) return fail(RBIS_ERR_INVALID, "base_map entry out of range");
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  // scratch (doubles): truth 25N + base 441*cols + out N + ints (map N + active 21, packed into doubles)
  const size_t n_truth = mem == RBIS_MEM_HOST ? 25 * N : 0, n_base = mem == RBIS_MEM_HOST ? 441 * (size_t)base_cols : 0;
  const size_t n_int = (N + RBIS_NUM_STATES + 1) / 2 + 1;
  if (h->misc.ensure(n_truth + n_base + N + n_int)) return fail(RBIS_ERR_ALLOC, "scratch allocation failed");
  double* d_truth = h->misc.p;
  double* d_base = d_truth + n_truth;
  double* d_out = d_base + n_base;
  int* d_int = reinterpret_cast<int*>(d_out + N);
  const double *tv = truth_vec, *tq = truth_quat, *bc = base_cov;
  if (mem == RBIS_MEM_HOST) {
    CUDA_TRY(cudaMemcpyAsync(d_truth, truth_vec, 21 * N * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(cudaMemcpyAsync(d_truth + 21 * N, truth_quat, 4 * N * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(cudaMemcpyAsync(d_base, base_cov, n_base * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    tv = d_truth; tq = d_truth + 21 * N; bc = d_base;
  }
  CUDA_TRY(cudaMemcpyAsync(d_int, active_idx, (size_t)n_active * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  if (base_map) CUDA_TRY(cudaMemcpyAsync(d_int + RBIS_NUM_STATES, base_map, N * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  double* o = mem == RBIS_MEM_DEVICE ? out : d_out;
  rbisk::window_nll_kernel<<<(unsigned)((N + 127) / 128), 128, 0, h->stream>>>(
      h->vec, h->quat, h->P, tv, tq, bc, base_map ? d_int + RBIS_NUM_STATES : nullptr, (long long)base_cols, n_active,
      d_int, (long long)N, o);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  if (mem == RBIS_MEM_HOST) CUDA_TRY(cudaMemcpyAsync(out, d_out, N * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  return 0;
}

int rbis_batch_record(rbis_batch_t* h, int32_t* ticket) {
  if (!h || !ticket) return fail(RBIS_ERR_INVALID, "null handle or ticket");
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  const int t = h->next_ticket;
  h->next_ticket = (t + 1) % 8;
  CUDA_TRY(cudaEventRecord(h->tickets[t], h->stream));
  // the record copies enqueued so far run on their own stream, which the main stream does not join
  h->ticket_rec_valid[t] = h->rec_copies;
  if (h->rec_copies) CUDA_TRY(cudaEventRecord(h->ticket_rec[t], h->rec_stream));
  *ticket = t;
  return 0;
}

int rbis_batch_wait(rbis_batch_t* h, int32_t ticket) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (ticket < 0 || ticket >= 8) return fail(RBIS_ERR_INVALID, "bad ticket");
  if (int rc = use_device(h)) return rc;
  CUDA_TRY(cudaEventSynchronize(h->tickets[ticket]));
  if (h->ticket_rec_valid[ticket]) CUDA_TRY(cudaEventSynchronize(h->ticket_rec[ticket]));
  return 0;
}

int rbis_stats_reduce_chunks(const double* chunks, int64_t n_chunks, double* out) {
  if (!chunks || !out || n_chunks < 0) return fail(RBIS_ERR_INVALID, "bad arguments");
  for (int k = 0; k < RBIS_NUM_STATS; k++) {
    double s = 0.0;
    for (int64_t c = 0; c < n_chunks; c++) s += chunks[c * RBIS_NUM_STATS + k];  // ascending chunk order
    out[k] = s;
  }
  return 0;
}

int rbis_measure_fp64_peak(int device, int iters, double* dfma_tflops, double* dmma_tflops) {
  if (iters <= 0) return fail(RBIS_ERR_INVALID, "iters must be positive");
  CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  const int blocks = prop.multiProcessorCount * 4, threads = 256;
  double* d_out = nullptr;
  CUDA_TRY(cudaMalloc(&d_out, (size_t)blocks * threads * sizeof(double)));
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventCreate(&e1));
  float ms = 0;
  for (int which = 0; which < 2; which++) {
    double best = 0;
    for (int rep = 0; rep < 4; rep++) {  // first repetition is the warm-up
      CUDA_TRY(cudaEventRecord(e0));
      if (which == 0) rbisk::dfma_peak_kernel<<<blocks, threads>>>(d_out, iters, 1.0000001);
      else rbisk::dmma_peak_kernel<<<blocks, threads>>>(d_out, iters, 1.0000001);
      CUDA_TRY(cudaEventRecord(e1));
      CUDA_TRY(cudaEventSynchronize(e1));
      CUDA_TRY(cudaGetLastError());
      CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
      double flops;
      if (which == 0) flops = (double)blocks * threads * rbisk::DFMA_CHAINS * 2.0 * iters * rbisk::DFMA_UNROLL;
      else flops = (double)blocks * (threads / 32) * rbisk::DMMA_CHAINS * rbisk::DMMA_UNROLL * 512.0 * iters;
      const double tf = flops / (ms * 1e-3) / 1e12;
      if (rep > 0 && tf > best) best = tf;
    }
    if (which == 0 && dfma_tflops) *dfma_tflops = best;
    if (which == 1 && dmma_tflops) *dmma_tflops = best;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d_out);
  return 0;
}

int rbis_batch_smooth_backward(rbis_batch_t* h, int32_t next_pred_slot, int32_t next_slot, int64_t n_steps,
                               const rbis_smooth_step_t* steps, double dt) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (n_steps < 0 || (n_steps > 0 && !steps)) return fail(RBIS_ERR_INVALID, "bad step list");
  if (!(dt > 0)) return fail(RBIS_ERR_INVALID, "dt must be positive");
  const int S = h->cfg.snapshot_slots;
  auto ok = [&](int32_t s) { return s >= 0 && s < S && h->snap_valid[(size_t)s]; };
  if (!ok(next_pred_slot) || !ok(next_slot)) return fail(RBIS_ERR_STATE, "start slots %d / %d are out of range or empty", next_pred_slot, next_slot);
  for (int64_t i = 0; i < n_steps; i++)
    if (!ok(steps[i].cur_slot) || !ok(steps[i].cur_pred_slot) || steps[i].out_slot < 0 || steps[i].out_slot >= S)
      return fail(RBIS_ERR_STATE, "smoothing step %lld names an out-of-range or empty snapshot slot", (long long)i);
  if (n_steps == 0) return 0;
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  static_assert(sizeof(rbis_smooth_step_t) == sizeof(rbisk::SmoothStep), "step layout");
  const size_t n_dbl = ((size_t)n_steps * sizeof(rbisk::SmoothStep) + 7) / 8;
  if (h->misc.ensure(n_dbl)) return fail(RBIS_ERR_ALLOC, "scratch allocation failed");
  CUDA_TRY(cudaMemcpyAsync(h->misc.p, steps, (size_t)n_steps * sizeof(rbisk::SmoothStep), cudaMemcpyHostToDevice, h->stream));
  const unsigned grid = (unsigned)((h->N + rbisk::SMOOTH_WARPS - 1) / rbisk::SMOOTH_WARPS);
  rbisk::rbis_smooth_kernel<<<grid, rbisk::SMOOTH_WARPS * 32, rbisk::SMOOTH_SMEM_BYTES, h->stream>>>(
      h->snap, (long long)h->N, next_pred_slot, next_slot, reinterpret_cast<const rbisk::SmoothStep*>(h->misc.p), (long long)n_steps,
      dt, h->cfg.g_val, h->cfg.chi_tol, h->cfg.ctor_folds_chi);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  for (int64_t i = 0; i < n_steps; i++) {
    h->snap_valid[(size_t)steps[i].out_slot] = 1;
    h->snap_dc[(size_t)steps[i].out_slot] = 0;  // smoothed covariances carry no structural zeros
  }
  CUDA_TRY(cudaStreamSynchronize(h->stream));  // `steps` scratch and the caller's array are free again
  return 0;
}

int rbis_batch_get_snapshot(rbis_batch_t* h, int32_t slot, double* vec, double* quat, double* cov, double* loglik, int mem) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (mem != RBIS_MEM_HOST && mem != RBIS_MEM_DEVICE) return fail(RBIS_ERR_INVALID, "bad mem");
  if (slot < 0 || slot >= h->cfg.snapshot_slots) return fail(RBIS_ERR_INVALID, "snapshot slot %d out of range", slot);
  if (!h->snap_valid[(size_t)slot]) return fail(RBIS_ERR_STATE, "snapshot slot %d is empty", slot);
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  const size_t N = (size_t)h->N;
  const double* base = h->snap + (size_t)slot * rbisk::SNAP_ROWS * N;
  const cudaMemcpyKind kind = mem == RBIS_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  if (vec) CUDA_TRY(cudaMemcpyAsync(vec, base, N * 21 * sizeof(double), kind, h->stream));
  if (quat) CUDA_TRY(cudaMemcpyAsync(quat, base + 21 * N, N * 4 * sizeof(double), kind, h->stream));
  if (loglik) CUDA_TRY(cudaMemcpyAsync(loglik, base + 25 * N, N * sizeof(double), kind, h->stream));
  if (cov) {
    double* dst = cov;
    if (mem == RBIS_MEM_HOST) {
      if (h->full_cov.ensure(N * 441)) return fail(RBIS_ERR_ALLOC, "covariance scratch allocation failed");
      dst = h->full_cov.p;
    }
    rbisk::unpack_cov_kernel<<<(unsigned)((N + 127) / 128), 128, 0, h->stream>>>(base + 26 * N, dst, (long long)N);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    if (mem == RBIS_MEM_HOST) CUDA_TRY(cudaMemcpyAsync(cov, dst, N * 441 * sizeof(double), kind, h->stream));
  }
  if (mem == RBIS_MEM_HOST) CUDA_TRY(cudaStreamSynchronize(h->stream));
  return 0;
}

int rbis_batch_notch_configure(rbis_batch_t* h, double notch_freq, double fs, int n_stages, int64_t cols) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (n_stages < 1 || n_stages > rbisk::MAX_NOTCH) return fail(RBIS_ERR_INVALID, "n_stages must be in [1, %d]", rbisk::MAX_NOTCH);
  if (!(notch_freq > 0) || !(fs > 0) || cols <= 0) return fail(RBIS_ERR_INVALID, "notch_freq, fs and cols must be positive");
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  for (int i = 0; i < n_stages; i++) {
    // IIRNotch::IIRNotch + secondOrderNotch, estimate_tools/src/estimate_tools/iir_notch.cpp:3-33, with the stage
    // frequencies of InsHandler (MSE/sensor_handlers.cpp:33-41: notch_freq * 2^i)
    double Wo = (notch_freq * std::pow(2, i)) / (fs / 2);
    double BW = Wo;
    const double Ab = std::fabs(10 * std::log10(.5));
    BW = BW * M_PI;
    Wo = Wo * M_PI;
    const double Gb = std::pow(10, -Ab / 20.);
    const double beta = (std::sqrt(1.0 - Gb * Gb) / Gb) * std::tan(BW / 2.0);
    const double gain = 1 / (1 + beta);
    h->notch.b[i][0] = gain * 1.0; h->notch.b[i][1] = gain * (-2.0 * std::cos(Wo)); h->notch.b[i][2] = gain * 1;
    h->notch.a[i][0] = 1.0; h->notch.a[i][1] = -2 * gain * std::cos(Wo); h->notch.a[i][2] = 2 * gain - 1;
  }
  h->notch.n_stages = n_stages;
  cudaFree(h->d_notch_state);
  h->d_notch_state = nullptr;
  const size_t n = (size_t)3 * rbisk::MAX_NOTCH * 4 * (size_t)cols;
  CUDA_TRY(cudaMalloc(&h->d_notch_state, n * sizeof(double)));
  CUDA_TRY(cudaMemsetAsync(h->d_notch_state, 0, n * sizeof(double), h->stream));  // x = y = 0, iir_notch.cpp:10-13
  h->notch_cols = cols;
  return 0;
}

int rbis_batch_notch_filter(rbis_batch_t* h, double* imu, int64_t rows, int mem) {
  if (!h) return fail(RBIS_ERR_INVALID, "null handle");
  if (!h->d_notch_state) return fail(RBIS_ERR_STATE, "rbis_batch_notch_configure has not been called");
  if (!imu || rows < 0) return fail(RBIS_ERR_INVALID, "bad imu chunk");
  if (mem != RBIS_MEM_HOST && mem != RBIS_MEM_DEVICE) return fail(RBIS_ERR_INVALID, "bad mem");
  if (rows == 0) return 0;
  if (int rc = use_device(h)) return rc;
  if (int rc = main_stream_work(h)) return rc;
  const size_t count = (size_t)rows * 6 * (size_t)h->notch_cols;
  double* d = imu;
  if (mem == RBIS_MEM_HOST) {
    if (h->notch_stage.ensure(count)) return fail(RBIS_ERR_ALLOC, "staging allocation failed");
    d = h->notch_stage.p;
    CUDA_TRY(cudaMemcpyAsync(d, imu, count * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  }
  rbisk::notch_kernel<<<dim3((unsigned)((h->notch_cols + 127) / 128), 3), 128, 0, h->stream>>>(d, (long long)rows, (long long)h->notch_cols,
                                                                                              h->d_notch_state, h->notch);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  if (mem == RBIS_MEM_HOST) {
    CUDA_TRY(cudaMemcpyAsync(imu, d, count * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
  }
  return 0;
}

}  // extern "C"
