// rbis_kernels.cuh -- sm_100a FP64 device code of the batched RBIS EKF hot path.
//
// Mapping (see DESIGN.md 4): ONE LANE PER FILTER, one CTA per SM.  A filter's 21x21 covariance is kept symmetric-packed
// and stays on chip for the whole fused program, split over two memories that are read concurrently: SHARED MEMORY as
// Ps[slot][lane] (conflict free) and TENSOR MEMORY, of which each thread owns its lane of the warp's 32-lane quarter,
// reached with tcgen05.ld/st.32x32b.x2; fetches are software pipelined (loads of column k+1 in flight while column k is
// computed).  Each fused-kernel translation unit (rbis_fused_*.cu) compiles it in one configuration, in a namespace of its own:
//   * dense    (RBIS_TPB 256, RBIS_PLACEMENT 1): all 231 slots on chip -- 113 in shared memory (the 15x15 "active" part:
//     rows/columns of v, chi, p, b_g, b_a, touched 5.5 times per slot and step), 118 in tensor memory (everything coupled
//     to the angular-velocity / acceleration rows, touched 2-3 times per step, plus the (b_a,b_a) block); 8 warps;
//   * decoupled (RBIS_TPB 384, RBIS_PLACEMENT 2, kernels with DC = true): only the 120 active slots exist -- 75 in shared
//     memory, the 9x9 block of (p, b_g, b_a) in tensor memory; 12 warps at 168 registers, the filter state parked in
//     spare tensor memory during measurement sweeps.  See "decoupled filters" below.
// State (21+4), log-likelihood and linearisation live in registers.  Per-op inputs (IMU rows, measurement rows) are
// coalesced structure-of-arrays loads.  No cross-lane communication, no barriers: filters are independent.
//
// Reference semantics restated (paths under /root/reference/state-estimator/src/mav_state_est/):
//   cov_propagate()  = insUpdateCovariance + getIMUProcessLinearizationContinuous  rbis.cpp:12-35,77-122
//   state_propagate()= insUpdateState                                               rbis.cpp:37-75
//   meas3<I0>() / meas_general() = matrixMeasurementGetKandCovDelta + indexed[PlusOrientation]Measurement
//                      + the covariance half of rbisApplyDelta                      rbis.cpp:124-227
//   meas_finish()    = the state half of rbisApplyDelta (addState)                  rbis.cpp:219-227
// Include guard for the default configuration only: the fused-kernel translation units (rbis_fused_tu.inc) and
// dev/kvariant.cu include this file with `#define rbisk <other namespace>` and their own RBIS_TPB / RBIS_PLACEMENT.
#if defined(rbisk) || !defined(RBIS_KERNELS_CUH_DEFAULT)
#ifndef rbisk
#define RBIS_KERNELS_CUH_DEFAULT
#endif
#include <cstdint>
#include <utility>

// compiler memory fence between shared-memory column groups (bounds load hoisting)
#define RBIS_SCHED_FENCE() asm volatile("" ::: "memory")
#ifndef RBIS_LATE_LOADS
#define RBIS_LATE_LOADS 0
#endif
#ifndef RBIS_PARK_STATE
#define RBIS_PARK_STATE 0
#endif
// The filter-state arithmetic between the covariance sweeps is a serial stretch in which the FP64 pipe idles for all
// warps of a scheduler at once (they run in step), so its instruction count matters more than its share suggests.  Hence
// one reciprocal instead of three divisions in the axis of a rotation increment, a squared-norm test before chiToQuat, R
// computed once per step for R dt, q^-1 g_vec and q v, sin / cos of the (small) half angle by their series, |chi| and
// 1/|chi| from one rsqrt, and one log of the determinant as the reference writes it (rbis.cpp:142).  Each differs from
// the reference's operation order by a few ulp per step (parity tests: <= 1e-12 per step).  Measured: DESIGN.md 4.6.

namespace rbisk {

constexpr int NS = 21;       // rbis_num_states
constexpr int NP = 231;      // packed upper triangle
#ifndef RBIS_TPB
#define RBIS_TPB 256
#endif
constexpr int TPB = RBIS_TPB;     // filters (= threads) per CTA
constexpr int SWEEP_TILE = 8;  // slots per pipelined tile of the measurement covariance sweep
constexpr int MAX_MEAS = 9;
constexpr int MAX_STREAMS = 8;
constexpr int MAX_CHUNKS = 9;
constexpr int SNAP_ROWS = 257;  // 21 vec + 4 quat + loglik + 231 covariance
// shared-R buffer of a stream: R (81 doubles), rows of L_R^-1 (81), D_R (9) -- see rbis_batch.cu decorrelate_block
constexpr int RS_W = 81, RS_D = 162, RS_STRIDE = 171;

__host__ __device__ constexpr int slot(int i, int j) { return i <= j ? j * (j + 1) / 2 + i : i * (i + 1) / 2 + j; }

// ---- placement of covariance slots ----------------------------------------------------------------
// active index = row/column of v (3..5), chi (6..8), p (9..11), b_g (15..17), b_a (18..20)
__host__ __device__ constexpr bool is_act(int k) { return k >= 3 && !(k >= 12 && k < 15); }
__host__ __device__ constexpr int col_of_slot(int s) { int j = 0; while ((j + 1) * (j + 2) / 2 <= s) j++; return j; }
__host__ __device__ constexpr int row_of_slot(int s) { return s - col_of_slot(s) * (col_of_slot(s) + 1) / 2; }
#ifndef RBIS_PLACEMENT
#define RBIS_PLACEMENT 1
#endif
static_assert(RBIS_PLACEMENT >= 1 && RBIS_PLACEMENT <= 3, "RBIS_PLACEMENT is 1, 2 or 3");
// RBIS_PARK_STATE: 0 = the filter state stays in registers; 2 = everything that a phase does not need is parked in spare
// tensor memory (20 doubles during the covariance step, all 26 during a measurement sweep) -- for the 168-register budget
// of 384 filters per CTA
static_assert(RBIS_PARK_STATE == 0 || RBIS_PARK_STATE == 2, "RBIS_PARK_STATE is 0 or 2");
#define RBIS_PARK_STATE_SLOTS (RBIS_PARK_STATE == 2 ? 26 : 0)
// Which memory holds slot (i <= j):
//   placement 1: the active part (5.5 accesses per slot and step, most values used by several FMAs) in shared memory,
//                whose loads land in any register, and the passive part (2-3 accesses) in tensor memory; 113 slots fit
//                in shared memory, so the (b_a,b_a) block and (17,17) stay in TMEM.
//   placement 3 (DC kernels only, <= 128 filters per CTA): the 120 active slots, all in shared memory.
//   placement 2 (DC kernels only, 384 filters per CTA): only the 120 active slots are on chip; the 9x9 block of
//                p, b_g, b_a (45 slots, the least accessed: 1-3 loads and at most one store per step) in tensor
//                memory, the 75 slots that involve v or chi in shared memory.
__host__ __device__ constexpr bool on_chip(int i, int j) {
#if RBIS_PLACEMENT == 2 || RBIS_PLACEMENT == 3
  return is_act(i) && is_act(j);
#else
  return true;
#endif
}
__host__ __device__ constexpr bool slot_in_tm(int i, int j) {
#if RBIS_PLACEMENT == 2
  return (i >= 9 && !(i >= 12 && i < 15)) && (j >= 9 && !(j >= 12 && j < 15));
#elif RBIS_PLACEMENT == 3
  return false;  // DC kernels with <= 128 filters per CTA: all 120 active slots fit in shared memory (123 KB)
#else
  return !(is_act(i) && is_act(j)) || i >= 18 || (i == 17 && j == 17);
#endif
}
struct Placement {
  short idx[NP];  // index within its memory
  bool tm[NP];
  int n_tm, n_sm;
};
constexpr Placement make_placement() {
  Placement pl{};
  int nt = 0, ns = 0;
  for (int j = 0; j < NS; j++)
    for (int i = 0; i <= j; i++) {
      const int s_ = slot(i, j);
      pl.tm[s_] = slot_in_tm(i, j);
      if (!on_chip(i, j)) { pl.idx[s_] = -1; continue; }
      pl.idx[s_] = (short)(pl.tm[s_] ? nt++ : ns++);
    }
  pl.n_tm = nt;
  pl.n_sm = ns;
  return pl;
}
constexpr Placement kPlace = make_placement();
__constant__ Placement c_place = make_placement();  // run-time copy for the general (slow) path
// (i <= j assumed below)
__host__ __device__ constexpr bool in_tm(int i, int j) { return kPlace.tm[slot(i, j)]; }
__host__ __device__ constexpr int tm_index(int i, int j) { return kPlace.idx[slot(i, j)]; }
__host__ __device__ constexpr int sm_index(int i, int j) { return kPlace.idx[slot(i, j)]; }

constexpr int N_TM = kPlace.n_tm;   // slots in tensor memory
constexpr int N_SM = kPlace.n_sm;   // slots in shared memory
// tensor memory: 128 lanes x 512 columns; warp w reaches lanes 32*(w%4)..+31 only, so the TPB/128 warps that share a
// lane quarter split the 512 columns: TM_COLS 32-bit columns = TM_COLS/2 doubles per thread
constexpr int TM_COLS = (512 / ((TPB + 127) / 128)) & ~1;
static_assert(TPB % 32 == 0, "whole warps");
static_assert(2 * (N_TM + RBIS_PARK_STATE_SLOTS) <= TM_COLS, "tensor-memory share of a thread exceeded");
static_assert(N_SM * TPB * 8 + 64 <= 232448, "shared-memory part exceeds 227 KB per CTA");
constexpr int SMEM_BYTES = N_SM * TPB * 8;
// offset (in doubles, from the lane's base pointer) of shared slot k
__host__ __device__ constexpr int sm_off(int k) { return k * TPB; }

// ---- decoupled filters (DC kernels) ---------------------------------------------------------------
// The rows of Ad for omega (0..2) and a (12..14) are identity and its columns for them are zero, so the couplings
// P[{omega,a}, .] never feed the 15x15 active block (v, chi, p, b_g, b_a); they only evolve by left-multiplication
// (Ad, I - K H).  A filter whose couplings are exactly zero -- every filter initialised with the reference's diagonal
// covariance, MSE/rbis_initializer.cpp:85-91 -- keeps them exactly zero until a measurement indexes omega or a, and
// the (omega,omega) / (a,a) blocks are overwritten by every IMU step (rbis.cpp:120-121).  The DC kernel variants
// exploit that, verified at run time by the host (coupling_check_kernel): they keep only the 120 active slots on
// chip and touch nothing else; results are bit-identical to the dense variants.
constexpr int N_ACT = 15;
constexpr int NP_ACT = N_ACT * (N_ACT + 1) / 2;
__host__ __device__ constexpr int act_col(int k) { return k < 9 ? 3 + k : 6 + k; }   // k-th active index
__host__ __device__ constexpr int act_pos(int c) { return c < 12 ? c - 3 : c - 6; }  // inverse
struct ActSlots {
  short s[NP_ACT];   // packed slots with both indices active, ascending
  short rest[NP - NP_ACT - 12];  // passive couplings (everything else except the (omega,omega) and (a,a) blocks)
  short blk[12];     // (omega,omega) then (a,a) blocks, upper triangles column by column
};
constexpr ActSlots make_act_slots() {
  ActSlots a{};
  int na = 0, nr = 0, nb = 0;
  for (int j = 0; j < NS; j++)
    for (int i = 0; i <= j; i++) {
      const bool blk = (j < 3) || (i >= 12 && j < 15);
      if (is_act(i) && is_act(j)) a.s[na++] = (short)slot(i, j);
      else if (blk) a.blk[nb++] = (short)slot(i, j);
      else a.rest[nr++] = (short)slot(i, j);
    }
  return a;
}
constexpr ActSlots kAct = make_act_slots();
__constant__ ActSlots c_act = make_act_slots();  // run-time indexable copy
constexpr int N_REST = NP - NP_ACT - 12;

struct StreamDesc {
  int m, has_orient, r_mode, n_chunks;
  int idx[MAX_MEAS];
  int chunk_start[MAX_CHUNKS];
  int chunk_len[MAX_CHUNKS];
  int chunk_fast[MAX_CHUNKS];  // >= 0: the chunk is the aligned index triple I0..I0+2 (I0 = chunk_fast) -> meas3<I0>
  const double* z;     // [rows][m][cols]
  const double* quat;  // [rows][4][cols]
  const double* R;     // r_mode 0: device copy of m*m column-major (+ RS_W / RS_D); 1: [m][N]; 2: one such table per row
  const int* map;      // column of z / quat read by filter n (nullptr: column n)
  long long cols;      // columns of z / quat (N without a map)
  long long r_stride;  // r_mode 2: doubles from the table of row r to that of row r + 1; 0 otherwise (every row reads R)
};

struct Op {
  int kind, stream;
  long long row;
  double dt;
};
// Op::kind: the values of RBIS_OP_IMU, RBIS_OP_MEAS, RBIS_OP_SNAPSHOT and RBIS_OP_RECORD (checked in rbis_batch.cu); every
// other kind the host lets through is RBIS_OP_RESTORE
constexpr int OP_IMU = 0, OP_MEAS = 1, OP_SNAPSHOT = 2, OP_RECORD = 4;

// ---- on-device synthesis of the input rows (SURVEY.md 8d; rbis_synth.cuh holds the kernels that MATERIALISE the rows) ----
// key = seed ^ filter * K1 ^ step * K2 ^ channel * K3;  a = splitmix64(key), b = splitmix64(a)
//   mode 0 (exact):  u1 = ((a >> 11) + 1) / (2^53 + 1), u2 = (b >> 11) / 2^53, n = sqrt(-2 ln u1) cos(2 pi u2) in double
//                    -- the integer part is bit-exact against numpy (pronto_b200/synth.py:normal), the libm calls to an ulp or two;
//   mode 1 (fast):   the same counters and hash, ONE hash per pair of channels (see syn_pair_k), ln / sqrt / cos in single
//                    precision with the SFU approximations (n carries ~1e-6 relative error, irrelevant for a noise sample).
// The SYN instantiations of the fused kernels draw mode-1 rows INSIDE the kernel with these same functions (same bits as the
// materialised rows), so a Monte-Carlo ensemble reads no per-filter input from HBM at all.
constexpr unsigned long long SYN_K1 = 0x9E3779B97F4A7C15ull, SYN_K2 = 0xC2B2AE3D27D4EB4Full, SYN_K3 = 0x165667B19E3779F9ull;
__host__ __device__ __forceinline__ unsigned long long splitmix64(unsigned long long x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
// kfs = seed ^ filter * K1 ^ step * K2 (the caller hoists what it can)
// Mode 1 draws channels in PAIRS (2k, 2k+1) from ONE hash of the even channel's key: radius from its top 24 bits, angle from
// the next 24, the even channel takes r cos(theta) and the odd one r cos(theta - pi/2) -- Box-Muller's two independent
// normals.  syn_pick(syn_pair_k(kfs, c & ~1), c & 1) is THE definition of channel c; code that needs both channels of a pair
// evaluates the pair once and gets the same bits.
struct SynPair {
  float r, th;
};
__device__ __forceinline__ SynPair syn_pair_k(unsigned long long kfs, unsigned even_channel) {
  const unsigned long long a = splitmix64(kfs ^ ((unsigned long long)even_channel * SYN_K3));
  const float u1 = ((float)(unsigned)(a >> 40) + 0.5f) * (1.0f / 16777216.0f);
  const float u2 = (float)((unsigned)(a >> 16) & 0xffffffu) * (1.0f / 16777216.0f);
  // -2 ln u1 = (-2 ln 2) lg2 u1 > 0; the SFU forms directly (sqrtf / __logf would add their range and rounding fix-ups)
  float l2, r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l2) : "f"(u1));
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(-1.3862943611198906f * l2));
  return {r, 6.2831853071795865f * u2};
}
__device__ __forceinline__ double syn_pick(const SynPair& p, unsigned odd) {
  return (double)(p.r * __cosf(odd ? p.th - 1.5707963267948966f : p.th));
}
template <int MODE>
__device__ __forceinline__ double syn_normal_k(unsigned long long kfs, unsigned channel) {
  if constexpr (MODE == 0) {
    const unsigned long long a = splitmix64(kfs ^ ((unsigned long long)channel * SYN_K3)), b = splitmix64(a);
    const double u1 = ((double)(a >> 11) + 1.0) * (1.0 / 9007199254740993.0);
    const double u2 = (double)(b >> 11) * (1.0 / 9007199254740992.0);
    return sqrt(-2.0 * log(u1)) * cos(2.0 * 3.14159265358979323846 * u2);
  } else {
    return syn_pick(syn_pair_k(kfs, channel & ~1u), channel & 1u);
  }
}
// channels c0 .. c0+COUNT-1 (c0 run time): one hash per pair touched
template <int MODE, int COUNT>
__device__ __forceinline__ void syn_normals_k(unsigned long long kfs, unsigned c0, double (&out)[COUNT]) {
  if constexpr (MODE == 0) {
#pragma unroll
    for (int a = 0; a < COUNT; a++) out[a] = syn_normal_k<0>(kfs, c0 + a);
  } else {
    SynPair p = syn_pair_k(kfs, c0 & ~1u);
#pragma unroll
    for (int a = 0; a < COUNT; a++) {
      const unsigned c = c0 + a;
      if (a > 0 && !(c & 1u)) p = syn_pair_k(kfs, c);
      out[a] = syn_pick(p, c & 1u);
    }
  }
}
template <int MODE>
__device__ __forceinline__ double syn_normal(unsigned long long seed, unsigned long long filter, unsigned long long step, unsigned channel) {
  return syn_normal_k<MODE>(seed ^ (filter * SYN_K1) ^ (step * SYN_K2), channel);
}
struct SynStreamK {
  const double* mean;       // device [rows][m]
  const double* mean_quat;  // device [rows][4] or nullptr
  const long long* step;    // device [rows]
  double sigma[9];
  double sigma_rot[3];
  int channel, channel_rot;
};
struct SynK {
  unsigned long long seed;
  long long first_filter;
  const double* imu_mean;   // device [rows][6]
  const long long* imu_step;
  double sigma_gyro, sigma_accel, dt;  // sigma < 0: per filter sqrt(q / dt)
  SynStreamK st[8];
};
// RBIS_OP_RECORD (REC kernel instantiations): bit f of `fields` records field f -- 0..20 state vector, 21..24 quaternion
// w, x, y, z, 25 log-likelihood, 26..46 covariance diagonal P(f-26, f-26) -- at out[row * k + pos][n], pos =
// popcount(fields & ((1 << f) - 1)).  After the fields, KParams::rec_cov_blocks selects covariance blocks: bit b is state
// block b (indices 3b..3b+2); with I the ascending selected indices, P(I[ii], I[jj]), ii <= jj, goes to position
// popcount(fields) + jj (jj + 1) / 2 + ii.  For a host output `out` is the call's staging buffer and the host has renumbered
// the RECORD rows into it (rbis_batch.cu).
constexpr int REC_FIELDS = 47;
constexpr int REC_BLOCKS = 7;
struct RecK {
  double* out;
  unsigned long long fields;
  long long k;  // popcount(fields) + nb (nb + 1) / 2, nb = 3 popcount(rec_cov_blocks)
};
// packed position of state index i within the selected covariance blocks cb (i's block selected)
__host__ __device__ __forceinline__ int rec_cov_index(unsigned cb, int i) {
#ifdef __CUDA_ARCH__
  return 3 * __popc(cb & ((1u << (i / 3)) - 1u)) + i % 3;
#else
  return 3 * __builtin_popcount(cb & ((1u << (i / 3)) - 1u)) + i % 3;
#endif
}
// the inverse: state index of packed position c
__host__ __device__ __forceinline__ int rec_cov_state(unsigned cb, int c) {
  int t = c / 3;
  for (int b = 0; b < REC_BLOCKS; b++)
    if ((cb >> b) & 1u) {
      if (t == 0) return 3 * b + c % 3;
      t--;
    }
  return -1;
}
// Innovation sets (INNOV kernel instantiations, which are REC instantiations too): every MEAS op on stream s with
// innov[s].out non-null writes row op.row of innov[s].out, [rows][k][N]: NIS = y^T S^-1 y (INNOV_NIS), then y_a = z_a - x-[idx_a] (INNOV_Y), then S(a,a) =
// P-(idx_a, idx_a) + R(a,a) (INNOV_S_DIAG), all from the prior state of the op; a filter that skips the row writes NaN.
constexpr int INNOV_NIS = 1, INNOV_Y = 2, INNOV_S_DIAG = 4;
struct InnovK {
  double* out;     // nullptr: no innovation set on this stream
  long long rows;
  int k, fields;   // k = NIS + m Y + m S_DIAG
};

struct KParams {
  long long N;
  double* vec;     // [21][N]
  double* quat;    // [4][N]
  double* P;       // [231][N]
  double* loglik;  // [N]
  const double* q_gyro;  // [N] each
  const double* q_accel;
  const double* q_gyro_bias;
  const double* q_accel_bias;
  const double* imu;  // [rows][6][imu_cols]
  const int* imu_map; // column of imu read by filter n (nullptr: column n)
  long long imu_cols;
  double* snap;       // [slots][257][N]
  const Op* ops;
  long long n_ops;
  double g_val, chi_tol;
  int ctor_folds_chi, renorm, n_snap;
  int block_offset;  // first CTA of this launch's range (launch groups)
  StreamDesc streams[MAX_STREAMS];
  SynK syn;          // SYN kernel instantiations only
  RecK rec;          // REC kernel instantiations only (last: the parameter offsets of everything above stay as they were)
  // MASK kernel instantiations only (appended for the same reason): bit s set = stream s has RBIS_STREAM_SKIP_NAN_ROWS, a
  // filter whose row of that stream holds a NaN in a value the update reads skips the MEAS op (see row_missing)
  unsigned skip_nan_streams;
  // REC kernel instantiations only (appended for the same reason): covariance blocks of the record set (see RecK)
  unsigned rec_cov_blocks;
  // INNOV kernel instantiations only (appended for the same reason): innovation sets per stream (see InnovK)
  InnovK innov[MAX_STREAMS];
};

// ------------------------------------------------------------------------------------------------
template <int... Is, class F>
__device__ __forceinline__ void static_for_impl(std::integer_sequence<int, Is...>, F&& f) {
  (f(std::integral_constant<int, Is>{}), ...);
}
template <int N, class F>
__device__ __forceinline__ void static_for(F&& f) {
  static_for_impl(std::make_integer_sequence<int, N>{}, static_cast<F&&>(f));
}

struct V3 {
  double x, y, z;
};
// The library is compiled with -fmad=false: every fused multiply-add is written out, so that all kernel variants and
// configurations of this file perform the same arithmetic bit for bit (the compiler's own contraction choices
// differ between instantiations).
__device__ __forceinline__ V3 cross(const V3& a, const V3& b) {
  return {fma(a.y, b.z, -(a.z * b.y)), fma(a.z, b.x, -(a.x * b.z)), fma(a.x, b.y, -(a.y * b.x))};
}
__device__ __forceinline__ double sumsq3(double x, double y, double z) { return fma(z, z, fma(y, y, x * x)); }
// acc + a x b  /  acc - a x b  as two FMAs per component
__device__ __forceinline__ V3 add_cross(const V3& acc, const V3& a, const V3& b) {
  return {fma(a.y, b.z, fma(-a.z, b.y, acc.x)), fma(a.z, b.x, fma(-a.x, b.z, acc.y)), fma(a.x, b.y, fma(-a.y, b.x, acc.z))};
}
__device__ __forceinline__ V3 sub_cross(const V3& acc, const V3& a, const V3& b) {
  return {fma(-a.y, b.z, fma(a.z, b.y, acc.x)), fma(-a.z, b.x, fma(a.x, b.z, acc.y)), fma(-a.x, b.y, fma(a.y, b.x, acc.z))};
}
__device__ __forceinline__ V3 axpy(double a, const V3& x, const V3& y) { return {fma(a, x.x, y.x), fma(a, x.y, y.y), fma(a, x.z, y.z)}; }

struct FilterState {
  double x[NS];
  double qw, qx, qy, qz;
  double ll;
};

// ---- quaternion helpers (Eigen semantics, SURVEY.md 8c) ----
struct Q4 {
  double w, x, y, z;
};
__device__ __forceinline__ Q4 qmul(const Q4& a, const Q4& b) {
  return {fma(-a.z, b.z, fma(-a.y, b.y, fma(-a.x, b.x, a.w * b.w))), fma(-a.z, b.y, fma(a.y, b.z, fma(a.x, b.w, a.w * b.x))),
          fma(-a.x, b.z, fma(a.z, b.x, fma(a.y, b.w, a.w * b.y))), fma(-a.y, b.x, fma(a.x, b.y, fma(a.z, b.w, a.w * b.z)))};
}
__device__ __forceinline__ Q4 qinv(const Q4& q) {
  const double n2 = fma(q.z, q.z, fma(q.y, q.y, fma(q.x, q.x, q.w * q.w)));
  if (n2 > 0) {
    const double r = 1.0 / n2;  // Eigen divides each coefficient; 1 ulp apart at most
    return {q.w * r, -q.x * r, -q.y * r, -q.z * r};
  }
  return {0, 0, 0, 0};
}
__device__ __forceinline__ V3 qrot(const Q4& q, const V3& v) {
  V3 u{q.x, q.y, q.z};
  V3 uv = cross(u, v);
  uv.x += uv.x; uv.y += uv.y; uv.z += uv.z;
  V3 c = cross(u, uv);
  return {fma(q.w, uv.x, v.x) + c.x, fma(q.w, uv.y, v.y) + c.y, fma(q.w, uv.z, v.z) + c.z};
}
// sin / cos of a small angle by their Taylor series (|x| <= 0.25: truncation below 3e-18 relative), the library routine
// otherwise: half rotation increments of a 1 kHz filter are ~1e-4
__device__ __forceinline__ void sincos_small(double x, double* sp, double* cp) {
  if (fabs(x) <= 0.25) {
    const double x2 = x * x;
    double ps = fma(x2, -1.0 / 6227020800.0, 1.0 / 39916800.0);
    ps = fma(x2, ps, -1.0 / 362880.0);
    ps = fma(x2, ps, 1.0 / 5040.0);
    ps = fma(x2, ps, -1.0 / 120.0);
    ps = fma(x2, ps, 1.0 / 6.0);
    *sp = fma(-x * x2, ps, x);
    double pc = fma(x2, 1.0 / 479001600.0, -1.0 / 3628800.0);
    pc = fma(x2, pc, 1.0 / 40320.0);
    pc = fma(x2, pc, -1.0 / 720.0);
    pc = fma(x2, pc, 1.0 / 24.0);
    pc = fma(x2, pc, -0.5);
    *cp = fma(x2, pc, 1.0);
    return;
  }
  sincos(x, sp, cp);
}
// quaternion of AngleAxis(|chi|, chi/|chi|)
__device__ __forceinline__ Q4 qexp(const V3& chi, double n) {
  double s, c;
  sincos_small(0.5 * n, &s, &c);
  const double rn = 1.0 / n;  // one reciprocal instead of three divisions (<= 1 ulp apart per component)
  return {c, s * (chi.x * rn), s * (chi.y * rn), s * (chi.z * rn)};
}
// the same from the SQUARED norm: one reciprocal square root gives both |chi| and 1/|chi|
__device__ __forceinline__ Q4 qexp2(const V3& chi, double n2) {
  const double rn = rsqrt(n2);
  double s, c;
  sincos_small(0.5 * (n2 * rn), &s, &c);
  return {c, s * (chi.x * rn), s * (chi.y * rn), s * (chi.z * rn)};
}
// subtractQuats(q1, q2) = axis*angle of q2^-1 * q1 (Eigen >= 3.3 AngleAxis, bot_mod2pi)
__device__ __forceinline__ V3 subtract_quats(const Q4& q1, const Q4& q2) {
  const Q4 r = qmul(qinv(q2), q1);
  double n = sqrt(sumsq3(r.x, r.y, r.z));
  if (n == 0.0) return {0, 0, 0};
  double angle = 2.0 * atan2(n, fabs(r.w));
  if (r.w < 0) n = -n;
  const double PI = 3.14159265358979323846;
  if (angle >= PI) angle -= 2 * PI;  // bot_mod2pi maps exactly pi to -pi, identity below
  return {r.x / n * angle, r.y / n * angle, r.z / n * angle};
}

// ---- synthesised input rows (SYN kernels and the materialising kernels of rbis_synth.cuh share these) ----
// measured orientation of a pose row: mean_quat (x) Exp(sigma_rot * n); plain products and sums in the order of
// pronto_b200/synth.py (no contraction: the library is built with -fmad=false)
template <int MODE>
__device__ __forceinline__ Q4 syn_quat(const double* __restrict__ mq, const double (&sigma_rot)[3], unsigned long long kfs, unsigned channel_rot) {
  double nn[3];
  syn_normals_k<MODE, 3>(kfs, channel_rot, nn);
  const V3 chi{sigma_rot[0] * nn[0], sigma_rot[1] * nn[1], sigma_rot[2] * nn[2]};
  const double nrm = sqrt(chi.x * chi.x + chi.y * chi.y + chi.z * chi.z);
  double sn = 0.0, cs = 1.0;
  if (nrm > 0) { sincos(0.5 * nrm, &sn, &cs); sn /= nrm; }
  const Q4 dq{cs, sn * chi.x, sn * chi.y, sn * chi.z};
  const Q4 t{mq[0], mq[1], mq[2], mq[3]};
  return {t.w * dq.w - t.x * dq.x - t.y * dq.y - t.z * dq.z, t.w * dq.x + t.x * dq.w + t.y * dq.z - t.z * dq.y,
          t.w * dq.y + t.y * dq.w + t.z * dq.x - t.x * dq.z, t.w * dq.z + t.z * dq.w + t.x * dq.y - t.y * dq.x};
}

// ------------------------------------------------------------------------------------------------
// Tensor-memory access.  No "memory" clobbers: the asm statements are volatile, so they keep their
// program order among themselves, while ordinary shared/global accesses may move around them.
// Loaded registers become valid only after tm_wait_ld(); consumers are tied to the wait by passing
// the raw registers through an empty volatile asm placed after it (tm_settle).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tm_ld2(uint32_t taddr, uint32_t& lo, uint32_t& hi) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(lo), "=r"(hi) : "r"(taddr));
}
__device__ __forceinline__ void tm_st2(uint32_t taddr, double v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr), "r"(__double2loint(v)), "r"(__double2hiint(v)));
}
__device__ __forceinline__ void tm_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;"); }
__device__ __forceinline__ void tm_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;"); }
__device__ __forceinline__ double tm_settle(uint32_t& lo, uint32_t& hi) {
  asm volatile("" : "+r"(lo), "+r"(hi));
  return __hiloint2double((int)hi, (int)lo);
}

// Input loads that must be ISSUED where they are written (top of an op) and consumed a few thousand
// cycles later: volatile, so ptxas cannot sink them next to their first use to save registers, which is
// what it does with plain __ldg and what exposed the full HBM latency once per op.
__device__ __forceinline__ double ldg_early(const double* ptr) {
  double v;
  asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(ptr));
  return v;
}

// Where the rows of a measurement op come from: HBM (st.z, st.quat), or -- SYN kernels -- drawn on the spot from the
// noise-free row and the filter's counters, with the expressions of the materialising kernels in rbis_synth.cuh.
template <bool SYN>
struct MeasSrc {
  const SynStreamK* ss;    // SYN only
  unsigned long long kfs;  // SYN only: seed ^ filter * K1 ^ step * K2
  template <bool EARLY = true>
  __device__ __forceinline__ double z(const StreamDesc& st, long long row, int a, long long sn) const {
    if constexpr (SYN) return fma(ss->sigma[a], syn_normal_k<1>(kfs, (unsigned)(ss->channel + a)), __ldg(ss->mean + row * st.m + a));
    else if constexpr (EARLY) return ldg_early(st.z + (row * st.m + a) * st.cols + sn);
    else return __ldg(st.z + (row * st.m + a) * st.cols + sn);
  }
  // rows a0, a0+1, a0+2
  __device__ __forceinline__ void z3(const StreamDesc& st, long long row, int a0, long long sn, double (&out)[3]) const {
    if constexpr (SYN) {
      double nn[3];
      syn_normals_k<1, 3>(kfs, (unsigned)(ss->channel + a0), nn);
#pragma unroll
      for (int a = 0; a < 3; a++) out[a] = fma(ss->sigma[a0 + a], nn[a], __ldg(ss->mean + row * st.m + a0 + a));
    } else {
#pragma unroll
      for (int a = 0; a < 3; a++) out[a] = ldg_early(st.z + (row * st.m + (a0 + a)) * st.cols + sn);
    }
  }
  __device__ __forceinline__ Q4 quat(const StreamDesc& st, long long row, long long sn) const {
    if constexpr (SYN) return syn_quat<1>(ss->mean_quat + row * 4, ss->sigma_rot, kfs, (unsigned)ss->channel_rot);
    else {
      const long long SN = st.cols;
      const double* qb = st.quat + row * 4 * SN + sn;
      return {__ldg(qb), __ldg(qb + SN), __ldg(qb + 2 * SN), __ldg(qb + 3 * SN)};
    }
  }
};

// Per-lane view of the covariance.
struct Cov {
  double* Ps;    // shared base + lane;  shared slot k at Ps[k * TPB]
  uint32_t tm;   // tensor-memory address of this thread's first column; slot k at tm + 2k
  // ---- either memory, compile-time (I, J): store ----
  template <int I, int J>
  __device__ __forceinline__ void set(double v) {
    constexpr int i = I < J ? I : J, j = I < J ? J : I;
    if constexpr (in_tm(i, j)) tm_st2(tm + 2 * tm_index(i, j), v);
    else Ps[sm_off(sm_index(i, j))] = v;
  }
  template <int R0, int C>
  __device__ __forceinline__ void setcol3(const V3& v) {
    set<R0, C>(v.x); set<R0 + 1, C>(v.y); set<R0 + 2, C>(v.z);
  }
};

// A fetch list L names N covariance elements at compile time: L::N, L::row(k), L::col(k).
template <int N>
struct Buf {
  double d[N];
  uint32_t lo[N], hi[N];
};
template <class L, int NB>
__device__ __forceinline__ void issue(const Cov& P, Buf<NB>& b) {
  static_assert(NB >= L::N, "buffer too small for the fetch list");
  static_for<L::N>([&](auto kc) {
    constexpr int k = kc;
    constexpr int i = L::row(k) < L::col(k) ? L::row(k) : L::col(k), j = L::row(k) < L::col(k) ? L::col(k) : L::row(k);
    if constexpr (in_tm(i, j)) tm_ld2(P.tm + 2 * tm_index(i, j), b.lo[k], b.hi[k]);
    else b.d[k] = P.Ps[sm_off(sm_index(i, j))];
  });
}
template <class L>
__host__ __device__ constexpr bool any_tm() {
  bool any = false;
  for (int k = 0; k < L::N; k++) {
    const int i = L::row(k) < L::col(k) ? L::row(k) : L::col(k), j = L::row(k) < L::col(k) ? L::col(k) : L::row(k);
    any = any || in_tm(i, j);
  }
  return any;
}
template <class L, int NB>
__device__ __forceinline__ void commit(Buf<NB>& b) {
  if constexpr (any_tm<L>()) tm_wait_ld();
  static_for<L::N>([&](auto kc) {
    constexpr int k = kc;
    constexpr int i = L::row(k) < L::col(k) ? L::row(k) : L::col(k), j = L::row(k) < L::col(k) ? L::col(k) : L::row(k);
    if constexpr (in_tm(i, j)) b.d[k] = tm_settle(b.lo[k], b.hi[k]);
  });
}

// rows R0.., R1.., ... (three each) of column C
template <int C, int... R0s>
struct ColRows {
  static constexpr int N = 3 * (int)sizeof...(R0s);
  static constexpr int row(int k) {
    constexpr int r0[] = {R0s...};
    return r0[k / 3] + k % 3;
  }
  static constexpr int col(int) { return C; }
};
// packed slots S0 .. S0+N-1
template <int S0, int N_>
struct SlotRun {
  static constexpr int N = N_;
  static constexpr int row(int k) { return row_of_slot(S0 + k); }
  static constexpr int col(int k) { return col_of_slot(S0 + k); }
};

// active packed slots kAct.s[K0 .. K0+N-1]
template <int K0, int N_>
struct ActRun {
  static constexpr int N = N_;
  static constexpr int row(int k) { return row_of_slot(kAct.s[K0 + k]); }
  static constexpr int col(int k) { return col_of_slot(kAct.s[K0 + k]); }
};
// the slots a whole-covariance sweep visits: all 231 (dense) or the 120 active ones (DC)
template <bool DC, int K0, int N_>
struct SweepRun_ { using type = SlotRun<K0, N_>; };
template <int K0, int N_>
struct SweepRun_<true, K0, N_> { using type = ActRun<K0, N_>; };
template <bool DC, int K0, int N_>
using SweepRun = typename SweepRun_<DC, K0, N_>::type;
template <bool DC>
constexpr int kSweepLen = DC ? NP_ACT : NP;

template <int... Cs>
struct ColList {
  static constexpr int n = (int)sizeof...(Cs);
  static constexpr int at(int k) {
    constexpr int c[] = {Cs...};
    return c[k];
  }
};

template <int K, class A, class B>
__device__ __forceinline__ auto& pick(A& a, B& b) {
  if constexpr (K == 0) return a;
  else return b;
}
__device__ __forceinline__ V3 v3at(const double* d, int k) { return {d[3 * k], d[3 * k + 1], d[3 * k + 2]}; }

// Software-pipelined sweep over the compile-time column list Cs...: the fetch of column k+1 is
// issued before column k is processed by f(column, values).  f may store to the covariance, but
// never to an element that the fetch of the NEXT column reads (checked per call site, see below).
template <template <int> class L, class Cols, class F>
__device__ __forceinline__ void for_columns(const Cov& P, Cols, F&& f) {
  constexpr int n = Cols::n;
  constexpr int LN = L<Cols::at(0)>::N;
  Buf<LN> b0, b1;
  issue<L<Cols::at(0)>>(P, b0);
  static_for<n>([&](auto kc) {
    constexpr int k = kc;
    auto& cur = pick<k % 2>(b0, b1);
    auto& nxt = pick<(k + 1) % 2>(b0, b1);
    commit<L<Cols::at(k)>>(cur);
    if constexpr (k + 1 < n) issue<L<Cols::at(k + 1 < n ? k + 1 : k)>>(P, nxt);
    f(std::integral_constant<int, Cols::at(k)>{}, cur.d, kc);
  });
}

// ------------------------------------------------------------------------------------------------
// Covariance propagation.  Ad = I + dt*Ac has non-identity block rows v, chi, p only, and because
// the p-columns of Ac are zero and chi's row has no v-column, Ad factors EXACTLY as
//     Ad = E_chi * E_v * E_p,   E_X = I + (block row X of dt*Ac),
// so  Ad P Ad^T = E_chi (E_v (E_p P E_p^T) E_v^T) E_chi^T : three in-place symmetric congruences,
// each touching one block row/column.  For E = I + N (N supported on block row I):
//     z_c   = P[I,c] + N[I,:] P[:,c]            for every column c
//     P'[I,c] = z_c (c outside I),   P'[I,I] = Z_I + sum_K Z_K N[I,K]^T
// Columns of omega and a (passive: their rows of Ad are identity and nothing reads them back) take
// all three congruences in ONE pass from the old values.  Products with the structural zeros/ones
// of Ad are skipped; everything else is the dense product's arithmetic up to summation order.
// ------------------------------------------------------------------------------------------------
struct Lin {  // linearisation point quantities, pre-scaled by dt where the reference scales Ac by dt
  V3 v;        // body velocity (unscaled)
  V3 wd;       // omega * dt
  V3 vd;       // v * dt
  V3 gd;       // (q^-1 g_vec) * dt
  double Rd[9];  // R * dt, row-major Rd[3*r + c]
  double dt;
};

// rows p:  z = P[p,c] + R dt (P[v,c] - v x P[chi,c])
__device__ __forceinline__ V3 zp(const Lin& L, const V3& pv, const V3& pc, const V3& pp) {
  const V3 t = sub_cross(pv, L.v, pc);
  return {fma(L.Rd[0], t.x, fma(L.Rd[1], t.y, fma(L.Rd[2], t.z, pp.x))), fma(L.Rd[3], t.x, fma(L.Rd[4], t.y, fma(L.Rd[5], t.z, pp.y))),
          fma(L.Rd[6], t.x, fma(L.Rd[7], t.y, fma(L.Rd[8], t.z, pp.z)))};
}
// rows v:  z = P[v,c] - wd x P[v,c] + gd x P[chi,c] - vd x P[bg,c] - dt P[ba,c]
__device__ __forceinline__ V3 zv(const Lin& L, const V3& pv, const V3& pc, const V3& pg, const V3& pa) {
  const V3 a = sub_cross(pv, L.wd, pv);
  const V3 b = add_cross(axpy(-L.dt, pa, {0.0, 0.0, 0.0}), L.gd, pc);  // second chain, joined at the end
  const V3 c = sub_cross(a, L.vd, pg);
  return {c.x + b.x, c.y + b.y, c.z + b.z};
}
// rows chi:  z = P[chi,c] - wd x P[chi,c] - dt P[bg,c]
__device__ __forceinline__ V3 zc(const Lin& L, const V3& pc, const V3& pg) { return sub_cross(axpy(-L.dt, pg, pc), L.wd, pc); }

// acc += sign * Z skew(u), Z given as three columns:  (Z skew(u))[:,0] = u.z Z1 - u.y Z2, ...
template <int SIGN>
__device__ __forceinline__ void acc_mul_skew(V3 acc[3], const V3 Z[3], const V3& u) {
  const double ux = SIGN * u.x, uy = SIGN * u.y, uz = SIGN * u.z;
  acc[0] = axpy(uz, Z[1], axpy(-uy, Z[2], acc[0]));
  acc[1] = axpy(ux, Z[2], axpy(-uz, Z[0], acc[1]));
  acc[2] = axpy(uy, Z[0], axpy(-ux, Z[1], acc[2]));
}

template <int C> using FetchEp = ColRows<C, 3, 6, 9>;        // rows v, chi, p
template <int C> using FetchEv = ColRows<C, 3, 6, 15, 18>;   // rows v, chi, bg, ba
template <int C> using FetchEc = ColRows<C, 6, 15>;          // rows chi, bg
template <int C> using FetchAll = ColRows<C, 3, 6, 9, 15, 18>;

// after_passive() returns the four process-noise values and before_ev() is called between E_p and E_v: the kernel
// issues the loads of the noise parameters / of the IMU sample there, so that those registers are not held
// through the phases with the highest pressure (see RBIS_LATE_LOADS).
struct QNoise {
  double q_gyro, q_accel, q_gyro_bias, q_accel_bias;
};
template <bool DC, class AfterPassive, class BeforeEv>
__device__ __forceinline__ void cov_propagate(Cov& P, const Lin& L, AfterPassive&& after_passive, BeforeEv&& before_ev) {
  const double dt = L.dt;
  // ---------------- passive columns omega (0..2), a (12..14): all three congruences in one pass ----------------
  if constexpr (!DC) {
    for_columns<FetchAll>(P, ColList<0, 1, 2, 12, 13, 14>{}, [&](auto cc, const double* d, auto) {
      constexpr int c = cc;
      const V3 pv = v3at(d, 0), pc = v3at(d, 1), pp = v3at(d, 2), pg = v3at(d, 3), pa = v3at(d, 4);
      P.setcol3<9, c>(zp(L, pv, pc, pp));
      P.setcol3<3, c>(zv(L, pv, pc, pg, pa));
      P.setcol3<6, c>(zc(L, pc, pg));
      RBIS_SCHED_FENCE();
    });
  }
  const QNoise qn = after_passive();
  const double q_gyro = qn.q_gyro, q_accel = qn.q_accel, q_gyro_bias = qn.q_gyro_bias, q_accel_bias = qn.q_accel_bias;
  // ---------------- E_p on the active block: block row p (9..11), sources v (3..5), chi (6..8) ----------------
  // column order p, v, chi, bg, ba.  Stores: (p,v) after the v columns, (p,chi) after the chi columns,
  // (p,p) after that, (p,c) per column for bg/ba -- none is read by a later fetch of this phase.
  {
    V3 Zp[3], T[3], Zb[3];
    for_columns<FetchEp>(P, ColList<9, 10, 11, 3, 4, 5, 6, 7, 8, 15, 16, 17, 18, 19, 20>{}, [&](auto cc, const double* d, auto stage) {
      constexpr int c = cc;
      const V3 z = zp(L, v3at(d, 0), v3at(d, 1), v3at(d, 2));
      if constexpr (c >= 9 && c < 12) Zp[c - 9] = z;
      else if constexpr (c >= 3 && c < 6) {
        T[c - 3] = z;
        P.setcol3<9, c>(z);
      } else if constexpr (c >= 6 && c < 9) {
        Zb[c - 6] = z;
        P.setcol3<9, c>(z);
        if constexpr (c == 8) {
          // T = Zv + Zc skew(v);  P'[p,p] = Zp + T (R dt)^T,  (T Rd^T)[i][j] = sum_k T[k].i * Rd[3j+k]
          acc_mul_skew<1>(T, Zb, L.v);
          P.set<9, 9>(fma(T[0].x, L.Rd[0], fma(T[1].x, L.Rd[1], fma(T[2].x, L.Rd[2], Zp[0].x))));
          P.set<9, 10>(fma(T[0].x, L.Rd[3], fma(T[1].x, L.Rd[4], fma(T[2].x, L.Rd[5], Zp[1].x))));
          P.set<9, 11>(fma(T[0].x, L.Rd[6], fma(T[1].x, L.Rd[7], fma(T[2].x, L.Rd[8], Zp[2].x))));
          P.set<10, 10>(fma(T[0].y, L.Rd[3], fma(T[1].y, L.Rd[4], fma(T[2].y, L.Rd[5], Zp[1].y))));
          P.set<10, 11>(fma(T[0].y, L.Rd[6], fma(T[1].y, L.Rd[7], fma(T[2].y, L.Rd[8], Zp[2].y))));
          P.set<11, 11>(fma(T[0].z, L.Rd[6], fma(T[1].z, L.Rd[7], fma(T[2].z, L.Rd[8], Zp[2].z))));
        }
      } else {
        P.setcol3<9, c>(z);
      }
    });
  }
  tm_wait_st();
  before_ev();
  // ---------------- E_v: block row v (3..5), sources v, chi, bg (15..17), ba (18..20) ----------------
  // column order v, chi, bg, ba, p.  P'[v,v] = Zv + Zv skew(wd) - Zc skew(gd) + Zg skew(vd) - dt Za + Qd[v,v]
  // is accumulated block by block; each Z block is stored as soon as it is complete.
  const double qg = q_gyro * dt, qa = q_accel * dt;
  {
    V3 Nv[3], Zb[3];
    for_columns<FetchEv>(P, ColList<3, 4, 5, 6, 7, 8, 15, 16, 17, 18, 19, 20, 9, 10, 11>{}, [&](auto cc, const double* d, auto stage) {
      constexpr int c = cc;
      const V3 z = zv(L, v3at(d, 0), v3at(d, 1), v3at(d, 2), v3at(d, 3));
      if constexpr (c >= 9 && c < 12) {
        P.setcol3<3, c>(z);
      } else {
        constexpr int k = c % 3;
        Zb[k] = z;
        if constexpr (c >= 18) P.set<c, c>(fma(q_accel_bias, dt, d[9 + k]));  // Qd[ba,ba]; (ba,ba) is not read again in this step
        if constexpr (k == 2) {
          if constexpr (c == 5) {
            Nv[0] = Zb[0]; Nv[1] = Zb[1]; Nv[2] = Zb[2];
            acc_mul_skew<1>(Nv, Zb, L.wd);
          } else if constexpr (c == 8) {
            acc_mul_skew<-1>(Nv, Zb, L.gd);
            static_for<3>([&](auto kk) { P.setcol3<3, 6 + kk>(Zb[kk]); });
          } else if constexpr (c == 17) {
            acc_mul_skew<1>(Nv, Zb, L.vd);
            static_for<3>([&](auto kk) { P.setcol3<3, 15 + kk>(Zb[kk]); });
          } else {
            static_for<3>([&](auto kk) { Nv[kk] = axpy(-dt, Zb[kk], Nv[kk]); });
            static_for<3>([&](auto kk) { P.setcol3<3, 18 + kk>(Zb[kk]); });
            // Qd[v,v] = dt (q_gyro (|v|^2 I - v v^T) + q_accel I)      (rbis.cpp:91-116)
            const double vv = sumsq3(L.v.x, L.v.y, L.v.z);
            P.set<3, 3>(Nv[0].x + fma(qg, fma(-L.v.x, L.v.x, vv), qa));
            P.set<3, 4>(fma(qg, -L.v.x * L.v.y, Nv[1].x));
            P.set<3, 5>(fma(qg, -L.v.x * L.v.z, Nv[2].x));
            P.set<4, 4>(Nv[1].y + fma(qg, fma(-L.v.y, L.v.y, vv), qa));
            P.set<4, 5>(fma(qg, -L.v.y * L.v.z, Nv[2].y));
            P.set<5, 5>(Nv[2].z + fma(qg, fma(-L.v.z, L.v.z, vv), qa));
          }
        }
      }
    });
  }
  tm_wait_st();
  // ---------------- E_chi: block row chi (6..8), sources chi, bg ----------------
  // column order chi, bg, v, p, ba.  P'[chi,chi] = Zc + Zc skew(wd) - dt Zg + Qd[chi,chi]
  {
    V3 Mc[3], Zb[3];
    for_columns<FetchEc>(P, ColList<6, 7, 8, 15, 16, 17, 3, 4, 5, 9, 10, 11, 18, 19, 20>{}, [&](auto cc, const double* d, auto stage) {
      constexpr int c = cc;
      const V3 z = zc(L, v3at(d, 0), v3at(d, 1));
      if constexpr (c >= 6 && c < 9) {
        Zb[c - 6] = z;
        if constexpr (c == 8) {
          Mc[0] = Zb[0]; Mc[1] = Zb[1]; Mc[2] = Zb[2];
          acc_mul_skew<1>(Mc, Zb, L.wd);
        }
      } else if constexpr (c >= 15 && c < 18) {
        constexpr int k = c - 15;
        Mc[k] = axpy(-dt, z, Mc[k]);
        P.setcol3<6, c>(z);
        P.set<c, c>(fma(q_gyro_bias, dt, d[3 + k]));  // Qd[bg,bg]; (bg,bg) is not read again in this step
        if constexpr (c == 17) {
          P.set<6, 6>(Mc[0].x + qg); P.set<6, 7>(Mc[1].x); P.set<6, 8>(Mc[2].x);
          P.set<7, 7>(Mc[1].y + qg); P.set<7, 8>(Mc[2].y);
          P.set<8, 8>(Mc[2].z + qg);
        }
      } else if constexpr (c >= 3 && c < 6) {
        // P'[chi, v_k] = z + Qd[chi, v_k];  Qd[v,chi] = dt q_gyro skew(v)  =>  Qd[chi_i, v_k] = qg*skew(v)[k][i]
        if constexpr (c == 3) P.setcol3<6, 3>({z.x, fma(qg, -L.v.z, z.y), fma(qg, L.v.y, z.z)});
        else if constexpr (c == 4) P.setcol3<6, 4>({fma(qg, L.v.z, z.x), z.y, fma(qg, -L.v.x, z.z)});
        else P.setcol3<6, 5>({fma(qg, -L.v.y, z.x), fma(qg, L.v.x, z.y), z.z});
      } else {
        P.setcol3<6, c>(z);
      }
    });
  }
  tm_wait_st();
  // overwrites of rbis.cpp:120-121 (nothing in this step reads these blocks; the DC kernel writes them to global
  // memory when a snapshot or the end of the program needs them)
  if constexpr (!DC) {
    P.set<12, 12>(q_accel); P.set<13, 13>(q_accel); P.set<14, 14>(q_accel);
    P.set<12, 13>(0.0); P.set<12, 14>(0.0); P.set<13, 14>(0.0);
    P.set<0, 0>(q_gyro); P.set<1, 1>(q_gyro); P.set<2, 2>(q_gyro);
    P.set<0, 1>(0.0); P.set<0, 2>(0.0); P.set<1, 2>(0.0);
    tm_wait_st();
  }
}

// chiToQuat on the filter state: fold vec chi into the quaternion when its norm exceeds the tolerance
__device__ __forceinline__ void fold_chi(FilterState& s, double chi_tol) {
  const V3 c{s.x[6], s.x[7], s.x[8]};
  // the common case is chi == 0 (folded by the previous update): compare squared norms, root only when folding
  const double n2 = sumsq3(c.x, c.y, c.z);
  if (n2 > chi_tol * chi_tol) {
    const Q4 q = qmul({s.qw, s.qx, s.qy, s.qz}, qexp2(c, n2));
    s.qw = q.w; s.qx = q.x; s.qy = q.y; s.qz = q.z;
    s.x[6] = 0; s.x[7] = 0; s.x[8] = 0;
  }
}

// addState(dstate) where dstate.vec = d (already added to s.x EXCEPT chi, passed separately) and
// dstate.quat = dq:  vec += d; chiToQuat(); quat *= dq
__device__ __forceinline__ void add_state_tail(FilterState& s, const V3& dchi, bool d_folded, const Q4& dq,
                                               double chi_tol, int renorm) {
  if (!d_folded) { s.x[6] += dchi.x; s.x[7] += dchi.y; s.x[8] += dchi.z; }
  fold_chi(s, chi_tol);
  if (d_folded) {
    const Q4 q = qmul({s.qw, s.qx, s.qy, s.qz}, dq);
    s.qw = q.w; s.qx = q.x; s.qy = q.y; s.qz = q.z;
  }
  if (renorm) {
    const double r = 1.0 / sqrt(fma(s.qz, s.qz, fma(s.qy, s.qy, fma(s.qx, s.qx, s.qw * s.qw))));
    s.qw *= r; s.qx *= r; s.qy *= r; s.qz *= r;
  }
}

// insUpdateState, rbis.cpp:37-75.  gb = q^-1 g_vec at the prior quaternion.  The caller has already added the position
// increment dp = (q v) dt, from the prior q and v.
__device__ __forceinline__ void state_propagate(FilterState& s, const V3& gyro, const V3& acc, double dt, const V3& gb,
                                                double chi_tol, int renorm) {
  const V3 w{gyro.x - s.x[15], gyro.y - s.x[16], gyro.z - s.x[17]};
  const V3 a{acc.x - s.x[18], acc.y - s.x[19], acc.z - s.x[20]};
  s.x[0] = w.x; s.x[1] = w.y; s.x[2] = w.z;
  s.x[12] = a.x; s.x[13] = a.y; s.x[14] = a.z;
  const V3 v{s.x[3], s.x[4], s.x[5]};
  const V3 wxv = cross(w, v);
  const V3 dv{(-wxv.x + (gb.x + a.x)) * dt, (-wxv.y + (gb.y + a.y)) * dt, (-wxv.z + (gb.z + a.z)) * dt};
  V3 dchi{w.x * dt, w.y * dt, w.z * dt};
  // dstate.chiToQuat()
  Q4 dq{1, 0, 0, 0};
  const double n2 = sumsq3(dchi.x, dchi.y, dchi.z);
  const bool folded = n2 > chi_tol * chi_tol;
  if (folded) dq = qexp2(dchi, n2);
  // addState
  s.x[3] += dv.x; s.x[4] += dv.y; s.x[5] += dv.z;
  add_state_tail(s, dchi, folded, dq, chi_tol, renorm);
}

// ---- parking of the filter state in this thread's spare tensor memory (slots N_TM ...) ----
// field k of the state: 0..20 vec, 21..24 quaternion, 25 log-likelihood; MASK selects the fields
__device__ __forceinline__ double& state_field(FilterState& s, int k) {
  return k < NS ? s.x[k] : k == 21 ? s.qw : k == 22 ? s.qx : k == 23 ? s.qy : k == 24 ? s.qz : s.ll;
}
template <uint32_t MASK>
__device__ __forceinline__ void park_state(const Cov& P, FilterState& s) {
  static_for<26>([&](auto kc) {
    constexpr int k = kc;
    if constexpr ((MASK >> k) & 1u) tm_st2(P.tm + 2 * (N_TM + k), state_field(s, k));
  });
}
template <uint32_t MASK>
__device__ __forceinline__ void unpark_state(const Cov& P, FilterState& s) {
  uint32_t lo[26], hi[26];
  static_for<26>([&](auto kc) {
    constexpr int k = kc;
    if constexpr ((MASK >> k) & 1u) tm_ld2(P.tm + 2 * (N_TM + k), lo[k], hi[k]);
  });
  tm_wait_ld();
  static_for<26>([&](auto kc) {
    constexpr int k = kc;
    if constexpr ((MASK >> k) & 1u) state_field(s, k) = tm_settle(lo[k], hi[k]);
  });
}
constexpr uint32_t PARK_EVERYTHING = (1u << 26) - 1;
#ifndef RBIS_PARK_COV_KEEP
#define RBIS_PARK_COV_KEEP 0u    // fields that stay in registers during the covariance step (bit mask, dev knob)
#endif
constexpr uint32_t PARK_MEAS_KEEP = 0u;  // fields that stay in registers during a measurement sweep (bit mask)
constexpr uint32_t PARK_ALL = PARK_EVERYTHING & ~PARK_MEAS_KEEP;
// during the covariance step: v, chi, p, b_g, b_a, quaternion, log-likelihood (omega and a are rewritten by the state
// step that follows; the linearisation point is already in Lin)
constexpr uint32_t PARK_COV = PARK_EVERYTHING & ~(0x7u | (0x7u << 12)) & ~(uint32_t)(RBIS_PARK_COV_KEEP);

// ---- rows missing per filter (MASK kernel instantiations, RBIS_STREAM_SKIP_NAN_ROWS) ----
// Row `row` of stream st is missing for this lane's filter when any z value the update reads in its column sn is NaN; the
// chi entries of an orientation stream are not read.  At most MAX_MEAS coalesced loads.
__device__ __forceinline__ bool row_missing(const StreamDesc& st, long long row, long long sn) {
  bool miss = false;
  for (int a = 0; a < st.m; a++) {
    const int i = st.idx[a];
    if (st.has_orient && i >= 6 && i <= 8) continue;
    miss = miss | (bool)isnan(__ldg(st.z + (row * st.m + a) * st.cols + sn));
  }
  return miss;
}
// A lane that skips runs the same instruction stream (the tensor-memory accesses and warp barriers of the updates are
// warp-collective) and keeps its old values: every store of an update selects the old value, `skip ? old : new`.  A
// select, not arithmetic on zeroed factors, which would turn a stored -0.0 into +0.0.  Without MASK the updates keep
// their plain statements (`if constexpr (MASK) ... else <statement>`): even an inlined identity wrapper around them
// changes the register allocation of the instantiations that exist without MASK.

// x[idx] with a runtime (warp-uniform) index: select chain, registers cannot be indexed dynamically
__device__ __forceinline__ double pick_state(const double (&x)[NS], int idx) {
  double v = x[0];
#pragma unroll
  for (int k = 1; k < NS; k++) v = (idx == k) ? x[k] : v;
  return v;
}

// ------------------------------------------------------------------------------------------------
// Measurement chunks.  A chunk is M consecutive rows a0..a0+M-1 of a stream, processed as a standard
// EKF update on the CURRENT covariance:  S = R + P[idx,idx];  K^T = S^-1 P[idx,:];
// P -= P[:,idx] S^-1 P[idx,:];  x += K r;  loglik += -log det S - r^T S^-1 r   (rbis.cpp:134-142).
// The host splits a stream into chunks only along blocks where R is block diagonal, for which
// processing the chunks in sequence is algebraically identical to the reference's single batch
// update (chain rule of the Gaussian likelihood); residuals of later chunks are taken against the
// already-updated vec, chi residuals against the accumulated chi delta.
//
// meas3<I0>: the chunk is the aligned index triple I0, I0+1, I0+2 (leg-odometry velocity 3..5, pose
// position 9..11, pose orientation 6..8, ...).  With S = L D L^T and Y = L^-1 P[idx,:] the update is
// P -= Y^T D^-1 Y, x += Y^T D^-1 L^-1 r: only Y (63 doubles) is held in registers, and the 231-slot
// sweep is software pipelined in tiles over both memories.
// ------------------------------------------------------------------------------------------------
template <int I0>
struct HPRow0 {  // elements (I0, c), (I0+1, c), (I0+2, c) for c = 3B..3B+2 -> nine per tile, one tile per index triple B
  template <int B>
  struct Tile {
    static constexpr int N = 9;
    static constexpr int row(int k) { return I0 + k % 3; }
    static constexpr int col(int k) { return 3 * B + k / 3; }
  };
};

template <bool DC>
__host__ __device__ constexpr int carried_block(int t) { return DC ? (t < 3 ? t + 1 : t + 2) : t; }
template <bool DC>
__host__ __device__ constexpr int carried_pos(int c) { return DC ? act_pos(c) : c; }

// DC: only the 15 active rows/columns exist (the couplings to omega / a are exactly zero, so are their gains).
// MASK: skip = the row is missing for this lane's filter, which then keeps covariance, state and log-likelihood (see row_missing).
// NISQ: *nisq += the chunk's quadratic form r^T S^-1 r (the same for meas1 / meas_block); their sum over the chunks of an
// update is its NIS (innovation sets, see InnovK).
template <int I0, bool DC, bool SYN, bool MASK = false, bool NISQ = false>
__device__ __forceinline__ void meas3(Cov& P, FilterState& s, const StreamDesc& st, const MeasSrc<SYN>& src, int a0, long long row, long long N,
                                      long long n, long long sn, const V3& dquat, const V3& chi0, bool skip = false,
                                      double* nisq = nullptr) {
  static_assert(!DC || (is_act(I0) && I0 % 3 == 0), "a DC kernel cannot update on omega / a indices");
  constexpr int NC = DC ? N_ACT : NS;        // columns of HP that are carried
  constexpr int NB = NC / 3;                 // index triples
  // t-th carried triple -> its block number; column c -> its position in Y
  constexpr auto blk = &carried_block<DC>;
  constexpr auto pos = &carried_pos<DC>;
  // issue the measurement loads first; they are consumed after the covariance work
  double z[3], Rdg[3];
  src.z3(st, row, a0, sn, z);
  if (st.r_mode == 1) {
#pragma unroll
    for (int a = 0; a < 3; a++) Rdg[a] = ldg_early(st.R + (long long)(a0 + a) * N + n);
  }
#if RBIS_PARK_STATE == 2
  park_state<PARK_ALL>(P, s);  // the sweep needs none of it; read back below
#endif
  // Y starts as HP = P[idx, :]
  double Y[3][NC];
  {
    Buf<9> b0, b1;
    issue<typename HPRow0<I0>::template Tile<blk(0)>>(P, b0);
    static_for<NB>([&](auto tc) {
      constexpr int t = tc;
      auto& cur = pick<t % 2>(b0, b1);
      auto& nxt = pick<(t + 1) % 2>(b0, b1);
      commit<typename HPRow0<I0>::template Tile<blk(t)>>(cur);
      if constexpr (t + 1 < NB) issue<typename HPRow0<I0>::template Tile<blk(t + 1 < NB ? t + 1 : t)>>(P, nxt);
#pragma unroll
      for (int k = 0; k < 9; k++) Y[k % 3][3 * t + k / 3] = cur.d[k];
    });
  }
  constexpr int J0 = pos(I0);
  // S (symmetric) = R + P[idx, idx]
  double S00, S10, S20, S11, S21, S22;
  if (st.r_mode == 1) {
    S00 = Rdg[0] + Y[0][J0]; S11 = Rdg[1] + Y[1][J0 + 1]; S22 = Rdg[2] + Y[2][J0 + 2];
    S10 = Y[1][J0]; S20 = Y[2][J0]; S21 = Y[2][J0 + 1];
  } else {
    const double* Rm = st.R + row * st.r_stride + a0 + (long long)st.m * a0;
    S00 = __ldg(Rm) + Y[0][J0]; S11 = __ldg(Rm + st.m + 1) + Y[1][J0 + 1]; S22 = __ldg(Rm + 2 * st.m + 2) + Y[2][J0 + 2];
    S10 = __ldg(Rm + 1) + Y[1][J0]; S20 = __ldg(Rm + 2) + Y[2][J0]; S21 = __ldg(Rm + st.m + 2) + Y[2][J0 + 1];
  }
  // LDL^T (no pivoting; S is SPD)
  const double d0 = S00, r0 = 1.0 / d0;
  const double l10 = S10 * r0, l20 = S20 * r0;
  const double d1 = fma(-l10 * l10, d0, S11), r1 = 1.0 / d1;
  const double l21 = fma(-l20 * l10, d0, S21) * r1;
  const double d2 = fma(-l21 * l21, d1, fma(-l20 * l20, d0, S22)), r2 = 1.0 / d2;
  // the reference takes ONE logarithm, of the determinant (rbis.cpp:142); the sum of three is the fallback where the
  // product of the pivots leaves the normal range
  const double pd = d0 * d1 * d2;
  const double logdet = (pd > 1e-290 && pd < 1e290) ? log(pd) : log(d0) + log(d1) + log(d2);
  // Y = L^-1 HP
#pragma unroll
  for (int c = 0; c < NC; c++) {
    Y[1][c] = fma(-l10, Y[0][c], Y[1][c]);
    Y[2][c] = fma(-l21, Y[1][c], fma(-l20, Y[0][c], Y[2][c]));
  }
  // covariance sweep: P[i,j] -= sum_a Y[a][i] * (Y[a][j] / d_a), packed order, tiles of SWEEP_TILE slots
  {
    constexpr int TS = SWEEP_TILE;
    constexpr int NSW = kSweepLen<DC>;
    constexpr int NT = (NSW + TS - 1) / TS;
    Buf<TS> b0, b1;
    issue<SweepRun<DC, 0, (NSW < TS ? NSW : TS)>>(P, b0);
    static_for<NT>([&](auto tc) {
      constexpr int t = tc;
      constexpr int s0 = t * TS;
      constexpr int len = (NSW - s0) < TS ? (NSW - s0) : TS;
      using Cur = SweepRun<DC, s0, len>;
      auto& cur = pick<t % 2>(b0, b1);
      auto& nxt = pick<(t + 1) % 2>(b0, b1);
      // commit / issue on exactly the slots of the tile
      if constexpr (any_tm<Cur>()) tm_wait_ld();
      static_for<len>([&](auto kc) {
        constexpr int k = kc;
        constexpr int i = Cur::row(k), j = Cur::col(k);
        if constexpr (in_tm(i, j)) cur.d[k] = tm_settle(cur.lo[k], cur.hi[k]);
      });
      if constexpr (t + 1 < NT) {
        constexpr int s1 = s0 + TS;
        constexpr int len1 = (NSW - s1) < TS ? (NSW - s1) : TS;
        using Nxt = SweepRun<DC, s1, len1>;
        static_for<len1>([&](auto kc) {
          constexpr int k = kc;
          constexpr int i = Nxt::row(k), j = Nxt::col(k);
          if constexpr (in_tm(i, j)) tm_ld2(P.tm + 2 * tm_index(i, j), nxt.lo[k], nxt.hi[k]);
          else nxt.d[k] = P.Ps[sm_off(sm_index(i, j))];
        });
      }
      static_for<len>([&](auto kc) {
        constexpr int k = kc;
        constexpr int i = Cur::row(k), j = Cur::col(k);
        constexpr int yi = pos(i), yj = pos(j);
        const double v = fma(-Y[0][yi], Y[0][yj] * r0, fma(-Y[1][yi], Y[1][yj] * r1, fma(-Y[2][yi], Y[2][yj] * r2, cur.d[k])));
        if constexpr (MASK) P.template set<i, j>(skip ? cur.d[k] : v);
        else P.template set<i, j>(v);
      });
      RBIS_SCHED_FENCE();
    });
  }
  tm_wait_st();
#if RBIS_PARK_STATE == 2
  unpark_state<PARK_ALL>(P, s);
#endif
  // residual against the current vec (prior + earlier chunks of this update)
  double r[3];
#pragma unroll
  for (int a = 0; a < 3; a++) {
    if (I0 == 6 && st.has_orient) {
      const double dq = (a == 0) ? dquat.x : (a == 1) ? dquat.y : dquat.z;
      const double c0 = (a == 0) ? chi0.x : (a == 1) ? chi0.y : chi0.z;
      r[a] = dq - (s.x[I0 + a] - c0);
    } else {
      r[a] = z[a] - s.x[I0 + a];
    }
  }
  // e = L^-1 r, u = D^-1 e, x += Y^T u
  const double e0 = r[0], e1 = fma(-l10, e0, r[1]), e2 = fma(-l21, e1, fma(-l20, e0, r[2]));
  const double u0 = e0 * r0, u1 = e1 * r1, u2 = e2 * r2;
  static_for<NC>([&](auto cc) {
    constexpr int c = cc;
    constexpr int xc = DC ? act_col(c) : c;
    if constexpr (MASK) s.x[xc] = skip ? s.x[xc] : fma(Y[0][c], u0, fma(Y[1][c], u1, fma(Y[2][c], u2, s.x[xc])));
    else s.x[xc] = fma(Y[0][c], u0, fma(Y[1][c], u1, fma(Y[2][c], u2, s.x[xc])));
  });
  if constexpr (MASK) s.ll = skip ? s.ll : s.ll + (-logdet - fma(e2, u2, fma(e1, u1, e0 * u0)));
  else s.ll += -logdet - fma(e2, u2, fma(e1, u1, e0 * u0));
  if constexpr (NISQ) *nisq += fma(e2, u2, fma(e1, u1, e0 * u0));
}

// Row idx (run time, warp uniform) of the covariance over the carried columns: all loads issued, ONE tensor-memory wait.
template <bool DC>
__device__ __forceinline__ void fetch_row(const Cov& P, int idx, double (&row)[DC ? N_ACT : NS]) {
  constexpr int NC = DC ? N_ACT : NS;
  uint32_t lo[NC], hi[NC];
  bool tm[NC];
  static_for<NC>([&](auto cc) {
    constexpr int c = cc;
    constexpr int col = DC ? act_col(c) : c;
    const int s_ = slot(idx, col);
    const int k = c_place.idx[s_];
    tm[c] = c_place.tm[s_];
    lo[c] = hi[c] = 0;
    row[c] = 0.0;
    if (tm[c]) tm_ld2(P.tm + 2 * k, lo[c], hi[c]);
    else row[c] = P.Ps[sm_off(k)];
  });
  tm_wait_ld();
  static_for<NC>([&](auto cc) {
    constexpr int c = cc;
    const double v = tm_settle(lo[c], hi[c]);
    row[c] = tm[c] ? v : row[c];
  });
}
// g[pos(idx)] for a run-time index (select chain)
template <bool DC>
__device__ __forceinline__ double pick_carried(const double (&g)[DC ? N_ACT : NS], int idx) {
  constexpr int NC = DC ? N_ACT : NS;
  double v = g[0];
  static_for<NC>([&](auto cc) {
    constexpr int c = cc;
    constexpr int col = DC ? act_col(c) : c;
    if (c > 0) v = (idx == col) ? g[c] : v;
  });
  return v;
}
// P -= g g^T r over the carried slots, pipelined tiles (MASK, skip: as in meas3)
template <bool DC, bool MASK = false>
__device__ __forceinline__ void rank1_sweep(Cov& P, const double (&g)[DC ? N_ACT : NS], double r, bool skip = false) {
  constexpr auto pos = &carried_pos<DC>;
  constexpr int TS = SWEEP_TILE;
  constexpr int NSW = kSweepLen<DC>;
  constexpr int NT = (NSW + TS - 1) / TS;
  Buf<TS> b0, b1;
  issue<SweepRun<DC, 0, (NSW < TS ? NSW : TS)>>(P, b0);
  static_for<NT>([&](auto tc) {
    constexpr int t = tc;
    constexpr int s0 = t * TS;
    constexpr int len = (NSW - s0) < TS ? (NSW - s0) : TS;
    using Cur = SweepRun<DC, s0, len>;
    auto& cur = pick<t % 2>(b0, b1);
    auto& nxt = pick<(t + 1) % 2>(b0, b1);
    commit<Cur>(cur);
    if constexpr (t + 1 < NT) {
      constexpr int s1 = s0 + TS;
      constexpr int len1 = (NSW - s1) < TS ? (NSW - s1) : TS;
      issue<SweepRun<DC, s1, len1>>(P, nxt);
    }
    static_for<len>([&](auto kc) {
      constexpr int k = kc;
      constexpr int i = Cur::row(k), j = Cur::col(k);
      if constexpr (MASK) P.template set<i, j>(skip ? cur.d[k] : fma(-g[pos(i)], g[pos(j)] * r, cur.d[k]));
      else P.template set<i, j>(fma(-g[pos(i)], g[pos(j)] * r, cur.d[k]));
    });
    RBIS_SCHED_FENCE();
  });
  tm_wait_st();
}

// meas1: a ONE-ROW chunk on any state index (yaw lock, vicon yaw, altimeter-style updates; and every row of an index set
// that is not an aligned triple when its noise is uncorrelated with the other rows).  The index is a run-time, warp-uniform
// value: the row P[idx, :] is fetched with run-time addressing (15 or 21 loads), everything after that -- the rank-1
// sweep P -= h h^T / s and the state update -- runs over compile-time slots with h in registers.
template <bool DC, bool SYN, bool MASK = false, bool NISQ = false>
__device__ __forceinline__ void meas1(Cov& P, FilterState& s, const StreamDesc& st, const MeasSrc<SYN>& src, int a0, int idx, long long row, long long N,
                                      long long n, long long sn, const V3& dquat, const V3& chi0, bool skip = false,
                                      double* nisq = nullptr) {
  constexpr int NC = DC ? N_ACT : NS;
  constexpr auto pos = &carried_pos<DC>;
  const double z = src.z(st, row, a0, sn);
  const double Rv = (st.r_mode == 1) ? ldg_early(st.R + (long long)a0 * N + n) : __ldg(st.R + row * st.r_stride + a0 + (long long)st.m * a0);
  double h[NC];
  fetch_row<DC>(P, idx, h);
  const double hii = pick_carried<DC>(h, idx);
  const double sv = Rv + hii;
  const double r = 1.0 / sv;
  rank1_sweep<DC, MASK>(P, h, r, skip);
  double rr;
  if (st.has_orient && idx >= 6 && idx <= 8) {
    const int k = idx - 6;
    const double dq = (k == 0) ? dquat.x : (k == 1) ? dquat.y : dquat.z;
    const double c0 = (k == 0) ? chi0.x : (k == 1) ? chi0.y : chi0.z;
    rr = dq - (pick_state(s.x, idx) - c0);
  } else {
    rr = z - pick_state(s.x, idx);
  }
  const double u = rr * r;
  static_for<NC>([&](auto cc) {
    constexpr int c = cc;
    constexpr int xc = DC ? act_col(c) : c;
    if constexpr (MASK) s.x[xc] = skip ? s.x[xc] : fma(h[c], u, s.x[xc]);
    else s.x[xc] = fma(h[c], u, s.x[xc]);
  });
  if constexpr (MASK) s.ll = skip ? s.ll : s.ll + (-log(sv) - rr * u);
  else s.ll += -log(sv) - rr * u;
  if constexpr (NISQ) *nisq += rr * u;
}

// meas_block: a chunk of M (2..9) rows with CORRELATED noise on any indices.  The host factors R_block = L D L^T; with
// z' = L^-1 z, H' = L^-1 H the block is M scalar measurements with uncorrelated noise D, applied one after the other
// (the same posterior and the same log-likelihood as the reference's single update, rbis.cpp:124-143, by the chain rule).
// Row a of H' combines the covariance rows idx_b, b <= a, so everything lives in registers: g = P H'_a^T (15 / 21
// doubles), a rank-1 sweep over compile-time slots, the state update.  No local-memory arrays, no separate kernel variant.
// Only the BLOCKS = true kernel variants contain it.
template <bool DC, bool SYN, bool MASK = false, bool NISQ = false>
__device__ __forceinline__ void meas_block(Cov& P, FilterState& s, const StreamDesc& st, const MeasSrc<SYN>& src, int a0, int M, long long row, long long N,
                                           long long n, long long sn, const V3& dquat, const V3& chi0, bool skip = false,
                                           double* nisq = nullptr) {
  constexpr int NC = DC ? N_ACT : NS;
  const double* W = st.R + row * st.r_stride + RS_W;
  const double* Dg = st.R + row * st.r_stride + RS_D;
  (void)N; (void)n;
  for (int a = 0; a < M; a++) {
    double g[NC];
    static_for<NC>([&](auto cc) { g[cc] = 0.0; });
    for (int b = 0; b <= a; b++) {
      const double w = __ldg(W + (a0 + a) * MAX_MEAS + (a0 + b));
      double rowv[NC];
      fetch_row<DC>(P, st.idx[a0 + b], rowv);
      static_for<NC>([&](auto cc) { g[cc] = fma(w, rowv[cc], g[cc]); });
    }
    double sv = __ldg(Dg + a0 + a), rp = 0.0;
    for (int b = 0; b <= a; b++) {
      const double w = __ldg(W + (a0 + a) * MAX_MEAS + (a0 + b));
      const int ib = st.idx[a0 + b];
      sv = fma(w, pick_carried<DC>(g, ib), sv);
      const double xi = pick_state(s.x, ib);
      double rb;
      if (st.has_orient && ib >= 6 && ib <= 8) {
        const int k = ib - 6;
        const double dq = (k == 0) ? dquat.x : (k == 1) ? dquat.y : dquat.z;
        const double c0 = (k == 0) ? chi0.x : (k == 1) ? chi0.y : chi0.z;
        rb = dq - (xi - c0);
      } else {
        rb = src.template z<false>(st, row, a0 + b, sn) - xi;
      }
      rp = fma(w, rb, rp);
    }
    const double r = 1.0 / sv;
    rank1_sweep<DC, MASK>(P, g, r, skip);
    const double u = rp * r;
    static_for<NC>([&](auto cc) {
      constexpr int c = cc;
      constexpr int xc = DC ? act_col(c) : c;
      if constexpr (MASK) s.x[xc] = skip ? s.x[xc] : fma(g[c], u, s.x[xc]);
      else s.x[xc] = fma(g[c], u, s.x[xc]);
    });
    if constexpr (MASK) s.ll = skip ? s.ll : s.ll + (-log(sv) - rp * u);
    else s.ll += -log(sv) - rp * u;
    if constexpr (NISQ) *nisq += rp * u;
  }
}

// state half of rbisApplyDelta for a whole measurement op: dstate = RBIS(K r) then addState.
// s.x already holds prior + K r (all chunks); chi0 is the prior vec chi.
__device__ __forceinline__ void meas_finish(FilterState& s, const V3& chi0, double chi_tol, int ctor_folds_chi,
                                            int renorm) {
  V3 dchi{s.x[6] - chi0.x, s.x[7] - chi0.y, s.x[8] - chi0.z};
  s.x[6] = chi0.x; s.x[7] = chi0.y; s.x[8] = chi0.z;
  Q4 dq{1, 0, 0, 0};
  const double n2 = sumsq3(dchi.x, dchi.y, dchi.z);
  const bool folded = ctor_folds_chi && (n2 > chi_tol * chi_tol);
  if (folded) dq = qexp2(dchi, n2);
  add_state_tail(s, dchi, folded, dq, chi_tol, renorm);
}

// ---- whole-covariance transfers between the on-chip layout and a [231][stride] global array ----
constexpr int XFER_TILE = 11;  // 231 = 21 * 11
__device__ __forceinline__ void cov_load_all(Cov& P, const double* __restrict__ src, long long stride) {
  static_for<NP>([&](auto sc) {
    constexpr int s_ = sc;
    P.template set<row_of_slot(s_), col_of_slot(s_)>(src[(long long)s_ * stride]);
  });
  tm_wait_st();
}
__device__ __forceinline__ void cov_store_all(const Cov& P, double* __restrict__ dst, long long stride, bool active) {
  static_for<NP / XFER_TILE>([&](auto tc) {
    constexpr int s0 = tc * XFER_TILE;
    Buf<XFER_TILE> b;
    issue<SlotRun<s0, XFER_TILE>>(P, b);
    commit<SlotRun<s0, XFER_TILE>>(b);
    if (active) {
#pragma unroll
      for (int k = 0; k < XFER_TILE; k++) dst[(long long)(s0 + k) * stride] = b.d[k];
    }
  });
}

// DC variants: only the active slots live on chip
__device__ __forceinline__ void cov_load_active(Cov& P, const double* __restrict__ src, long long stride) {
  static_for<NP_ACT>([&](auto kc) {
    constexpr int s_ = kAct.s[kc];
    P.template set<row_of_slot(s_), col_of_slot(s_)>(src[(long long)s_ * stride]);
  });
  tm_wait_st();
}
__device__ __forceinline__ void cov_store_active(const Cov& P, double* __restrict__ dst, long long stride, bool active) {
  constexpr int TILE = 12;  // 120 = 10 * 12
  static_for<NP_ACT / TILE>([&](auto tc) {
    constexpr int k0 = tc * TILE;
    Buf<TILE> b;
    issue<ActRun<k0, TILE>>(P, b);
    commit<ActRun<k0, TILE>>(b);
    if (active) {
      static_for<TILE>([&](auto kc) {
        constexpr int s_ = kAct.s[k0 + kc];
        dst[(long long)s_ * stride] = b.d[kc];
      });
    }
  });
}
// the (omega,omega) and (a,a) blocks as every IMU step leaves them (rbis.cpp:120-121), written to a [231][stride] array
__device__ __forceinline__ void store_overwritten_blocks(double* __restrict__ dst, long long stride, double q_gyro, double q_accel) {
  static_for<12>([&](auto kc) {
    constexpr int s_ = kAct.blk[kc];
    constexpr int i = row_of_slot(s_), j = col_of_slot(s_);
    dst[(long long)s_ * stride] = (i != j) ? 0.0 : (j < 3 ? q_gyro : q_accel);
  });
}

// ---- innovation sets (see InnovK) ----
// P(idx, idx) for a run-time, warp-uniform index: the addressing of fetch_row
__device__ __forceinline__ double cov_diag(const Cov& P, int idx) {
  const int s_ = slot(idx, idx);
  const int k = c_place.idx[s_];
  const bool tm = c_place.tm[s_];
  uint32_t lo = 0, hi = 0;
  double v = 0.0;
  if (tm) tm_ld2(P.tm + 2 * k, lo, hi);
  else v = P.Ps[sm_off(k)];
  tm_wait_ld();
  const double t = tm_settle(lo, hi);
  return tm ? t : v;
}
__device__ __forceinline__ double innov_nan() { return __longlong_as_double(0x7ff8000000000000ll); }
// R(a, a) of a stream row: the shared table, the row's table (r_stride) or the per-filter diagonal [m][N]
__device__ __forceinline__ double r_diag(const StreamDesc& st, int a, long long row, long long N, long long n) {
  return st.r_mode == 1 ? __ldg(st.R + (long long)a * N + n) : __ldg(st.R + row * st.r_stride + a + (long long)st.m * a);
}
// y_a = z_a - x-[idx_a] (the component of dquat at the chi indices of an orientation stream), as the chunks form their
// residuals before any chunk has run
template <bool SYN>
__device__ __forceinline__ double innov_y(const FilterState& s, const StreamDesc& st, const MeasSrc<SYN>& src, int a, long long row,
                                          long long sn, const V3& dquat) {
  const int i = st.idx[a];
  if (st.has_orient && i >= 6 && i <= 8) return i == 6 ? dquat.x : i == 7 ? dquat.y : dquat.z;
  return src.template z<false>(st, row, a, sn) - pick_state(s.x, i);
}
// y and S(a,a) of this lane's filter at the start of a MEAS op, one coalesced store each, straight to the output (nothing
// is held across the chunks); NaN for a filter that skips the row.  m, idx and the fields are warp uniform, so the
// tensor-memory loads stay warp-aligned.
template <bool SYN>
__device__ __forceinline__ void innov_begin(const InnovK& iv, const Cov& P, const FilterState& s, const StreamDesc& st, const MeasSrc<SYN>& src,
                                            long long row, long long N, long long n, long long sn, const V3& dquat, bool active, bool skip) {
  double* const d = iv.out + row * iv.k * N + n;
  const int m = st.m;
  const int oy = iv.fields & INNOV_NIS, os = oy + ((iv.fields & INNOV_Y) ? m : 0);
  for (int a = 0; a < m; a++) {
    if (iv.fields & INNOV_Y) {
      const double y = innov_y<SYN>(s, st, src, a, row, sn, dquat);
      if (active) d[(long long)(oy + a) * N] = skip ? innov_nan() : y;
    }
    if (iv.fields & INNOV_S_DIAG) {
      const double v = cov_diag(P, st.idx[a]) + r_diag(st, a, row, N, n);
      if (active) d[(long long)(os + a) * N] = skip ? innov_nan() : v;
    }
  }
}

// ---- RBIS_OP_RECORD (see RecK) ----
// record field F < 26: the state in registers
template <int F>
__device__ __forceinline__ double rec_state_field(const FilterState& s) {
  if constexpr (F < NS) return s.x[F];
  else if constexpr (F == 21) return s.qw;
  else if constexpr (F == 22) return s.qx;
  else if constexpr (F == 23) return s.qy;
  else if constexpr (F == 24) return s.qz;
  else return s.ll;
}
// The chosen fields of this lane's filter, with the values an RBIS_OP_SNAPSHOT at the same position stores: the diagonal
// from shared / tensor memory through the slot helpers; in the DC kernels the (omega,omega) / (a,a) diagonals as
// store_overwritten_blocks writes them, or the parked p.P values before the first IMU step.  `fields` is uniform, so the
// tensor-memory loads stay warp-aligned; each chosen field is one coalesced 8-byte store per lane.
template <bool DC>
__device__ __forceinline__ void record_fields(const KParams& p, const Cov& P, const FilterState& s, long long row, long long n, bool active,
                                              bool imu_seen) {
  const long long N = p.N;
  const unsigned long long fields = p.rec.fields;
  double* const d = p.rec.out + row * p.rec.k * N + n;
  static_for<REC_FIELDS>([&](auto fc) {
    constexpr int f = fc;
    if (!((fields >> f) & 1ull)) return;
    double v;
    if constexpr (f < 26) {
      v = rec_state_field<f>(s);
    } else {
      constexpr int i = f - 26, s_ = slot(i, i);
      if constexpr (DC && !is_act(i)) {
        v = imu_seen ? __ldg((i < 3 ? p.q_gyro : p.q_accel) + n) : p.P[(long long)s_ * N + n];
      } else {
        Buf<1> b;
        issue<SlotRun<s_, 1>>(P, b);
        commit<SlotRun<s_, 1>>(b);
        v = b.d[0];
      }
    }
    if (active) d[(long long)__popcll(fields & ((1ull << f) - 1)) * N] = v;
  });
  // ---- covariance blocks: the values of an RBIS_OP_SNAPSHOT's slot(i, j), loaded through the tiles SNAPSHOT uses.  cb is
  // uniform, so a tile without a selected slot is skipped by the whole warp and the tensor-memory loads stay warp-aligned.
  const unsigned cb = p.rec_cov_blocks;
  if (!cb) return;
  double* const dc = d + (long long)__popcll(fields) * N;
  auto sel = [&](int i, int j) { return ((cb >> (i / 3)) & (cb >> (j / 3)) & 1u) != 0; };
  auto put = [&](int i, int j, double v) {  // i <= j, both blocks selected
    const int ii = rec_cov_index(cb, i), jj = rec_cov_index(cb, j);
    if (active) dc[(long long)(jj * (jj + 1) / 2 + ii) * N] = v;
  };
  if constexpr (DC) {
    constexpr int TILE = 12;  // the tiles of cov_store_active
    static_for<NP_ACT / TILE>([&](auto tc) {
      constexpr int k0 = tc * TILE;
      bool any = false;
      static_for<TILE>([&](auto kc) { any = any || sel(row_of_slot(kAct.s[k0 + kc]), col_of_slot(kAct.s[k0 + kc])); });
      if (!any) return;
      Buf<TILE> b;
      issue<ActRun<k0, TILE>>(P, b);
      commit<ActRun<k0, TILE>>(b);
      static_for<TILE>([&](auto kc) {
        constexpr int s_ = kAct.s[k0 + kc];
        constexpr int i = row_of_slot(s_), j = col_of_slot(s_);
        if (sel(i, j)) put(i, j, b.d[kc]);
      });
    });
    static_for<N_REST>([&](auto kc) {
      constexpr int s_ = kAct.rest[kc];
      constexpr int i = row_of_slot(s_), j = col_of_slot(s_);
      if (sel(i, j)) put(i, j, 0.0);
    });
    static_for<12>([&](auto kc) {
      constexpr int s_ = kAct.blk[kc];
      constexpr int i = row_of_slot(s_), j = col_of_slot(s_);
      if (sel(i, j))
        put(i, j, imu_seen ? ((i != j) ? 0.0 : __ldg((j < 3 ? p.q_gyro : p.q_accel) + n)) : p.P[(long long)s_ * N + n]);
    });
  } else {
    static_for<NP / XFER_TILE>([&](auto tc) {  // the tiles of cov_store_all
      constexpr int s0 = tc * XFER_TILE;
      bool any = false;
      static_for<XFER_TILE>([&](auto kc) { any = any || sel(row_of_slot(s0 + kc), col_of_slot(s0 + kc)); });
      if (!any) return;
      Buf<XFER_TILE> b;
      issue<SlotRun<s0, XFER_TILE>>(P, b);
      commit<SlotRun<s0, XFER_TILE>>(b);
      static_for<XFER_TILE>([&](auto kc) {
        constexpr int i = row_of_slot(s0 + kc), j = col_of_slot(s0 + kc);
        if (sel(i, j)) put(i, j, b.d[kc]);
      });
    });
  }
}

// ------------------------------------------------------------------------------------------------
// The fused kernel: every lane loads its filter, runs the whole op program, stores it back.
// BLOCKS = true variants also contain meas1 and meas_block (one-row chunks, chunks of correlated rows); they are launched
// only for programs that have such chunks, so that the common program (aligned triples only) keeps its registers and
// code layout: merely compiling the two paths into it costs 3-8 %.
// ------------------------------------------------------------------------------------------------
// DC = true is launched when the host has verified that every filter's omega / a couplings are exactly zero and no
// measurement of the program indexes omega or a (see "decoupled filters" above).
// SYN = true: the input rows are drawn inside the kernel (KParams::syn, mode-1 generator) instead of being read from HBM.
// REC = true: the program has RBIS_OP_RECORD ops (KParams::rec); launched only then, so that other programs keep their code.
// MASK = true: some stream of the program has RBIS_STREAM_SKIP_NAN_ROWS (KParams::skip_nan_streams); instantiated with BLOCKS
// only (and without SYN), launched only for such programs.
// INNOV = true (with REC): a MEAS op of the program writes an innovation set (KParams::innov); launched only then, so that
// programs that only record keep the code of the REC instantiations.
template <bool BLOCKS, bool DC = false, bool SYN = false, bool REC = false, bool MASK = false, bool INNOV = false>
__global__ void __launch_bounds__(TPB, 1) rbis_fused_kernel(const __grid_constant__ KParams p) {
  static_assert(!MASK || (BLOCKS && !SYN), "MASK instantiations have the one-row / correlated-block paths and read z from HBM");
  static_assert(!INNOV || REC, "INNOV instantiations are REC instantiations with the innovation path");
  extern __shared__ __align__(16) double smem[];
  __shared__ uint32_t tm_base_s;
  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  // ---- tensor memory: all 512 columns; warp w owns lanes 32*(w%4).. and columns TM_COLS*(w/4).. ----
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"((uint32_t)__cvta_generic_to_shared(&tm_base_s)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tm_base = tm_base_s;

  const long long N = p.N;
  long long n = ((long long)blockIdx.x + p.block_offset) * TPB + tid;
  const bool active = n < N;
  if (!active) n = N - 1;  // idle lanes shadow the last filter and never store

  Cov P;
  P.Ps = smem + tid;
  P.tm = tm_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)((warp >> 2) * TM_COLS);
  FilterState s;
  static_for<NS>([&](auto i) { s.x[i] = p.vec[(long long)i * N + n]; });
  s.qw = p.quat[n]; s.qx = p.quat[N + n]; s.qy = p.quat[2 * N + n]; s.qz = p.quat[3 * N + n];
  s.ll = p.loglik[n];
  if constexpr (DC) cov_load_active(P, p.P + n, N);
  else cov_load_all(P, p.P + n, N);
  bool imu_seen = false;  // DC: an IMU step ran since the (omega,omega) / (a,a) blocks in p.P were current

  auto load_op = [&](long long i) {
    Op o;
    long long w0, w1;  // Op is 24 bytes: three 8-byte loads
    asm volatile("ld.global.nc.s64 %0, [%1];" : "=l"(w0) : "l"(reinterpret_cast<const long long*>(p.ops + i)));
    asm volatile("ld.global.nc.s64 %0, [%1];" : "=l"(w1) : "l"(reinterpret_cast<const long long*>(p.ops + i) + 1));
    o.kind = (int)(w0 & 0xffffffffll); o.stream = (int)(w0 >> 32); o.row = w1;
    asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(o.dt) : "l"(&p.ops[i].dt));
    return o;
  };
  const long long imu_n = p.imu_map ? (long long)__ldg(p.imu_map + n) : n;
  // SYN: the filter's part of the counter key and its IMU noise levels
  unsigned long long syn_kf = 0;
  double syn_sg = 0.0, syn_sa = 0.0;
  if constexpr (SYN) {
    syn_kf = p.syn.seed ^ ((unsigned long long)(p.syn.first_filter + n) * SYN_K1);
    syn_sg = p.syn.sigma_gyro >= 0 ? p.syn.sigma_gyro : sqrt(__ldg(p.q_gyro + n) / p.syn.dt);
    syn_sa = p.syn.sigma_accel >= 0 ? p.syn.sigma_accel : sqrt(__ldg(p.q_accel + n) / p.syn.dt);
  }
  Op op_next = load_op(0);
  for (long long oi = 0; oi < p.n_ops; oi++) {
    const Op op = op_next;
    if (oi + 1 < p.n_ops) op_next = load_op(oi + 1);  // fetched one op ahead: its latency hides behind this op
    if (op.kind == OP_IMU) {
      // ---- IMU process step ----
      const double* base = p.imu + op.row * 6 * p.imu_cols + imu_n;
      const long long Ni = p.imu_cols;
      V3 gyro, acc;
      QNoise qn;
      auto load_q = [&]() {
        qn.q_gyro = ldg_early(p.q_gyro + n); qn.q_accel = ldg_early(p.q_accel + n);
        qn.q_gyro_bias = ldg_early(p.q_gyro_bias + n); qn.q_accel_bias = ldg_early(p.q_accel_bias + n);
      };
      auto load_inputs = [&]() {
        if constexpr (SYN) {
          const unsigned long long kfs = syn_kf ^ ((unsigned long long)__ldg(p.syn.imu_step + op.row) * SYN_K2);
          const double* mu = p.syn.imu_mean + op.row * 6;
          double nn[6];
          syn_normals_k<1, 6>(kfs, 0u, nn);
          gyro = {fma(syn_sg, nn[0], __ldg(mu)), fma(syn_sg, nn[1], __ldg(mu + 1)), fma(syn_sg, nn[2], __ldg(mu + 2))};
          acc = {fma(syn_sa, nn[3], __ldg(mu + 3)), fma(syn_sa, nn[4], __ldg(mu + 4)), fma(syn_sa, nn[5], __ldg(mu + 5))};
        } else {
          gyro = {ldg_early(base), ldg_early(base + Ni), ldg_early(base + 2 * Ni)};
          acc = {ldg_early(base + 3 * Ni), ldg_early(base + 4 * Ni), ldg_early(base + 5 * Ni)};
        }
      };
#if !RBIS_LATE_LOADS
      load_inputs();
      load_q();
#endif
      const double dt = op.dt;
      const Q4 q{s.qw, s.qx, s.qy, s.qz};
      // the rotation matrix is needed for R dt anyway: q^-1 g_vec = -g_val * (third row of R) and q v = R v come from it
      // (equal to the quaternion forms up to rounding and to |q|^2 - 1, which the reference lets drift at 1e-16 per step)
      const double tx_ = 2 * q.x, ty_ = 2 * q.y, tz_ = 2 * q.z;
      const double twx_ = tx_ * q.w, twy_ = ty_ * q.w, twz_ = tz_ * q.w;
      const double txx_ = tx_ * q.x, txy_ = ty_ * q.x, txz_ = tz_ * q.x;
      const double tyy_ = ty_ * q.y, tyz_ = tz_ * q.y, tzz_ = tz_ * q.z;
      const double R00 = 1 - (tyy_ + tzz_), R01 = txy_ - twz_, R02 = txz_ + twy_;
      const double R10 = txy_ + twz_, R11 = 1 - (txx_ + tzz_), R12 = tyz_ - twx_;
      const double R20 = txz_ - twy_, R21 = tyz_ + twx_, R22 = 1 - (txx_ + tyy_);
      const V3 gb{-p.g_val * R20, -p.g_val * R21, -p.g_val * R22};
      {
        const double vx = s.x[3], vy = s.x[4], vz = s.x[5];
        s.x[9] += fma(R02, vz, fma(R01, vy, R00 * vx)) * dt;
        s.x[10] += fma(R12, vz, fma(R11, vy, R10 * vx)) * dt;
        s.x[11] += fma(R22, vz, fma(R21, vy, R20 * vx)) * dt;
      }
      Lin L;
      L.v = {s.x[3], s.x[4], s.x[5]};
      L.wd = {s.x[0] * dt, s.x[1] * dt, s.x[2] * dt};  // omega of the PRIOR state (previous sample)
      L.vd = {L.v.x * dt, L.v.y * dt, L.v.z * dt};
      L.gd = {gb.x * dt, gb.y * dt, gb.z * dt};
      L.dt = dt;
      L.Rd[0] = R00 * dt; L.Rd[1] = R01 * dt; L.Rd[2] = R02 * dt;
      L.Rd[3] = R10 * dt; L.Rd[4] = R11 * dt; L.Rd[5] = R12 * dt;
      L.Rd[6] = R20 * dt; L.Rd[7] = R21 * dt; L.Rd[8] = R22 * dt;
#if RBIS_PARK_STATE == 2
      park_state<PARK_COV>(P, s);
#endif
      imu_seen = true;
      cov_propagate<DC>(P, L,
                    [&]() {
#if RBIS_LATE_LOADS
                      load_q();
#endif
                      return qn;
                    },
                    [&]() {
#if RBIS_LATE_LOADS
                      load_inputs();
#endif
                    });
#if RBIS_PARK_STATE == 2
      unpark_state<PARK_COV>(P, s);
#endif
      state_propagate(s, gyro, acc, dt, gb, p.chi_tol, p.renorm);
    } else if (op.kind == OP_MEAS) {
      // ---- indexed / indexed-plus-orientation measurement ----
      const StreamDesc& st = p.streams[op.stream];
      const long long sn = st.map ? (long long)__ldg(st.map + n) : n;
      MeasSrc<SYN> src{};
      if constexpr (SYN) {
        src.ss = &p.syn.st[op.stream];
        src.kfs = syn_kf ^ ((unsigned long long)__ldg(src.ss->step + op.row) * SYN_K2);
      }
      // MASK: a filter whose row is missing runs the sweeps like every lane and keeps its values (see row_missing)
      bool skip = false;
      if constexpr (MASK) {
        if ((p.skip_nan_streams >> op.stream) & 1u) skip = row_missing(st, op.row, sn);
      }
      V3 dquat{0, 0, 0};
      if (st.has_orient) dquat = subtract_quats(src.quat(st, op.row, sn), {s.qw, s.qx, s.qy, s.qz});  // rbis.cpp:199
      // INNOV: an innovation set on this stream (uniform branch) gets y and S(a,a) now and the NIS after the chunks
      double nisq = 0.0;
      if constexpr (INNOV) {
        if (p.innov[op.stream].out) innov_begin<SYN>(p.innov[op.stream], P, s, st, src, op.row, N, n, sn, dquat, active, skip);
      }
      const V3 chi0{s.x[6], s.x[7], s.x[8]};
      for (int ci = 0; ci < st.n_chunks; ci++) {
        const int a0 = st.chunk_start[ci];
        const int fast = st.chunk_fast[ci];
        switch (fast) {
          case 0: if constexpr (!DC) meas3<0, false, SYN, MASK, INNOV>(P, s, st, src, a0, op.row, N, n, sn, dquat, chi0, skip, &nisq); break;
          case 3: meas3<3, DC, SYN, MASK, INNOV>(P, s, st, src, a0, op.row, N, n, sn, dquat, chi0, skip, &nisq); break;
          case 6: meas3<6, DC, SYN, MASK, INNOV>(P, s, st, src, a0, op.row, N, n, sn, dquat, chi0, skip, &nisq); break;
          case 9: meas3<9, DC, SYN, MASK, INNOV>(P, s, st, src, a0, op.row, N, n, sn, dquat, chi0, skip, &nisq); break;
          case 12: if constexpr (!DC) meas3<12, false, SYN, MASK, INNOV>(P, s, st, src, a0, op.row, N, n, sn, dquat, chi0, skip, &nisq); break;
          case 15: meas3<15, DC, SYN, MASK, INNOV>(P, s, st, src, a0, op.row, N, n, sn, dquat, chi0, skip, &nisq); break;
          case 18: meas3<18, DC, SYN, MASK, INNOV>(P, s, st, src, a0, op.row, N, n, sn, dquat, chi0, skip, &nisq); break;
          default:
            if constexpr (BLOCKS) {
              if (fast >= 100) {  // one-row chunk on state index fast - 100
                meas1<DC, SYN, MASK, INNOV>(P, s, st, src, a0, fast - 100, op.row, N, n, sn, dquat, chi0, skip, &nisq);
              } else {            // correlated rows: decorrelated scalar updates
                meas_block<DC, SYN, MASK, INNOV>(P, s, st, src, a0, st.chunk_len[ci], op.row, N, n, sn, dquat, chi0, skip, &nisq);
              }
            }
            break;
        }
      }
      if constexpr (INNOV) {
        const InnovK& iv = p.innov[op.stream];
        if (iv.out && (iv.fields & INNOV_NIS) && active) iv.out[op.row * iv.k * N + n] = skip ? innov_nan() : nisq;
      }
      if (!MASK || !skip) meas_finish(s, chi0, p.chi_tol, p.ctor_folds_chi, p.renorm);
    } else if (op.kind == OP_SNAPSHOT) {
      // ---- snapshot into ring slot ----
      double* d = p.snap + op.row * SNAP_ROWS * N + n;
      if (active) {
        static_for<NS>([&](auto i) { d[(long long)i * N] = s.x[i]; });
        d[21 * N] = s.qw; d[22 * N] = s.qx; d[23 * N] = s.qy; d[24 * N] = s.qz;
        d[25 * N] = s.ll;
      }
      if constexpr (DC) {
        double* dc = d + 26 * N;
        cov_store_active(P, dc, N, active);
        if (active) {
          static_for<N_REST>([&](auto kc) {
            constexpr int s_ = kAct.rest[kc];
            dc[(long long)s_ * N] = 0.0;
          });
          if (imu_seen) store_overwritten_blocks(dc, N, __ldg(p.q_gyro + n), __ldg(p.q_accel + n));
          else static_for<12>([&](auto kc) {
            constexpr int s_ = kAct.blk[kc];
            dc[(long long)s_ * N] = p.P[(long long)s_ * N + n];
          });
        }
      } else {
        cov_store_all(P, d + 26 * N, N, active);
      }
    } else {
      if constexpr (REC) {
        if (op.kind == OP_RECORD) {
          // ---- record the chosen fields into record row op.row ----
          record_fields<DC>(p, P, s, op.row, n, active, imu_seen);
          continue;
        }
      }
      // ---- restore from ring slot ----
      const double* d = p.snap + op.row * SNAP_ROWS * N + n;
      static_for<NS>([&](auto i) { s.x[i] = d[(long long)i * N]; });
      s.qw = d[21 * N]; s.qx = d[22 * N]; s.qy = d[23 * N]; s.qz = d[24 * N];
      s.ll = d[25 * N];
      if constexpr (DC) {
        const double* dc = d + 26 * N;
        cov_load_active(P, dc, N);
        // the slot's (omega,omega) / (a,a) blocks become the current ones: parked in p.P (this lane's own column)
        if (active) static_for<12>([&](auto kc) {
          constexpr int s_ = kAct.blk[kc];
          p.P[(long long)s_ * N + n] = dc[(long long)s_ * N];
        });
        imu_seen = false;
      } else {
        cov_load_all(P, d + 26 * N, N);
      }
    }
  }

  if (active) {
    static_for<NS>([&](auto i) { p.vec[(long long)i * N + n] = s.x[i]; });
    p.quat[n] = s.qw; p.quat[N + n] = s.qx; p.quat[2 * N + n] = s.qy; p.quat[3 * N + n] = s.qz;
    p.loglik[n] = s.ll;
  }
  if constexpr (DC) {
    cov_store_active(P, p.P + n, N, active);
    if (active && imu_seen) store_overwritten_blocks(p.P + n, N, __ldg(p.q_gyro + n), __ldg(p.q_accel + n));
  } else {
    cov_store_all(P, p.P + n, N, active);
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tm_base) : "memory");
}

#ifndef RBIS_FUSED_ONLY
// ------------------------------------------------------------------------------------------------
// layout conversion: full column-major 441 <-> packed upper 231 (both [k][N])
// ------------------------------------------------------------------------------------------------
__global__ void pack_cov_kernel(const double* __restrict__ full, double* __restrict__ packed, long long N) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  for (int j = 0; j < NS; j++)
    for (int i = 0; i <= j; i++) packed[(long long)slot(i, j) * N + n] = full[(long long)(i + NS * j) * N + n];
}
__global__ void unpack_cov_kernel(const double* __restrict__ packed, double* __restrict__ full, long long N) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  for (int j = 0; j < NS; j++)
    for (int i = 0; i < NS; i++) full[(long long)(i + NS * j) * N + n] = packed[(long long)slot(i, j) * N + n];
}
// flag[0] |= 1 when any filter has a non-zero coupling between {omega, a} and the rest (kAct.rest slots) in a
// [231][N] packed covariance.  -0.0 counts as zero; NaN as non-zero.
__global__ void coupling_check_kernel(const double* __restrict__ packed, long long N, int* __restrict__ flag) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  bool nz = false;
  if (n < N) {
    for (int k = 0; k < N_REST; k++) nz = nz || !(packed[(long long)c_act.rest[k] * N + n] == 0.0);
  }
  if (__any_sync(0xffffffffu, nz) && (threadIdx.x & 31) == 0) atomicOr(flag, 1);
}
__global__ void fill_kernel(double* __restrict__ dst, double v, long long count) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) dst[i] = v;
}
#endif  // RBIS_FUSED_ONLY

}  // namespace rbisk
#endif  // include guard (default configuration)
