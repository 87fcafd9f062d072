// rbis_stats.cuh -- ensemble statistics (fixed-order chunk reduction) and FP64 peak microbenchmarks.
//
// Error definition: SE/noise_id/noise_id.cpp:37-38  (e = est; e.subtractState(truth); e.quatToChi()),
// NEES over velocity + chi + position (the active set of SE/noise_id/roll_forward.cpp:54-57).
#pragma once
#include "rbis_kernels.cuh"

namespace rbisk {

constexpr int NSTAT = 96;
constexpr int NPF = 23;  // per-filter outputs: e[21], NEES, loglik

// Where stats_kernel reads its filters: the live arrays or a snapshot slot ([21][N] vec, [4][N] quat, packed [231][N]
// covariance, [N] loglik; one table, gridDim.y = 1) ...
struct StatsArrays {
  const double *vec, *quat, *P, *loglik;
  __device__ __forceinline__ double x(int f, long long n, long long N) const {  // record field f < 26 (see RecK)
    return f < 21 ? vec[(long long)f * N + n] : f < 25 ? quat[(long long)(f - 21) * N + n] : loglik[n];
  }
  __device__ __forceinline__ double cov(int i, int j, long long n, long long N) const {  // P(3 + i, 3 + j), i <= j < 9
    return P[(long long)slot(3 + i, 3 + j) * N + n];
  }
};
// ... or record rows ([rows][k][N], the layout of RecK): row blockIdx.y of `rows`, one table per row.  Fields 0..25 sit at
// positions 0..25; the covariance blocks include v, chi and p, so P(3 + i, 3 + j) is at kf + jj (jj + 1) / 2 + ii with
// ii = base + i, jj = base + j (base = 3 when the omega block is recorded too).
struct StatsRecords {
  const double* rows;
  long long k;
  int kf, base;  // popcount(fields); packed covariance index of state index 3
  __device__ __forceinline__ double x(int f, long long n, long long N) const {
    return rows[((long long)blockIdx.y * k + f) * N + n];
  }
  __device__ __forceinline__ double cov(int i, int j, long long n, long long N) const {
    const int ii = base + i, jj = base + j;
    return rows[((long long)blockIdx.y * k + kf + jj * (jj + 1) / 2 + ii) * N + n];
  }
};

// One CTA per chunk of blockDim.x filters (and per table: blockIdx.y, with truth [21] / [4] and chunks [gridDim.x][96] per
// table).  Each statistic is reduced with the same fixed binary tree (stride blockDim/2 ... 1) so the result depends on
// nothing but the per-filter values and the chunk size: it is identical for any GPU count, for each source, and
// reproducible on the host.
template <class Src>
__global__ void __launch_bounds__(1024) stats_kernel(const Src src, const double* __restrict__ tvec, const double* __restrict__ tquat,
                                                     int per_filter, long long N, double* __restrict__ out_pf, double* __restrict__ out_chunks) {
  extern __shared__ double red[];
  const int t = threadIdx.x;
  const long long n = (long long)blockIdx.x * blockDim.x + t;
  const bool live = n < N;
  tvec += (long long)blockIdx.y * 21;
  tquat += (long long)blockIdx.y * 4;
  out_chunks += (long long)blockIdx.y * gridDim.x * NSTAT;
  double val[48];
#pragma unroll
  for (int k = 0; k < 48; k++) val[k] = 0.0;
  if (live) {
    double e[NS];
#pragma unroll
    for (int i = 0; i < NS; i++) e[i] = src.x(i, n, N) - (per_filter ? tvec[(long long)i * N + n] : tvec[i]);
    const Q4 q{src.x(21, n, N), src.x(22, n, N), src.x(23, n, N), src.x(24, n, N)};
    const Q4 tq = per_filter ? Q4{tquat[n], tquat[N + n], tquat[2 * N + n], tquat[3 * N + n]}
                             : Q4{tquat[0], tquat[1], tquat[2], tquat[3]};
    const V3 dchi = subtract_quats(q, tq);  // Log(truth^-1 * est)
    e[6] = dchi.x; e[7] = dchi.y; e[8] = dchi.z;
    // NEES over indices 3..11: Cholesky of the 9x9 block, forward solve
    double L[9][9];
#pragma unroll
    for (int j = 0; j < 9; j++)
#pragma unroll
      for (int i = 0; i <= j; i++) L[j][i] = src.cov(i, j, n, N);  // lower: L[row][col]
    double y[9];
    double nees = 0;
#pragma unroll
    for (int j = 0; j < 9; j++) {
      double d = L[j][j];
#pragma unroll
      for (int k = 0; k < j; k++) d -= L[j][k] * L[j][k];
      d = sqrt(d);
      L[j][j] = d;
      const double rd = 1.0 / d;
#pragma unroll
      for (int i = j + 1; i < 9; i++) {
        double v = L[i][j];
#pragma unroll
        for (int k = 0; k < j; k++) v -= L[i][k] * L[j][k];
        L[i][j] = v * rd;
      }
      double v = e[3 + j];
#pragma unroll
      for (int k = 0; k < j; k++) v -= L[j][k] * y[k];
      y[j] = v * rd;
      nees += y[j] * y[j];
    }
    const double ll = src.x(25, n, N);
    bool finite = isfinite(nees) && isfinite(ll);
#pragma unroll
    for (int i = 0; i < NS; i++) finite = finite && isfinite(e[i]);
    if (out_pf) {
#pragma unroll
      for (int i = 0; i < NS; i++) out_pf[(long long)i * N + n] = e[i];
      out_pf[21LL * N + n] = nees;
      out_pf[22LL * N + n] = ll;
    }
    if (finite) {
#pragma unroll
      for (int i = 0; i < NS; i++) {
        val[i] = e[i];
        val[21 + i] = __dmul_rn(e[i], e[i]);
      }
      val[42] = nees;
      val[43] = __dmul_rn(nees, nees);
      val[44] = ll;
      val[47] = (nees >= 2.7003895 && nees <= 19.0227678) ? 1.0 : 0.0;  // chi2(9) 2.5% / 97.5% quantiles
    } else {
      val[45] = 1.0;
    }
    val[46] = 1.0;
  }
  static_for<48>([&](auto k) {
    red[t] = val[k];
    __syncthreads();
    for (int s = blockDim.x >> 1; s > 0; s >>= 1) {
      if (t < s) red[t] = __dadd_rn(red[t], red[t + s]);
      __syncthreads();
    }
    if (t == 0) out_chunks[(long long)blockIdx.x * NSTAT + k] = red[0];
    __syncthreads();
  });
  // the reserved statistics 48..95 are zero, also for chunks of fewer than 96 filters
  for (int k = 48 + t; k < NSTAT; k += blockDim.x) out_chunks[(long long)blockIdx.x * NSTAT + k] = 0.0;
}

// chi2(m) 2.5 % / 97.5 % quantiles for m = 1..9 (scipy.stats.chi2.ppf; m = 9 is the pair of stats_kernel)
__constant__ double c_chi2_lo[9] = {0.000982069117, 0.050635616, 0.215795283, 0.484418557, 0.831211613,
                                    1.23734425,     1.68986918,  2.17973075,  2.7003895};
__constant__ double c_chi2_hi[9] = {5.02388619, 7.37775891, 9.3484036, 11.1432868, 12.832502,
                                    14.4493753, 16.0127643, 17.5345461, 19.0227678};
constexpr int NINNOV = 33;  // statistics of an innovation table; the rest of the 96 are zero
// Ensemble statistics of innovation rows ([rows][k][N], the layout of InnovK with INNOV_NIS at position 0): row blockIdx.y of
// `rows`, one CTA per chunk of blockDim.x filters, one table [gridDim.x][96] per row.  [0] sum NIS, [1] sum NIS^2, [2] finite
// NIS, [3] NIS inside the central 95 % of chi2(m), [4] non-finite NIS, [5] filters, [6 + a] sum y_a, [15 + a] sum y_a^2,
// [24 + a] sum y_a^2 / S(a,a); only filters with a finite NIS enter [0], [1], [3] and [6..32].  The fixed binary tree of
// stats_kernel, so a numpy restatement reproduces every table bit for bit.
__global__ void __launch_bounds__(1024) innov_stats_kernel(const double* __restrict__ rows, long long k, int m, int fields, long long N,
                                                           double* __restrict__ out_chunks) {
  extern __shared__ double red[];
  const int t = threadIdx.x;
  const long long n = (long long)blockIdx.x * blockDim.x + t;
  rows += (long long)blockIdx.y * k * N;
  out_chunks += (long long)blockIdx.y * gridDim.x * NSTAT;
  double val[NINNOV];
#pragma unroll
  for (int i = 0; i < NINNOV; i++) val[i] = 0.0;
  if (n < N) {
    const double nis = rows[n];
    if (isfinite(nis)) {
      val[0] = nis;
      val[1] = __dmul_rn(nis, nis);
      val[2] = 1.0;
      val[3] = (nis >= c_chi2_lo[m - 1] && nis <= c_chi2_hi[m - 1]) ? 1.0 : 0.0;
      if (fields & INNOV_Y) {
        const int os = 1 + m;  // S(a,a) follows y
#pragma unroll
        for (int a = 0; a < MAX_MEAS; a++) {
          if (a < m) {
            const double y = rows[(long long)(1 + a) * N + n];
            const double y2 = __dmul_rn(y, y);
            val[6 + a] = y;
            val[15 + a] = y2;
            if (fields & INNOV_S_DIAG) val[24 + a] = __ddiv_rn(y2, rows[(long long)(os + a) * N + n]);
          }
        }
      }
    } else {
      val[4] = 1.0;
    }
    val[5] = 1.0;
  }
  static_for<NINNOV>([&](auto i) {
    red[t] = val[i];
    __syncthreads();
    for (int s = blockDim.x >> 1; s > 0; s >>= 1) {
      if (t < s) red[t] = __dadd_rn(red[t], red[t + s]);
      __syncthreads();
    }
    if (t == 0) out_chunks[(long long)blockIdx.x * NSTAT + i] = red[0];
    __syncthreads();
  });
  for (int i = NINNOV + t; i < NSTAT; i += blockDim.x) out_chunks[(long long)blockIdx.x * NSTAT + i] = 0.0;
}

// Final reduction of a chunk table on the device: totals[k] = sum over chunks in ASCENDING chunk order (one thread per
// statistic, a plain sequential sum: the same order as rbis_stats_reduce_chunks on the host).  One CTA per table:
// table blockIdx.x is [n_chunks][96] at table + blockIdx.x * n_chunks * 96, its totals at totals + blockIdx.x * 96.
__global__ void reduce_chunk_table_kernel(const double* __restrict__ table, long long n_chunks, double* __restrict__ totals) {
  const int k = threadIdx.x;
  if (k >= NSTAT) return;
  table += (long long)blockIdx.x * n_chunks * NSTAT;
  totals += (long long)blockIdx.x * NSTAT;
  double s = 0.0;
  for (long long c = 0; c < n_chunks; c++) s = __dadd_rn(s, table[c * NSTAT + k]);
  totals[k] = s;
}

// ---- windowed noise-identification likelihood (SE/noise_id/noise_id.cpp:36-40,44-65) ----
// One lane per filter: e = head (-) truth (subtractState + quatToChi), C = cov - base_cov[:, map[n]] (the covariance the
// same window accumulates under zero process noise), out = log det C_AA + e_A^T C_AA^-1 e_A = -loglike_normalized(e_A, 0, C_AA).
__global__ void window_nll_kernel(const double* __restrict__ vec, const double* __restrict__ quat, const double* __restrict__ P,
                                  const double* __restrict__ tvec, const double* __restrict__ tquat,
                                  const double* __restrict__ base_cov, const int* __restrict__ base_map, long long base_cols,
                                  int n_active, const int* __restrict__ active, long long N, double* __restrict__ out) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  double e[NS];
  for (int i = 0; i < NS; i++) e[i] = vec[(long long)i * N + n] - tvec[(long long)i * N + n];
  const Q4 q{quat[n], quat[N + n], quat[2 * N + n], quat[3 * N + n]};
  const Q4 tq{tquat[n], tquat[N + n], tquat[2 * N + n], tquat[3 * N + n]};
  const V3 dchi = subtract_quats(q, tq);
  // quatToChi after subtractState: chi = Log(truth^-1 * est); the vec chi difference is dropped by the reference only
  // if the fold happened -- subtractState subtracts vec (chi included) and quatToChi OVERWRITES chi (eigen_utils)
  e[6] = dchi.x; e[7] = dchi.y; e[8] = dchi.z;
  const long long bc = base_map ? (long long)base_map[n] : n;
  double L[NS][NS], D[NS], y[NS];
  double logdet = 0, quad = 0;
  for (int k = 0; k < n_active; k++) {
    const int ik = active[k];
    double d = P[(long long)slot(ik, ik) * N + n] - base_cov[(long long)(ik + NS * ik) * base_cols + bc];
    for (int p = 0; p < k; p++) d -= L[k][p] * L[k][p] * D[p];
    D[k] = d;
    logdet += log(d);
    for (int i = k + 1; i < n_active; i++) {
      const int ii = active[i];
      double v = P[(long long)slot(ii, ik) * N + n] - base_cov[(long long)(ii + NS * ik) * base_cols + bc];
      for (int p = 0; p < k; p++) v -= L[i][p] * L[k][p] * D[p];
      L[i][k] = v / d;
    }
  }
  for (int i = 0; i < n_active; i++) {
    double v = -e[active[i]];  // diff = mu - x with mu = 0
    for (int k = 0; k < i; k++) v -= L[i][k] * y[k];
    y[i] = v;
    quad += v * v / D[i];
  }
  out[n] = logdet + quad;
}

// ---- FP64 roofline denominators ----
constexpr int DFMA_CHAINS = 8;
constexpr int DFMA_UNROLL = 32;
__global__ void __launch_bounds__(256) dfma_peak_kernel(double* out, int iters, double a) {
  double x[DFMA_CHAINS];
#pragma unroll
  for (int c = 0; c < DFMA_CHAINS; c++) x[c] = 1e-3 * threadIdx.x + c;
  const double b = a * 0.5 - 0.5;
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int u = 0; u < DFMA_UNROLL; u++)
#pragma unroll
      for (int c = 0; c < DFMA_CHAINS; c++) x[c] = fma(x[c], a, b);
  }
  double s = 0;
#pragma unroll
  for (int c = 0; c < DFMA_CHAINS; c++) s += x[c];
  out[(long long)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

constexpr int DMMA_CHAINS = 8;
constexpr int DMMA_UNROLL = 8;
__global__ void __launch_bounds__(256) dmma_peak_kernel(double* out, int iters, double a) {
  double c0[DMMA_CHAINS], c1[DMMA_CHAINS];
#pragma unroll
  for (int c = 0; c < DMMA_CHAINS; c++) { c0[c] = 1e-3 * threadIdx.x + c; c1[c] = c0[c] + 0.5; }
  const double av = a * 1e-3, bv = a * 2e-3;
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int u = 0; u < DMMA_UNROLL; u++)
#pragma unroll
      for (int c = 0; c < DMMA_CHAINS; c++)
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                     : "+d"(c0[c]), "+d"(c1[c])
                     : "d"(av), "d"(bv));
  }
  double s = 0;
#pragma unroll
  for (int c = 0; c < DMMA_CHAINS; c++) s += c0[c] + c1[c];
  out[(long long)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// ------------------------------------------------------------------------------------------------
// IMU conditioning ("next" row 4 of SURVEY.md 8f): InsHandler::doFilter (MSE/sensor_handlers.cpp:155-162) = a cascade of
// IIRNotch::processSample (estimate_tools/src/estimate_tools/iir_notch.cpp:35-60) on the three accelerometer channels,
// for every column of an IMU chunk [rows][6][cols], in place.  One thread per column and channel; its n_stages x
// (x0,x1,y0,y1) of filter state stay in registers over the rows of the chunk and persist in `state`
// ([3][MAX_NOTCH][4][cols]) between calls.  HBM-bound: 24 B read + 24 B written per row and column.
// ------------------------------------------------------------------------------------------------
constexpr int MAX_NOTCH = 4;
struct NotchCoeffs {
  double b[MAX_NOTCH][3], a[MAX_NOTCH][3];
  int n_stages;
};
__global__ void __launch_bounds__(128) notch_kernel(double* __restrict__ imu, long long rows, long long cols, double* __restrict__ state,
                                                    const __grid_constant__ NotchCoeffs co) {
  // one thread per (column, accelerometer channel): blockIdx.y is the channel
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int ch = blockIdx.y;
  if (c >= cols) return;
  double st[MAX_NOTCH][4];
#pragma unroll
  for (int i = 0; i < MAX_NOTCH; i++)
#pragma unroll
    for (int k = 0; k < 4; k++) st[i][k] = (i < co.n_stages) ? state[((long long)(ch * MAX_NOTCH + i) * 4 + k) * cols + c] : 0.0;
  auto sample = [&](double v) {
#pragma unroll
    for (int i = 0; i < MAX_NOTCH; i++) {
      if (i < co.n_stages) {
        // output = (input, x0, x1) . b - (0, y0, y1) . a, summed left to right as Eigen's 3-vector dot does
        const double xb = v * co.b[i][0] + st[i][0] * co.b[i][1] + st[i][1] * co.b[i][2];
        const double ya = 0 * co.a[i][0] + st[i][2] * co.a[i][1] + st[i][3] * co.a[i][2];
        const double out = xb - ya;
        st[i][1] = st[i][0]; st[i][0] = v;
        st[i][3] = st[i][2]; st[i][2] = out;
        v = out;
      }
    }
    return v;
  };
  // the recursion is serial in time, the loads are not: NOTCH_ROWS rows are fetched ahead of the arithmetic
  constexpr int NOTCH_ROWS = 8;
  double* base = imu + (long long)(3 + ch) * cols + c;
  const long long stride = 6 * cols;
  long long r = 0;
  for (; r + NOTCH_ROWS <= rows; r += NOTCH_ROWS) {
    double v[NOTCH_ROWS];
#pragma unroll
    for (int k = 0; k < NOTCH_ROWS; k++) v[k] = base[(r + k) * stride];
#pragma unroll
    for (int k = 0; k < NOTCH_ROWS; k++) base[(r + k) * stride] = sample(v[k]);
  }
  for (; r < rows; r++) base[r * stride] = sample(base[r * stride]);
#pragma unroll
  for (int i = 0; i < MAX_NOTCH; i++)
#pragma unroll
    for (int k = 0; k < 4; k++)
      if (i < co.n_stages) state[((long long)(ch * MAX_NOTCH + i) * 4 + k) * cols + c] = st[i][k];
}

}  // namespace rbisk
