// rbis_group.cuh -- the WARP-GROUP mapping of the fused RBIS kernel: G lanes (2, 4, 8 or 16) cooperate on one filter.
//
// Why it exists (DESIGN.md 4.7).  The lane-per-filter kernels of rbis_kernels.cuh need >= 148 x 384 filters to fill a
// B200; a 4,096-filter ensemble (BASELINE configs[1]) or a 65,536-filter ensemble split over 8 GPUs (8,192 each) leaves
// 11-22 of 148 SMs busy and every busy scheduler latency bound.  Here a filter's work is spread over G lanes, so the same
// ensemble brings G times as many warps and each warp's dependent chain per step is ~G times shorter.
//
// Layout.  A filter's covariance lives in shared memory as a FULL NA x NA matrix, row-major, NA = 15 (DC: the active
// block v, chi, p, b_g, b_a; see "decoupled filters" in rbis_kernels.cuh) or 21 (dense), with BOTH triangles kept equal
// bit for bit: every element (i, j) is computed once, by the lane that owns column max(i, j), and stored to (i, j) and
// (j, i).  The packed upper triangle is read at the start of a launch / RESTORE and written at its end / SNAPSHOT.  The
// leading dimension NA is odd and the per-filter stride is = G (mod 16) doubles, which makes the column accesses (lane l ->
// column l + G j), their mirrored row accesses and the broadcast reads of whole rows conflict free for 8-byte accesses.
// The filter state (21 + 4 + log-likelihood) is REPLICATED in the G lanes of the group: every lane runs the serial state
// arithmetic (insUpdateState, the 3x3 LDL^T, addState) redundantly, with the device functions of the lane-per-filter
// kernel, and the lanes split the covariance work by columns:
//   IMU step  cov = Ad cov Ad^T + Qd (MSE/rbis.cpp:113-118) as the three congruences Ad = E_chi E_v E_p of
//             rbisk::cov_propagate, each a column pass (lane owns columns) and a 3-row pass, see g_cov_propagate;
//   update    S = R + P[idx,idx], LDL^T and Y = L^-1 P[idx,:] in every lane (broadcast reads of the three rows), then
//             P[i,j] -= sum_a Y[a][i] Y[a][j] / d_a for i <= j in the lane's own columns j (rbis.cpp:134-140).
// EVERY ELEMENT IS COMPUTED BY THE SAME EXPRESSION AS IN THE LANE-PER-FILTER KERNELS (the library is compiled with
// -fmad=false and every fused multiply-add is explicit), so the two mappings give bit-identical results: the mapping is
// a scheduling decision the caller cannot observe (tests/test_gpu_group.py), and statistics of a sharded ensemble do
// not depend on how many GPUs -- hence which mapping per shard -- it runs on.
// Lanes synchronise with __syncwarp() only; a CTA is any number of warps (chosen by the host so that the ensemble
// spreads over all SMs), there is no CTA-wide barrier and no tensor memory.
//
// Included after rbis_kernels.cuh, into the same namespace, by the warp-group translation units (rbis_fused_g*.cu).
#ifndef RBIS_GROUP_CUH_
#define RBIS_GROUP_CUH_

namespace rbisk {
namespace grp {

template <int G, bool DC>
struct Geo {
  static_assert(G == 2 || G == 4 || G == 8 || G == 16, "lanes per filter");
  static constexpr int NA = DC ? N_ACT : NS;   // matrix dimension
  static constexpr int LD = NA;                // leading dimension (odd: 15 or 21)
  static constexpr int FPW = 32 / G;           // filters per warp
  static constexpr int NJ = (NA + G - 1) / G;  // columns (rows) a lane owns at most
  static constexpr int stride_() {
    int s = NA * LD;
    while (s % 16 != G % 16) s++;
    return s;
  }
  static constexpr int S = stride_();          // doubles per filter in shared memory
  // matrix positions of the block rows Ad touches / reads
  static constexpr int PV = DC ? 0 : 3, PC = DC ? 3 : 6, PP = DC ? 6 : 9, PG = DC ? 9 : 15, PA = DC ? 12 : 18;
};
template <bool DC>
__device__ __forceinline__ int pos_of(int idx) { return DC ? (idx < 12 ? idx - 3 : idx - 6) : idx; }
template <bool DC>
__host__ __device__ constexpr int idx_of(int pos) { return DC ? act_col(pos) : pos; }

// x[I0 + A] for an aligned triple base I0 in {0, 3, .., 18} (run time, warp uniform)
template <int A>
__device__ __forceinline__ double pick_triple(const double (&x)[NS], int I0) {
  double v = x[A];
#pragma unroll
  for (int t = 1; t < NS / 3; t++) v = (I0 == 3 * t) ? x[3 * t + A] : v;
  return v;
}
__device__ __forceinline__ double sel3(const V3& v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : v.z); }
// The lane's j-th column: index, and whether it exists (lanes beyond the matrix edge work on a copy of the last column
// and do not store, which keeps the code free of branches).
template <int G, int NA>
struct Own {
  static constexpr int NJ = (NA + G - 1) / G;
  int c[NJ];
  bool own[NJ];
  __device__ __forceinline__ explicit Own(int l) {
#pragma unroll
    for (int j = 0; j < NJ; j++) {
      const int cj = l + G * j;
      own[j] = ((j + 1) * G <= NA) || cj < NA;
      c[j] = own[j] ? cj : NA - 1;
    }
  }
};
// One row of acc_mul_skew<SIGN>(acc, Z, u) (rbis_kernels.cuh): acc[k], Z[k] are component i of the k-th column vector.
template <int SIGN>
__device__ __forceinline__ void row_mul_skew(double (&acc)[3], const double (&Z)[3], const V3& u) {
  const double ux = SIGN * u.x, uy = SIGN * u.y, uz = SIGN * u.z;
  acc[0] = fma(uz, Z[1], fma(-uy, Z[2], acc[0]));
  acc[1] = fma(ux, Z[2], fma(-uz, Z[0], acc[1]));
  acc[2] = fma(uy, Z[0], fma(-ux, Z[1], acc[2]));
}
__device__ __forceinline__ V3 ld3(const double* b, int stride) { return {b[0], b[stride], b[2 * stride]}; }

// ------------------------------------------------------------------------------------------------
// insUpdateCovariance (rbis.cpp:77-122) for one filter; l = lane within the group.  The same three in-place symmetric
// congruences Ad = E_chi E_v E_p as rbisk::cov_propagate, element for element the same expressions:
//   column pass of E_X   z_c = (E_X P)[X, c] for every column c -- the lane's own columns, zp / zv / zc of rbis_kernels.cuh;
//                        stored as P[X, c] and mirrored to P[c, X]; for c inside X the 3x3 block is left unsymmetric
//                        (element (X_i, X_k) = z of column X_k) until
//   row pass of E_X      P'[X_i, X_j] = Z_X + sum_K Z_K N[X,K]^T from ROW X_i of what the column pass left, for j >= i,
//                        written to both triangles (three lanes, one row each).
// The row pass of one congruence and the column pass of the next touch disjoint data and run in the same phase:
//   A  E_p columns | B  E_p rows + E_v columns | C  E_v rows + E_chi columns | D  E_chi rows,
// each phase = loads, __syncwarp, arithmetic + stores, __syncwarp (a store of one lane never overtakes another lane's load).
// ------------------------------------------------------------------------------------------------
template <int G, bool DC>
__device__ __forceinline__ void g_cov_propagate(double* Pf, const int l, const Lin& L, const QNoise& qn) {
  using GE = Geo<G, DC>;
  constexpr int NA = GE::NA, LD = GE::LD, NJ = GE::NJ;
  constexpr int PV = GE::PV, PC = GE::PC, PP = GE::PP, PG = GE::PG, PA = GE::PA;
  constexpr int NR = (3 + G - 1) / G;  // rows of a 3-row pass per lane (1 for G >= 4)
  const Own<G, NA> w(l);
  const double dt = L.dt;
  const double qg = qn.q_gyro * dt, qa = qn.q_accel * dt;
  // the lane's rows of a row pass: component i = l + G jr (< 3)
  int ri[NR];
  bool rown[NR];
#pragma unroll
  for (int jr = 0; jr < NR; jr++) { const int i = l + G * jr; rown[jr] = i < 3; ri[jr] = rown[jr] ? i : 2; }

  // ---------------- phase A: E_p columns.  z = zp(P[v,c], P[chi,c], P[p,c]) -> P[p,c] ----------------
  {
    V3 z[NJ];
    static_for<NJ>([&](auto jc) {
      constexpr int j = jc;
      const double* b = Pf + w.c[j];
      z[j] = zp(L, ld3(b + PV * LD, LD), ld3(b + PC * LD, LD), ld3(b + PP * LD, LD));
    });
    __syncwarp();
    static_for<NJ>([&](auto jc) {
      constexpr int j = jc;
      const int c = w.c[j];
      if (w.own[j]) {
        double* b = Pf + c;
        b[PP * LD] = z[j].x; b[(PP + 1) * LD] = z[j].y; b[(PP + 2) * LD] = z[j].z;
        if (c < PP || c >= PP + 3) {  // mirror, except inside the (p,p) block (completed by the row pass)
          double* m = Pf + c * LD + PP;
          m[0] = z[j].x; m[1] = z[j].y; m[2] = z[j].z;
        }
      }
    });
    __syncwarp();
  }
  // ---------------- phase B: E_p rows (P'[p,p] = Zp + (Zv + Zc skew(v)) (R dt)^T)  +  E_v columns ----------------
  {
    double outp[NR][3];
#pragma unroll
    for (int jr = 0; jr < NR; jr++) {
      const double* r = Pf + (PP + ri[jr]) * LD;
      double T[3] = {r[PV], r[PV + 1], r[PV + 2]};
      const double Zb[3] = {r[PC], r[PC + 1], r[PC + 2]};
      const double Zp[3] = {r[PP], r[PP + 1], r[PP + 2]};
      row_mul_skew<1>(T, Zb, L.v);
#pragma unroll
      for (int j = 0; j < 3; j++) outp[jr][j] = fma(T[0], L.Rd[3 * j], fma(T[1], L.Rd[3 * j + 1], fma(T[2], L.Rd[3 * j + 2], Zp[j])));
    }
    V3 z[NJ];
    double pad[NJ];  // the column's own diagonal element when it is a b_a column
    static_for<NJ>([&](auto jc) {
      constexpr int j = jc;
      const double* b = Pf + w.c[j];
      const V3 pa = ld3(b + PA * LD, LD);
      z[j] = zv(L, ld3(b + PV * LD, LD), ld3(b + PC * LD, LD), ld3(b + PG * LD, LD), pa);
      pad[j] = sel3(pa, w.c[j] - PA);
    });
    __syncwarp();
#pragma unroll
    for (int jr = 0; jr < NR; jr++) {
      if (rown[jr]) {
        const int i = ri[jr];
#pragma unroll
        for (int j = 0; j < 3; j++)
          if (j >= i) { Pf[(PP + i) * LD + PP + j] = outp[jr][j]; Pf[(PP + j) * LD + PP + i] = outp[jr][j]; }
      }
    }
    static_for<NJ>([&](auto jc) {
      constexpr int j = jc;
      const int c = w.c[j];
      if (w.own[j]) {
        double* b = Pf + c;
        b[PV * LD] = z[j].x; b[(PV + 1) * LD] = z[j].y; b[(PV + 2) * LD] = z[j].z;
        if (c < PV || c >= PV + 3) {
          double* m = Pf + c * LD + PV;
          m[0] = z[j].x; m[1] = z[j].y; m[2] = z[j].z;
        }
        if (c >= PA && c < PA + 3) b[c * LD] = fma(qn.q_accel_bias, dt, pad[j]);  // Qd[ba,ba]
      }
    });
    __syncwarp();
  }
  // ---------------- phase C: E_v rows (P'[v,v])  +  E_chi columns ----------------
  {
    const double vv = sumsq3(L.v.x, L.v.y, L.v.z);
    double outv[NR][3];
#pragma unroll
    for (int jr = 0; jr < NR; jr++) {
      const int i = ri[jr];
      const double* r = Pf + (PV + i) * LD;
      const double Zv[3] = {r[PV], r[PV + 1], r[PV + 2]};
      const double Zc[3] = {r[PC], r[PC + 1], r[PC + 2]};
      const double Zg[3] = {r[PG], r[PG + 1], r[PG + 2]};
      const double Za[3] = {r[PA], r[PA + 1], r[PA + 2]};
      double Nv[3] = {Zv[0], Zv[1], Zv[2]};
      row_mul_skew<1>(Nv, Zv, L.wd);
      row_mul_skew<-1>(Nv, Zc, L.gd);
      row_mul_skew<1>(Nv, Zg, L.vd);
#pragma unroll
      for (int k = 0; k < 3; k++) Nv[k] = fma(-dt, Za[k], Nv[k]);
      // + Qd[v,v] = dt (q_gyro (|v|^2 I - v v^T) + q_accel I)      (rbis.cpp:91-116)
      const double vi = sel3(L.v, i);
      const double vj[3] = {L.v.x, L.v.y, L.v.z};
#pragma unroll
      for (int j = 0; j < 3; j++) outv[jr][j] = (j == i) ? Nv[j] + fma(qg, fma(-vi, vi, vv), qa) : fma(qg, -vi * vj[j], Nv[j]);
    }
    V3 z[NJ];
    double pgd[NJ];
    static_for<NJ>([&](auto jc) {
      constexpr int j = jc;
      const int c = w.c[j];
      const double* b = Pf + c;
      const V3 pg = ld3(b + PG * LD, LD);
      V3 zz = zc(L, ld3(b + PC * LD, LD), pg);
      pgd[j] = sel3(pg, c - PG);
      // P'[chi, v_k] = z + Qd[chi, v_k],  Qd[chi_i, v_k] = dt q_gyro skew(v)[k][i]
      const int k = c - PV;
      if (k >= 0 && k < 3) {
        const V3 sk = k == 0 ? V3{0.0, -L.v.z, L.v.y} : (k == 1 ? V3{L.v.z, 0.0, -L.v.x} : V3{-L.v.y, L.v.x, 0.0});
        if (k != 0) zz.x = fma(qg, sk.x, zz.x);
        if (k != 1) zz.y = fma(qg, sk.y, zz.y);
        if (k != 2) zz.z = fma(qg, sk.z, zz.z);
      }
      z[j] = zz;
    });
    __syncwarp();
#pragma unroll
    for (int jr = 0; jr < NR; jr++) {
      if (rown[jr]) {
        const int i = ri[jr];
#pragma unroll
        for (int j = 0; j < 3; j++)
          if (j >= i) { Pf[(PV + i) * LD + PV + j] = outv[jr][j]; Pf[(PV + j) * LD + PV + i] = outv[jr][j]; }
      }
    }
    static_for<NJ>([&](auto jc) {
      constexpr int j = jc;
      const int c = w.c[j];
      if (w.own[j]) {
        double* b = Pf + c;
        b[PC * LD] = z[j].x; b[(PC + 1) * LD] = z[j].y; b[(PC + 2) * LD] = z[j].z;
        if (c < PC || c >= PC + 3) {
          double* m = Pf + c * LD + PC;
          m[0] = z[j].x; m[1] = z[j].y; m[2] = z[j].z;
        }
        if (c >= PG && c < PG + 3) b[c * LD] = fma(qn.q_gyro_bias, dt, pgd[j]);  // Qd[bg,bg]
      }
    });
    __syncwarp();
  }
  // ---------------- phase D: E_chi rows.  P'[chi,chi] = Zc + Zc skew(wd) - dt Zg + Qd[chi,chi] ----------------
  {
    double outc[NR][3];
#pragma unroll
    for (int jr = 0; jr < NR; jr++) {
      const int i = ri[jr];
      const double* r = Pf + (PC + i) * LD;
      const double Zc[3] = {r[PC], r[PC + 1], r[PC + 2]};
      const double Zg[3] = {r[PG], r[PG + 1], r[PG + 2]};
      double Mc[3] = {Zc[0], Zc[1], Zc[2]};
      row_mul_skew<1>(Mc, Zc, L.wd);
#pragma unroll
      for (int k = 0; k < 3; k++) Mc[k] = fma(-dt, Zg[k], Mc[k]);
#pragma unroll
      for (int j = 0; j < 3; j++) outc[jr][j] = (j == i) ? Mc[j] + qg : Mc[j];
    }
    __syncwarp();
#pragma unroll
    for (int jr = 0; jr < NR; jr++) {
      if (rown[jr]) {
        const int i = ri[jr];
#pragma unroll
        for (int j = 0; j < 3; j++)
          if (j >= i) { Pf[(PC + i) * LD + PC + j] = outc[jr][j]; Pf[(PC + j) * LD + PC + i] = outc[jr][j]; }
      }
    }
    if constexpr (!DC) {
      // overwrites of rbis.cpp:120-121: the owner of a column omega_k / a_k rewrites its three block elements
      static_for<NJ>([&](auto jc) {
        constexpr int j = jc;
        const int c = w.c[j];
        if (w.own[j]) {
          if (c < 3) { Pf[c] = c == 0 ? qn.q_gyro : 0.0; Pf[LD + c] = c == 1 ? qn.q_gyro : 0.0; Pf[2 * LD + c] = c == 2 ? qn.q_gyro : 0.0; }
          if (c >= 12 && c < 15) {
            Pf[12 * LD + c] = c == 12 ? qn.q_accel : 0.0; Pf[13 * LD + c] = c == 13 ? qn.q_accel : 0.0; Pf[14 * LD + c] = c == 14 ? qn.q_accel : 0.0;
          }
        }
      });
    }
    __syncwarp();
  }
}

// P[i,j] -= sum_a Y[a][i] (Y[a][j] r_a) over the upper triangle i <= j of the lane's own columns j, mirrored into the lower
// triangle: the expression of rbisk::meas3 / rank1_sweep element for element.  NY = rows of Y (3 or 1).  wj[j][a] = the
// lane's own Y[a][c_j] * r_a, formed BEFORE the barrier that precedes the sweep (a mirrored store of another lane may
// overwrite the lower-triangle element it was read from).  Column slot j only visits rows k < G (j + 1): the rest lie
// below the diagonal for every lane.  MASK, skip: the filter's row is missing, its lanes store back the values they loaded
// (the matrix keeps its bits); the G lanes of a group read the same z, so they agree on skip.
template <int G, bool DC, int NY, bool MASK = false>
__device__ __forceinline__ void g_sweep(double* Pf, const Own<G, Geo<G, DC>::NA>& w, const double (&Y)[NY][Geo<G, DC>::NA],
                                        const double (&wj)[Geo<G, DC>::NJ][NY], bool skip = false) {
  using GE = Geo<G, DC>;
  constexpr int NA = GE::NA, LD = GE::LD, NJ = GE::NJ;
  static_for<NJ>([&](auto jc) {
    constexpr int j = jc;
    constexpr int KMAX = (G * (j + 1) < NA) ? G * (j + 1) : NA;
    const int c = w.c[j];
    double* b = Pf + c;
    double* m = Pf + c * LD;
    double v[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; k++) v[k] = b[k * LD];
#pragma unroll
    for (int k = 0; k < KMAX; k++) {
      double acc = v[k];
#pragma unroll
      for (int a = NY - 1; a >= 0; a--) acc = fma(-Y[a][k], wj[j][a], acc);
      if constexpr (MASK) acc = skip ? v[k] : acc;
      if (w.own[j] && (k < G * j || k <= c)) { b[k * LD] = acc; m[k] = acc; }
    }
  });
}

// Aligned index triple I0..I0+2 (leg-odometry velocity, pose position / orientation, ...): rbis.cpp:124-143 with
// S = L D L^T, Y = L^-1 P[idx,:], P -= Y^T D^-1 Y, x += Y^T D^-1 L^-1 r.  Same arithmetic as rbisk::meas3.
// NISQ: *nisq += the chunk's quadratic form, as in rbisk::meas3 (the same for g_meas1 / g_meas_block).
template <int G, bool DC, bool SYN, bool MASK = false, bool NISQ = false>
__device__ __forceinline__ void g_meas3(double* Pf, const int l, FilterState& s, const StreamDesc& st, const MeasSrc<SYN>& src, int a0, int I0,
                                        long long row, long long N, long long n, long long sn, const V3& dquat, const V3& chi0,
                                        bool skip = false, double* nisq = nullptr) {
  using GE = Geo<G, DC>;
  constexpr int NA = GE::NA, LD = GE::LD, NJ = GE::NJ;
  double z[3], Rdg[3];
  src.z3(st, row, a0, sn, z);
  if (st.r_mode == 1) {
#pragma unroll
    for (int a = 0; a < 3; a++) Rdg[a] = ldg_early(st.R + (long long)(a0 + a) * N + n);
  }
  const Own<G, NA> w(l);
  const int p0 = pos_of<DC>(I0);
  const double* r0p = Pf + p0 * LD;  // rows p0, p0+1, p0+2 of P: HP = C cov (rbis.cpp:134)
  double Y[3][NA];
#pragma unroll
  for (int k = 0; k < NA; k++) { Y[0][k] = r0p[k]; Y[1][k] = r0p[LD + k]; Y[2][k] = r0p[2 * LD + k]; }
  double yo[NJ][3];  // the lane's own columns of HP
#pragma unroll
  for (int j = 0; j < NJ; j++) { yo[j][0] = r0p[w.c[j]]; yo[j][1] = r0p[LD + w.c[j]]; yo[j][2] = r0p[2 * LD + w.c[j]]; }
  // S = R + P[idx,idx]
  double S00 = r0p[p0], S10 = r0p[LD + p0], S20 = r0p[2 * LD + p0], S11 = r0p[LD + p0 + 1], S21 = r0p[2 * LD + p0 + 1],
         S22 = r0p[2 * LD + p0 + 2];
  if (st.r_mode == 1) {
    S00 += Rdg[0]; S11 += Rdg[1]; S22 += Rdg[2];
  } else {
    const double* Rm = st.R + row * st.r_stride + a0 + (long long)st.m * a0;
    S00 += __ldg(Rm); S11 += __ldg(Rm + st.m + 1); S22 += __ldg(Rm + 2 * st.m + 2);
    S10 += __ldg(Rm + 1); S20 += __ldg(Rm + 2); S21 += __ldg(Rm + st.m + 2);
  }
  __syncwarp();  // every lane has read the three rows before any lane overwrites its part of them
  const double d0 = S00, r0 = 1.0 / d0;
  const double l10 = S10 * r0, l20 = S20 * r0;
  const double d1 = fma(-l10 * l10, d0, S11), r1 = 1.0 / d1;
  const double l21 = fma(-l20 * l10, d0, S21) * r1;
  const double d2 = fma(-l21 * l21, d1, fma(-l20 * l20, d0, S22)), r2 = 1.0 / d2;
  const double pd = d0 * d1 * d2;
  const double logdet = (pd > 1e-290 && pd < 1e290) ? log(pd) : log(d0) + log(d1) + log(d2);
#pragma unroll
  for (int c = 0; c < NA; c++) {
    Y[1][c] = fma(-l10, Y[0][c], Y[1][c]);
    Y[2][c] = fma(-l21, Y[1][c], fma(-l20, Y[0][c], Y[2][c]));
  }
  double wj[NJ][3];
#pragma unroll
  for (int j = 0; j < NJ; j++) {
    const double y1 = fma(-l10, yo[j][0], yo[j][1]);
    const double y2 = fma(-l21, y1, fma(-l20, yo[j][0], yo[j][2]));
    wj[j][0] = yo[j][0] * r0; wj[j][1] = y1 * r1; wj[j][2] = y2 * r2;
  }
  g_sweep<G, DC, 3, MASK>(Pf, w, Y, wj, skip);
  __syncwarp();
  double r[3];
  if (I0 == 6 && st.has_orient) {
    r[0] = dquat.x - (s.x[6] - chi0.x); r[1] = dquat.y - (s.x[7] - chi0.y); r[2] = dquat.z - (s.x[8] - chi0.z);
  } else {
    r[0] = z[0] - pick_triple<0>(s.x, I0); r[1] = z[1] - pick_triple<1>(s.x, I0); r[2] = z[2] - pick_triple<2>(s.x, I0);
  }
  const double e0 = r[0], e1 = fma(-l10, e0, r[1]), e2 = fma(-l21, e1, fma(-l20, e0, r[2]));
  const double u0 = e0 * r0, u1 = e1 * r1, u2 = e2 * r2;
  static_for<NA>([&](auto cc) {
    constexpr int c = cc;
    constexpr int xc = idx_of<DC>(c);
    if constexpr (MASK) s.x[xc] = skip ? s.x[xc] : fma(Y[0][c], u0, fma(Y[1][c], u1, fma(Y[2][c], u2, s.x[xc])));
    else s.x[xc] = fma(Y[0][c], u0, fma(Y[1][c], u1, fma(Y[2][c], u2, s.x[xc])));
  });
  if constexpr (MASK) s.ll = skip ? s.ll : s.ll + (-logdet - fma(e2, u2, fma(e1, u1, e0 * u0)));
  else s.ll += -logdet - fma(e2, u2, fma(e1, u1, e0 * u0));
  if constexpr (NISQ) *nisq += fma(e2, u2, fma(e1, u1, e0 * u0));
}

// One-row chunk on state index idx (rbisk::meas1).
template <int G, bool DC, bool SYN, bool MASK = false, bool NISQ = false>
__device__ __forceinline__ void g_meas1(double* Pf, const int l, FilterState& s, const StreamDesc& st, const MeasSrc<SYN>& src, int a0, int idx,
                                        long long row, long long N, long long n, long long sn, const V3& dquat, const V3& chi0,
                                        bool skip = false, double* nisq = nullptr) {
  using GE = Geo<G, DC>;
  constexpr int NA = GE::NA, LD = GE::LD, NJ = GE::NJ;
  const double z = src.z(st, row, a0, sn);
  const double Rv = (st.r_mode == 1) ? ldg_early(st.R + (long long)a0 * N + n) : __ldg(st.R + row * st.r_stride + a0 + (long long)st.m * a0);
  const Own<G, NA> w(l);
  const int pi = pos_of<DC>(idx);
  const double* rp = Pf + pi * LD;
  double h[1][NA];
#pragma unroll
  for (int k = 0; k < NA; k++) h[0][k] = rp[k];
  double wj[NJ][1];
#pragma unroll
  for (int j = 0; j < NJ; j++) wj[j][0] = rp[w.c[j]];
  const double sv = Rv + rp[pi];
  __syncwarp();
  const double r = 1.0 / sv;
#pragma unroll
  for (int j = 0; j < NJ; j++) wj[j][0] *= r;
  g_sweep<G, DC, 1, MASK>(Pf, w, h, wj, skip);
  __syncwarp();
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
  static_for<NA>([&](auto cc) {
    constexpr int c = cc;
    constexpr int xc = idx_of<DC>(c);
    if constexpr (MASK) s.x[xc] = skip ? s.x[xc] : fma(h[0][c], u, s.x[xc]);
    else s.x[xc] = fma(h[0][c], u, s.x[xc]);
  });
  if constexpr (MASK) s.ll = skip ? s.ll : s.ll + (-log(sv) - rr * u);
  else s.ll += -log(sv) - rr * u;
  if constexpr (NISQ) *nisq += rr * u;
}

// A chunk of M correlated rows, decorrelated by the host (rbisk::meas_block): M scalar updates with rows
// H'_a = sum_{b<=a} w_ab H_b and noise D_a.
template <int G, bool DC, bool SYN, bool MASK = false, bool NISQ = false>
__device__ __forceinline__ void g_meas_block(double* Pf, const int l, FilterState& s, const StreamDesc& st, const MeasSrc<SYN>& src, int a0, int M,
                                             long long row, long long sn, const V3& dquat, const V3& chi0, bool skip = false,
                                             double* nisq = nullptr) {
  using GE = Geo<G, DC>;
  constexpr int NA = GE::NA, LD = GE::LD, NJ = GE::NJ;
  const double* W = st.R + row * st.r_stride + RS_W;
  const double* Dg = st.R + row * st.r_stride + RS_D;
  const Own<G, NA> w(l);
  for (int a = 0; a < M; a++) {
    double g[1][NA];
    double wj[NJ][1];
#pragma unroll
    for (int k = 0; k < NA; k++) g[0][k] = 0.0;
#pragma unroll
    for (int j = 0; j < NJ; j++) wj[j][0] = 0.0;
    for (int b = 0; b <= a; b++) {
      const double wt = __ldg(W + (a0 + a) * MAX_MEAS + (a0 + b));
      const double* rp = Pf + pos_of<DC>(st.idx[a0 + b]) * LD;
#pragma unroll
      for (int k = 0; k < NA; k++) g[0][k] = fma(wt, rp[k], g[0][k]);
#pragma unroll
      for (int j = 0; j < NJ; j++) wj[j][0] = fma(wt, rp[w.c[j]], wj[j][0]);  // the lane's own g[c_j], bitwise equal to g[0][c_j]
    }
    double sv = __ldg(Dg + a0 + a), rp_ = 0.0;
    for (int b = 0; b <= a; b++) {
      const double wt = __ldg(W + (a0 + a) * MAX_MEAS + (a0 + b));
      const int ib = st.idx[a0 + b];
      const int pb = pos_of<DC>(ib);
      double gi = g[0][0];
#pragma unroll
      for (int k = 1; k < NA; k++) gi = (pb == k) ? g[0][k] : gi;
      sv = fma(wt, gi, sv);
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
      rp_ = fma(wt, rb, rp_);
    }
    __syncwarp();
    const double r = 1.0 / sv;
#pragma unroll
    for (int j = 0; j < NJ; j++) wj[j][0] *= r;
    g_sweep<G, DC, 1, MASK>(Pf, w, g, wj, skip);
    __syncwarp();
    const double u = rp_ * r;
    static_for<NA>([&](auto cc) {
      constexpr int c = cc;
      constexpr int xc = idx_of<DC>(c);
      if constexpr (MASK) s.x[xc] = skip ? s.x[xc] : fma(g[0][c], u, s.x[xc]);
      else s.x[xc] = fma(g[0][c], u, s.x[xc]);
    });
    if constexpr (MASK) s.ll = skip ? s.ll : s.ll + (-log(sv) - rp_ * u);
    else s.ll += -log(sv) - rp_ * u;
    if constexpr (NISQ) *nisq += rp_ * u;
  }
}

// ---- packed [231][stride] global array <-> the filter's full matrix in shared memory ----
// The lane's columns c, rows k <= c: upper triangle, mirrored into the lower one on load.
template <int G, bool DC>
__device__ __forceinline__ void g_cov_load(double* Pf, const int l, const double* __restrict__ src, long long stride) {
  using GE = Geo<G, DC>;
  constexpr int NA = GE::NA, LD = GE::LD, NJ = GE::NJ;
#pragma unroll
  for (int j = 0; j < NJ; j++) {
    const int c = l + G * j;
    if ((j + 1) * G <= NA || c < NA) {
      const int ic = DC ? (c < 9 ? c + 3 : c + 6) : c;
      const int base = ic * (ic + 1) / 2;
#pragma unroll
      for (int k = 0; k < NA; k++) {
        if (k <= c) {
          const int ik = idx_of<DC>(k);
          const double v = src[(long long)(base + ik) * stride];
          Pf[k * LD + c] = v;
          Pf[c * LD + k] = v;
        }
      }
    }
  }
  __syncwarp();
}
template <int G, bool DC>
__device__ __forceinline__ void g_cov_store(const double* Pf, const int l, double* __restrict__ dst, long long stride, bool active) {
  using GE = Geo<G, DC>;
  constexpr int NA = GE::NA, LD = GE::LD, NJ = GE::NJ;
  if (!active) return;
#pragma unroll
  for (int j = 0; j < NJ; j++) {
    const int c = l + G * j;
    if ((j + 1) * G <= NA || c < NA) {
      const int ic = DC ? (c < 9 ? c + 3 : c + 6) : c;
      const int base = ic * (ic + 1) / 2;
#pragma unroll
      for (int k = 0; k < NA; k++) {
        if (k <= c) {
          const int ik = idx_of<DC>(k);
          dst[(long long)(base + ik) * stride] = Pf[k * LD + c];
        }
      }
    }
  }
}

// RBIS_OP_RECORD: the fields of rbisk::record_fields with the same values; the state is replicated in the group, so lane l
// stores the fields whose output position is l modulo G.  Diagonal (i, i) belongs to the lane of column i: one __syncwarp.
template <int G, bool DC>
__device__ __forceinline__ void g_record_fields(const KParams& p, const double* Pf, const int l, const FilterState& s, const QNoise& qn,
                                                long long row, long long n, bool active, bool imu_seen) {
  constexpr int LD = Geo<G, DC>::LD;
  const long long N = p.N;
  const unsigned long long fields = p.rec.fields;
  double* const d = p.rec.out + row * p.rec.k * N + n;
  __syncwarp();
  static_for<REC_FIELDS>([&](auto fc) {
    constexpr int f = fc;
    if (!((fields >> f) & 1ull)) return;
    const int pos = __popcll(fields & ((1ull << f) - 1));
    if ((pos & (G - 1)) != l) return;
    double v;
    if constexpr (f < 26) {
      v = rec_state_field<f>(s);
    } else {
      constexpr int i = f - 26;
      if constexpr (DC && !is_act(i)) {
        v = imu_seen ? (i < 3 ? qn.q_gyro : qn.q_accel) : p.P[(long long)slot(i, i) * N + n];
      } else {
        constexpr int a = DC ? act_pos(i) : i;
        v = Pf[a * LD + a];
      }
    }
    if (active) d[(long long)pos * N] = v;
  });
  // ---- covariance blocks (see RecK): position popcount(fields) + q, q = jj (jj + 1) / 2 + ii, belongs to lane l when it is l
  // modulo G; the value is the element the SNAPSHOT branch stores for slot(i, j)
  const unsigned cb = p.rec_cov_blocks;
  if (!cb) return;
  const int kf = __popcll(fields), nb = 3 * __popc(cb), nq = nb * (nb + 1) / 2;
  double* const dc = d + (long long)kf * N;
  int q = (l - kf) & (G - 1), jj = 0, ii = q;
  while (ii > jj) { ii -= jj + 1; jj++; }
  for (; q < nq; q += G) {
    const int i = rec_cov_state(cb, ii), j = rec_cov_state(cb, jj);
    double v;
    if constexpr (DC) {
      if (is_act(i) && is_act(j)) v = Pf[act_pos(i) * LD + act_pos(j)];
      else if (j < 3 || (i >= 12 && j < 15)) v = imu_seen ? ((i != j) ? 0.0 : (j < 3 ? qn.q_gyro : qn.q_accel)) : p.P[(long long)slot(i, j) * N + n];
      else v = 0.0;  // kAct.rest: exactly zero in a decoupled filter
    } else {
      v = Pf[i * LD + j];
    }
    if (active) dc[(long long)q * N] = v;
    ii += G;
    while (ii > jj) { ii -= jj + 1; jj++; }
  }
}

// Innovation sets: the entries of rbisk::innov_begin with the same values; entry e of the row belongs to lane e modulo G.
template <int G, bool DC, bool SYN>
__device__ __forceinline__ void g_innov_begin(const InnovK& iv, const double* Pf, const int l, const FilterState& s, const StreamDesc& st,
                                              const MeasSrc<SYN>& src, long long row, long long N, long long n, long long sn, const V3& dquat,
                                              bool active, bool skip) {
  constexpr int LD = Geo<G, DC>::LD;
  double* const d = iv.out + row * iv.k * N + n;
  const int m = st.m;
  const int oy = iv.fields & INNOV_NIS, os = oy + ((iv.fields & INNOV_Y) ? m : 0);
  for (int a = 0; a < m; a++) {
    if ((iv.fields & INNOV_Y) && ((oy + a) & (G - 1)) == l) {
      const double y = innov_y<SYN>(s, st, src, a, row, sn, dquat);
      if (active) d[(long long)(oy + a) * N] = skip ? innov_nan() : y;
    }
    if ((iv.fields & INNOV_S_DIAG) && ((os + a) & (G - 1)) == l) {
      const int pi = pos_of<DC>(st.idx[a]);
      const double v = Pf[pi * LD + pi] + r_diag(st, a, row, N, n);
      if (active) d[(long long)(os + a) * N] = skip ? innov_nan() : v;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// The fused kernel, warp-group mapping.  Same parameter block, op program and semantics as rbisk::rbis_fused_kernel;
// all chunk kinds (aligned triples, one-row chunks, correlated blocks) are compiled in (the indices are run-time
// shared-memory addresses here, so the general paths cost the common program nothing).
// MAXW = warps per CTA the launch may use (register budget: 8 -> 255 registers, 16 -> 128).
// ------------------------------------------------------------------------------------------------
// SYN = true: input rows drawn inside the kernel (KParams::syn), as in rbisk::rbis_fused_kernel.
// REC = true: programs with RBIS_OP_RECORD ops (KParams::rec), as in rbisk::rbis_fused_kernel.
// MASK = true: programs with RBIS_STREAM_SKIP_NAN_ROWS streams (KParams::skip_nan_streams), as in rbisk::rbis_fused_kernel.
// INNOV = true (with REC): programs that write innovation sets (KParams::innov), as in rbisk::rbis_fused_kernel.
// GATE = true (with MASK): programs with NIS gates or INNOV_APPLIED (KParams::gate_streams), as in rbisk::rbis_fused_kernel.
template <int G, bool DC, int MAXW, bool SYN = false, bool REC = false, bool MASK = false, bool INNOV = false, bool GATE = false>
__global__ void __launch_bounds__(32 * MAXW, 1) rbis_group_kernel(const __grid_constant__ KParams p) {
  static_assert(!(MASK && SYN), "MASK instantiations read z from HBM");
  static_assert(!INNOV || REC, "INNOV instantiations are REC instantiations with the innovation path");
  static_assert(!GATE || MASK, "GATE instantiations are MASK instantiations with the gate");
  using GE = Geo<G, DC>;
  constexpr int FPW = GE::FPW, S = GE::S;
  extern __shared__ __align__(16) double smem[];
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int l = lane % G;
  const int wpc = blockDim.x >> 5;
  const long long N = p.N;
  long long n = (((long long)blockIdx.x + p.block_offset) * wpc + warp) * FPW + lane / G;
  const bool active = n < N;
  if (!active) n = N - 1;  // idle groups shadow the last filter and never store
  const bool writer = active && l == 0;
  double* Pf = smem + (size_t)(warp * FPW + lane / G) * S;

  FilterState s;
  static_for<NS>([&](auto i) { s.x[i] = p.vec[(long long)i * N + n]; });
  s.qw = p.quat[n]; s.qx = p.quat[N + n]; s.qy = p.quat[2 * N + n]; s.qz = p.quat[3 * N + n];
  s.ll = p.loglik[n];
  g_cov_load<G, DC>(Pf, l, p.P + n, N);
  bool imu_seen = false;  // DC: an IMU step ran since the (omega,omega) / (a,a) blocks in p.P were current

  auto load_op = [&](long long i) {
    Op o;
    long long w0, w1;
    asm volatile("ld.global.nc.s64 %0, [%1];" : "=l"(w0) : "l"(reinterpret_cast<const long long*>(p.ops + i)));
    asm volatile("ld.global.nc.s64 %0, [%1];" : "=l"(w1) : "l"(reinterpret_cast<const long long*>(p.ops + i) + 1));
    o.kind = (int)(w0 & 0xffffffffll); o.stream = (int)(w0 >> 32); o.row = w1;
    asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(o.dt) : "l"(&p.ops[i].dt));
    return o;
  };
  const long long imu_n = p.imu_map ? (long long)__ldg(p.imu_map + n) : n;
  QNoise qn;
  qn.q_gyro = __ldg(p.q_gyro + n); qn.q_accel = __ldg(p.q_accel + n);
  qn.q_gyro_bias = __ldg(p.q_gyro_bias + n); qn.q_accel_bias = __ldg(p.q_accel_bias + n);

  // Ops are fetched two ahead, and the INPUT ROWS of the next op are prefetched into L1 while the current op runs: with
  // one or two warps per scheduler nothing else hides the latency of a first touch of HBM.
  auto prefetch = [&](const double* ptr) { asm volatile("prefetch.global.L1 [%0];" ::"l"(ptr)); };
  unsigned long long syn_kf = 0;
  double syn_sg = 0.0, syn_sa = 0.0;
  if constexpr (SYN) {
    syn_kf = p.syn.seed ^ ((unsigned long long)(p.syn.first_filter + n) * SYN_K1);
    syn_sg = p.syn.sigma_gyro >= 0 ? p.syn.sigma_gyro : sqrt(__ldg(p.q_gyro + n) / p.syn.dt);
    syn_sa = p.syn.sigma_accel >= 0 ? p.syn.sigma_accel : sqrt(__ldg(p.q_accel + n) / p.syn.dt);
  }
  auto prefetch_inputs = [&](const Op& o) {
    if (o.kind == OP_IMU) {
      const double* base = p.imu + o.row * 6 * p.imu_cols + imu_n;
#pragma unroll
      for (int k = 0; k < 6; k++) prefetch(base + k * p.imu_cols);
    } else if (o.kind == OP_MEAS) {
      const StreamDesc& st = p.streams[o.stream];
      const long long sn = st.map ? (long long)__ldg(st.map + n) : n;
      const double* zb = st.z + o.row * st.m * st.cols + sn;
      for (int a = 0; a < st.m; a++) prefetch(zb + a * st.cols);
      if (st.has_orient) {
        const double* qb = st.quat + o.row * 4 * st.cols + sn;
#pragma unroll
        for (int k = 0; k < 4; k++) prefetch(qb + k * st.cols);
      }
    }
  };
  Op op1 = load_op(0);
  Op op2 = p.n_ops > 1 ? load_op(1) : op1;
  for (long long oi = 0; oi < p.n_ops; oi++) {
    const Op op = op1;
    op1 = op2;
    if (oi + 2 < p.n_ops) op2 = load_op(oi + 2);
    if constexpr (!SYN) {
      if (oi + 1 < p.n_ops) prefetch_inputs(op1);
    }
    if (op.kind == OP_IMU) {
      // ---- IMU process step: same linearisation / state code as the lane-per-filter kernel ----
      const double* base = p.imu + op.row * 6 * p.imu_cols + imu_n;
      const long long Ni = p.imu_cols;
      V3 gyro, acc;
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
      const double dt = op.dt;
      const Q4 q{s.qw, s.qx, s.qy, s.qz};
      const double tx_ = 2 * q.x, ty_ = 2 * q.y, tz_ = 2 * q.z;
      const double twx_ = tx_ * q.w, twy_ = ty_ * q.w, twz_ = tz_ * q.w;
      const double txx_ = tx_ * q.x, txy_ = ty_ * q.x, txz_ = tz_ * q.x;
      const double tyy_ = ty_ * q.y, tyz_ = tz_ * q.y, tzz_ = tz_ * q.z;
      const double R00 = 1 - (tyy_ + tzz_), R01 = txy_ - twz_, R02 = txz_ + twy_;
      const double R10 = txy_ + twz_, R11 = 1 - (txx_ + tzz_), R12 = tyz_ - twx_;
      const double R20 = txz_ - twy_, R21 = tyz_ + twx_, R22 = 1 - (txx_ + tyy_);
      const V3 gb{-p.g_val * R20, -p.g_val * R21, -p.g_val * R22};
      Lin L;
      L.v = {s.x[3], s.x[4], s.x[5]};
      L.wd = {s.x[0] * dt, s.x[1] * dt, s.x[2] * dt};  // omega of the PRIOR state (rbis_update_interface.cpp:38-39)
      L.vd = {L.v.x * dt, L.v.y * dt, L.v.z * dt};
      L.gd = {gb.x * dt, gb.y * dt, gb.z * dt};
      L.dt = dt;
      L.Rd[0] = R00 * dt; L.Rd[1] = R01 * dt; L.Rd[2] = R02 * dt;
      L.Rd[3] = R10 * dt; L.Rd[4] = R11 * dt; L.Rd[5] = R12 * dt;
      L.Rd[6] = R20 * dt; L.Rd[7] = R21 * dt; L.Rd[8] = R22 * dt;
      {
        const double vx = s.x[3], vy = s.x[4], vz = s.x[5];
        s.x[9] += fma(R02, vz, fma(R01, vy, R00 * vx)) * dt;
        s.x[10] += fma(R12, vz, fma(R11, vy, R10 * vx)) * dt;
        s.x[11] += fma(R22, vz, fma(R21, vy, R20 * vx)) * dt;
      }
      imu_seen = true;
      g_cov_propagate<G, DC>(Pf, l, L, qn);
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
      // MASK: a filter whose row is missing passes the warp barriers like every lane and keeps its values
      bool skip = false;
      if constexpr (MASK) {
        if ((p.skip_nan_streams >> op.stream) & 1u) skip = row_missing(st, op.row, sn);
      }
      V3 dquat{0, 0, 0};
      if (st.has_orient) dquat = subtract_quats(src.quat(st, op.row, sn), {s.qw, s.qx, s.qy, s.qz});  // rbis.cpp:199
      // GATE: as in rbisk::rbis_fused_kernel; the G lanes of a group compute the same NIS from the same Pf entries and inputs,
      // so they take the same decision
      const bool missing = skip;
      double gnis = 0.0;
      if constexpr (GATE) {
        if ((p.gate_streams >> op.stream) & 1u) {
          constexpr int LD = GE::LD;
          gnis = gate_nis<SYN>(st, src, s, op.row, N, n, sn, dquat, [&](int a, int b) {
            const int i = min(st.idx[a], st.idx[b]), j = max(st.idx[a], st.idx[b]);  // the upper triangle, as g_record_fields reads it
            return Pf[pos_of<DC>(i) * LD + pos_of<DC>(j)];
          });
          skip = missing || gate_rejects(p, op.stream, n, gnis);
        }
      }
      // INNOV: an innovation set on this stream (uniform branch), as in rbisk::rbis_fused_kernel
      double nisq = 0.0;
      if constexpr (INNOV) {
        if (p.innov[op.stream].out) g_innov_begin<G, DC, SYN>(p.innov[op.stream], Pf, l, s, st, src, op.row, N, n, sn, dquat, active, missing);
      }
      const V3 chi0{s.x[6], s.x[7], s.x[8]};
      for (int ci = 0; ci < st.n_chunks; ci++) {
        const int a0 = st.chunk_start[ci];
        const int fast = st.chunk_fast[ci];
        if (fast >= 0 && fast < 100) g_meas3<G, DC, SYN, MASK, INNOV>(Pf, l, s, st, src, a0, fast, op.row, N, n, sn, dquat, chi0, skip, &nisq);
        else if (fast >= 100) g_meas1<G, DC, SYN, MASK, INNOV>(Pf, l, s, st, src, a0, fast - 100, op.row, N, n, sn, dquat, chi0, skip, &nisq);
        else g_meas_block<G, DC, SYN, MASK, INNOV>(Pf, l, s, st, src, a0, st.chunk_len[ci], op.row, sn, dquat, chi0, skip, &nisq);
      }
      if constexpr (INNOV && GATE) {
        innov_end(p, op, N, n, writer, missing, skip, gnis, nisq);
      } else if constexpr (INNOV) {
        const InnovK& iv = p.innov[op.stream];
        if (iv.out && (iv.fields & INNOV_NIS) && l == 0 && active) iv.out[op.row * iv.k * N + n] = skip ? innov_nan() : nisq;
      }
      if (!MASK || !skip) meas_finish(s, chi0, p.chi_tol, p.ctor_folds_chi, p.renorm);
    } else if (op.kind == OP_SNAPSHOT) {
      // ---- snapshot into ring slot ----
      double* d = p.snap + op.row * SNAP_ROWS * N + n;
      if (writer) {
        static_for<NS>([&](auto i) { d[(long long)i * N] = s.x[i]; });
        d[21 * N] = s.qw; d[22 * N] = s.qx; d[23 * N] = s.qy; d[24 * N] = s.qz;
        d[25 * N] = s.ll;
      }
      double* dc = d + 26 * N;
      g_cov_store<G, DC>(Pf, l, dc, N, active);
      if constexpr (DC) {
        if (active) {
          for (int k = l; k < N_REST; k += G) dc[(long long)c_act.rest[k] * N] = 0.0;
          for (int k = l; k < 12; k += G) {
            const int s_ = c_act.blk[k];
            const int jc = col_of_slot(s_), ir = s_ - jc * (jc + 1) / 2;
            dc[(long long)s_ * N] = imu_seen ? ((ir != jc) ? 0.0 : (jc < 3 ? qn.q_gyro : qn.q_accel)) : p.P[(long long)s_ * N + n];
          }
        }
      }
    } else {
      if constexpr (REC) {
        if (op.kind == OP_RECORD) {
          // ---- record the chosen fields into record row op.row ----
          g_record_fields<G, DC>(p, Pf, l, s, qn, op.row, n, active, imu_seen);
          continue;
        }
      }
      // ---- restore from ring slot ----
      const double* d = p.snap + op.row * SNAP_ROWS * N + n;
      static_for<NS>([&](auto i) { s.x[i] = d[(long long)i * N]; });
      s.qw = d[21 * N]; s.qx = d[22 * N]; s.qy = d[23 * N]; s.qz = d[24 * N];
      s.ll = d[25 * N];
      const double* dc = d + 26 * N;
      __syncwarp();
      g_cov_load<G, DC>(Pf, l, dc, N);
      if constexpr (DC) {
        // the slot's (omega,omega) / (a,a) blocks become the current ones: parked in p.P (this filter's own column)
        if (active)
          for (int k = l; k < 12; k += G) {
            const int s_ = c_act.blk[k];
            p.P[(long long)s_ * N + n] = dc[(long long)s_ * N];
          }
        imu_seen = false;
      }
    }
  }

  if (writer) {
    static_for<NS>([&](auto i) { p.vec[(long long)i * N + n] = s.x[i]; });
    p.quat[n] = s.qw; p.quat[N + n] = s.qx; p.quat[2 * N + n] = s.qy; p.quat[3 * N + n] = s.qz;
    p.loglik[n] = s.ll;
  }
  g_cov_store<G, DC>(Pf, l, p.P + n, N, active);
  if constexpr (DC) {
    if (active && imu_seen)
      for (int k = l; k < 12; k += G) {
        const int s_ = c_act.blk[k];
        const int jc = col_of_slot(s_), ir = s_ - jc * (jc + 1) / 2;
        p.P[(long long)s_ * N + n] = (ir != jc) ? 0.0 : (jc < 3 ? qn.q_gyro : qn.q_accel);
      }
  }
}

template <int G, bool DC>
constexpr int group_smem_bytes(int warps_per_cta) { return warps_per_cta * Geo<G, DC>::FPW * Geo<G, DC>::S * 8; }

}  // namespace grp
}  // namespace rbisk
#endif  // RBIS_GROUP_CUH_
