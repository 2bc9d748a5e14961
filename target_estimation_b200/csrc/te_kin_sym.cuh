// te_kin_sym.cuh -- register-resident symmetric-covariance step of the linear kinematic models with a position measurement
// (uniform velocity n = 6, uniform acceleration n = 9; m = 3) for one lane, streaming straight from / to HBM.
//
// Same idea as te_av_sym.cuh: the step needs only the state and the UPPER triangle of the covariance as input (the
// covariance is symmetric up to rounding in the reference too), so a lane loads 6 + 21 (UV) or 9 + 45 (UA) doubles plus t
// and n_meas instead of the tile's 44 / 92 fields, keeps them in registers, and writes the full matrix back (both halves:
// the stored format stays the reference's full P).  Arithmetic:
//   predict (src/types/uniform_*.cpp updateA, src/kalman.cpp:84-88): per position (r, c), r <= c, of the 3 x 3 block grid the
//       NB x NB macro matrix m' = Abar m Abar^T + Q with Abar = [1 dt h; 0 1 dt; 0 0 1], rows first, then columns -- the
//       reference's order; the mirrored position (c, r) is the transposed macro matrix and is not computed
//   update  (src/kalman.cpp:90-95) with C = [I3 0]:  S = P'[0:3,0:3] + R = L L^T,  Z = L^-1 P'[0:3,:],
//       x += Z^T L^-1 (y - x'[0:3]),  P = P' - Z^T Z   ( = (I - K C) P' with K = P'[:,0:3] S^-1 )
//
// AXIS: the axis-blocked form, for pools in which no registered class couples the x / y / z axes (te_pool::all_axis).  Index
// i = a * 3 + r of the state belongs to axis r = i % 3; every covariance entry (i, j) with i % 3 != j % 3 is then exactly +-0 in
// HBM on every tick (DESIGN.md section 2), so the lane loads and stores only x, the in-axis entries of the upper triangle (3 NB x
// NB blocks: UV 9 of 21, UA 18 of 45), t and n_meas.  tick() runs the same operations in the same order, minus the terms that
// are structurally zero: the off-diagonal blocks of the predict, the off-diagonal entries of S and L (S is diagonal), and every
// term of u, Z, x and P that carries one of them.  Each dropped term is a +-0 product added to a value, so the kept results
// are bit for bit those of the full form (tests/test_gpu_axis_blocks.py).
#pragma once
#include "te_av_sym.cuh"

namespace te {

template <int TYPE, bool AXIS = false>
struct KinSym {
  using MT = Model<TYPE>;
  using LY = Layout<TYPE>;
  static constexpr int N = MT::N, M = 3, B = 3, NB = MT::NB;
  static_assert(MT::M == 3 && MT::B == 3, "position-measurement kinematic models");
  double x[N];
  SymP<N> P;
  double t;
  long long nm;
  // does entry (i, j) carry information?  (the blocked form never touches the others)
  static __device__ __forceinline__ constexpr bool kept(int i, int j) { return !AXIS || i % B == j % B; }

  __device__ __forceinline__ void load(const double* in) {
#pragma unroll
    for (int i = 0; i < N; ++i) x[i] = in[(LY::F_X + i) * TILE];
    t = in[LY::F_T * TILE];
    nm = reinterpret_cast<const long long*>(in)[LY::F_NMEAS * TILE];
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
      for (int j = 0; j < N; ++j)
        if (i <= j && kept(i, j)) P(i, j) = in[(LY::F_P + i * N + j) * TILE];
  }

  // one TargetManager::update(id, dt[, meas]) of this lane's target
  __device__ __forceinline__ void tick(int action, double dt, const double* meas, const double* __restrict__ Q, const double* __restrict__ R) {
    // ---- predict ----
    const double h = 0.5 * dt * dt;   // Ones * 0.5 * dt * dt (uniform_acceleration.cpp:98)
#pragma unroll
    for (int i = 0; i < B; ++i) {
      if (NB == 3) {
        x[i] = x[i] + dt * x[i + B] + h * x[i + 2 * B];
        x[i + B] = x[i + B] + dt * x[i + 2 * B];
      } else {
        x[i] = x[i] + dt * x[i + B];
      }
    }
#pragma unroll
    for (int r = 0; r < B; ++r) {
#pragma unroll
      for (int c = 0; c < B; ++c) {
        if (r <= c && (!AXIS || r == c)) {   // block (r, c) couples axis r with axis c
          double m[NB][NB];
#pragma unroll
          for (int a = 0; a < NB; ++a)
#pragma unroll
            for (int b = 0; b < NB; ++b) m[a][b] = P(a * B + r, b * B + c);
#pragma unroll
          for (int b = 0; b < NB; ++b) {   // A P : rows
            if (NB == 3) {
              m[0][b] = m[0][b] + dt * m[1][b] + h * m[2][b];
              m[1][b] = m[1][b] + dt * m[2][b];
            } else {
              m[0][b] = m[0][b] + dt * m[1][b];
            }
          }
#pragma unroll
          for (int a = 0; a < NB; ++a) {   // (A P) A^T : columns
            if (NB == 3) {
              m[a][0] = m[a][0] + dt * m[a][1] + h * m[a][2];
              m[a][1] = m[a][1] + dt * m[a][2];
            } else {
              m[a][0] = m[a][0] + dt * m[a][1];
            }
          }
#pragma unroll
          for (int a = 0; a < NB; ++a)
#pragma unroll
            for (int b = 0; b < NB; ++b)
              if (r < c || a <= b) P(a * B + r, b * B + c) = m[a][b] + __ldg(&Q[(a * B + r) * N + (b * B + c)]);
        }
      }
    }
    // ---- update ----
    if (action == ACT_UPDATE) {
      Chol<M> ch;
#pragma unroll
      for (int i = 0; i < M; ++i)
#pragma unroll
        for (int j = 0; j < M; ++j)
          if (j <= i && kept(i, j)) ch.at(i, j) = P(j, i) + __ldg(&R[i * M + j]);
      if (AXIS) {   // S diagonal: factor()'s d of column k is S_kk, its inverse square root the only operation left
#pragma unroll
        for (int k = 0; k < M; ++k) ch.L[k][k] = rsqrt(ch.L[k][k]);
      } else {
        ch.factor();
      }
      double u[M];   // L^-1 (y - x'[0:3])
#pragma unroll
      for (int k = 0; k < M; ++k) {
        double s = meas[k] - x[k];
#pragma unroll
        for (int m = 0; m < M; ++m)
          if (m < k && !AXIS) s -= ch.L[k][m] * u[m];
        u[k] = s * ch.L[k][k];
      }
      double Z[M][N];   // L^-1 P'[0:3,:] (forward substitution; the diagonal of ch holds 1 / L_kk); blocked: row k = axis(j) only
#pragma unroll
      for (int j = 0; j < N; ++j) {
#pragma unroll
        for (int k = 0; k < M; ++k) {
          if (!kept(k, j)) continue;
          double s = P(k, j);
#pragma unroll
          for (int m = 0; m < M; ++m)
            if (m < k && !AXIS) s -= ch.L[k][m] * Z[m][j];
          Z[k][j] = s * ch.L[k][k];
        }
#pragma unroll
        for (int k = 0; k < M; ++k)
          if (kept(k, j)) x[j] += Z[k][j] * u[k];
      }
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j)
          if (i <= j && kept(i, j)) {
            double s = P(i, j);
#pragma unroll
            for (int k = 0; k < M; ++k)
              if (kept(k, i)) s -= Z[k][i] * Z[k][j];
            P(i, j) = s;
          }
      nm += 1;      // updateMeasurement (src/target_interface.cpp:142-146)
    }
    t = t + dt;     // updateTime (:148-152)
  }

  // packed: only the upper triangle is written (the pool mirrors it on demand, te_pool.cu ensure_full).  The blocked form is
  // always packed and writes the in-axis entries only -- into the lane's own slot, whose cross-axis entries are already +-0.  A
  // compacting tick writes into another target's old slot: cross_zeros then clears the cross-axis entries of the upper triangle,
  // which the slot's previous owner may have left non-zero (a NaN from a non-finite p0_scale).
  __device__ __forceinline__ void store(double* out, bool packed, bool cross_zeros = false) const {
#pragma unroll
    for (int i = 0; i < N; ++i) out[(LY::F_X + i) * TILE] = x[i];
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
      for (int j = 0; j < N; ++j) {
        if (!kept(i, j)) {
          if (i <= j && cross_zeros) out[(LY::F_P + i * N + j) * TILE] = 0.0;
          continue;
        }
        const double v = i <= j ? P.v[i * N - (i * (i - 1)) / 2 + (j - i)] : P.v[j * N - (j * (j - 1)) / 2 + (i - j)];
        if (i <= j || !packed) out[(LY::F_P + i * N + j) * TILE] = v;
      }
    out[LY::F_T * TILE] = t;
    reinterpret_cast<long long*>(out)[LY::F_NMEAS * TILE] = nm;
  }
};

}  // namespace te
