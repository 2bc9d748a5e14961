// te_sweep.cuh -- sm_100a kernels of te_pool_earliest_intersections, te_pool_nearest_targets and te_pool_gated_targets (te_sweep.cu):
// for each of a chunk of queries, the k targets of the pool with the smallest key, selected on the device without sorting the pool.
//   keys            per query, one 64-bit key per slot, ~0 for a slot that is no candidate; candidates are counted.  Three producers:
//                   sweep_key_kernel (the bits of isolver_kernel's delta for a hit, see sweep_broadcast_kernel), near_key_kernel
//                   (the bits of the distance for a target inside the query sphere) and gate_key_kernel (the bits of the Mahalanobis
//                   d^2 for a target inside the gate)
//   hist / select   radix select over the 96-bit composite (rank(key), slot) in eight 12-bit digits: one histogram of the keys that
//                   still match the selected prefix, then the digit bucket that holds the k-th; refinement stops as soon as that
//                   bucket is small (usually after the second digit)
//   collect         every key at or below the boundary bucket: at most k - 1 + SWEEP_SLACK candidates per query
//   output          after a stable sort of the candidates by slot, then by rank (cub::DeviceSegmentedSort): rows of (id, value)
// A candidate's key orders like its value (a non-negative double's bits order like the value); rank() maps -0.0 to 0, so a delta of
// -0.0 ranks as 0 while the key keeps the bits that query() returns.  Slots are in ascending-id order, so (rank, slot) order is
// (value, id) order.
#pragma once
#include <cub/block/block_scan.cuh>

#include "te_kernels.cuh"

namespace te {

constexpr int SWEEP_MAX_CHUNK = 32;     // queries per chunk (the y dimension of the selection kernels' grids)
constexpr int SWEEP_BINS = 4096;        // 12-bit digits
constexpr int SWEEP_PASSES = 8;         // 96 bits = 64-bit key + 32-bit slot: (rank, slot) is unique, so 8 digits always resolve
constexpr unsigned SWEEP_SLACK = 2048;  // a boundary bucket of at most this many keys is collected whole
constexpr unsigned long long SWEEP_MISS = ~0ull;

__host__ __device__ inline int sweep_shift(int pass) { return 84 - 12 * pass; }   // lowest bit of digit `pass` in the 96-bit composite
__device__ __forceinline__ unsigned long long sweep_rank(unsigned long long key) { return key == 0x8000000000000000ull ? 0ull : key; }

// the selected prefix of the composite (rank, slot): a composite matches when (rank & mk) == pk and (slot & ms) == ps
struct SweepSel {
  unsigned long long pk, mk;
  unsigned ps, ms;
  unsigned kk;     // rank still to place inside the boundary bucket (1-based)
  unsigned take;   // rows to return: min(k, hits)
  int done;
};

__device__ __forceinline__ unsigned sweep_digit(unsigned long long r, unsigned s, int sh) {
  if (sh >= 32) return (unsigned)(r >> (sh - 32)) & (SWEEP_BINS - 1);
  if (sh + 12 <= 32) return (s >> sh) & (SWEEP_BINS - 1);
  return (unsigned)((r << (32 - sh)) | (unsigned long long)(s >> sh)) & (SWEEP_BINS - 1);
}

__device__ __forceinline__ void sweep_set_digit(SweepSel& S, unsigned b, int sh) {
  if (sh >= 32) {
    S.pk |= (unsigned long long)b << (sh - 32);
    S.mk |= (unsigned long long)(SWEEP_BINS - 1) << (sh - 32);
  } else if (sh + 12 <= 32) {
    S.ps |= b << sh;
    S.ms |= (unsigned)(SWEEP_BINS - 1) << sh;
  } else {   // the digit straddles the key's low bits and the slot's high bits
    const int lo = 32 - sh;
    S.pk |= b >> lo;
    S.mk |= (1ull << (12 - lo)) - 1;
    S.ps |= (b & ((1u << lo) - 1)) << sh;
    S.ms |= ((1u << lo) - 1) << sh;
  }
}

// isolver_kernel (dense form: query = slot) computes every target's delta for one sphere; these two kernels feed it and read it.
// The sweep runs the very kernel te_isolver_query runs rather than a second copy of derive_outputs + the quartic: nvcc leaves most FP64
// multiplies and adds unrounded in PTX and ptxas contracts them into FMAs according to the surrounding code, so a copy inlined into
// another kernel gives other bits (measured on angular-rates pools: about half of the deltas differed in the last bits).
static __global__ void sweep_broadcast_kernel(int n, const double* __restrict__ sphere /*t1, x, y, z, radius*/, double* __restrict__ t1,
                                              double* __restrict__ origin, double* __restrict__ radius) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  t1[s] = sphere[0];
  origin[3 * s] = sphere[1];
  origin[3 * s + 1] = sphere[2];
  origin[3 * s + 2] = sphere[3];
  radius[s] = sphere[4];
}

// delta (written by isolver_kernel in place) -> key: the bits of delta for a hit (delta >= 0), SWEEP_MISS otherwise; hits counted
static __global__ void sweep_key_kernel(int n, unsigned long long* __restrict__ keys, unsigned long long* __restrict__ hits) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  bool hit = false;
  if (s < n) {
    const double d = __longlong_as_double((long long)keys[s]);
    hit = d >= 0.0;
    if (!hit) keys[s] = SWEEP_MISS;
  }
  const unsigned b = __ballot_sync(0xffffffffu, hit);
  if ((threadIdx.x & 31) == 0 && b) atomicAdd(hits, (unsigned long long)__popc(b));
}

// position (the first three doubles of gather_estimates_kernel's pose7 of every slot) -> key: the bits of the distance to the point
// for a target inside the sphere (dist <= radius; NaN never is), SWEEP_MISS otherwise; inside targets counted.  Every operation is
// rounded on its own, in this order, so numpy reproduces the distance bit for bit: ((dx^2 + dy^2) + dz^2), then the square root.
// dist >= +0 always, so its bits order like its value and sweep_rank leaves them as they are.
static __global__ void near_key_kernel(int n, const double* __restrict__ pose7, double px, double py, double pz, double radius,
                                       unsigned long long* __restrict__ keys, unsigned long long* __restrict__ inside) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  bool in = false;
  if (s < n) {
    const double dx = __dsub_rn(pose7[7 * (size_t)s], px);
    const double dy = __dsub_rn(pose7[7 * (size_t)s + 1], py);
    const double dz = __dsub_rn(pose7[7 * (size_t)s + 2], pz);
    const double dist = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
    in = dist <= radius;
    keys[s] = in ? (unsigned long long)__double_as_longlong(dist) : SWEEP_MISS;
  }
  const unsigned b = __ballot_sync(0xffffffffu, in);
  if ((threadIdx.x & 31) == 0 && b) atomicAdd(inside, (unsigned long long)__popc(b));
}

// The gating query (te_pool_gated_targets) splits its work in two: gate_prep_kernel, once per run of queries at the same t1, turns
// every slot's covariance into the Cholesky factor of its position innovation covariance S; gate_key_kernel, once per query, turns
// the slot's position (pose7 of gather_estimates_kernel) and that factor into the Mahalanobis d^2.  Every operation is rounded on
// its own (__dadd_rn / __dmul_rn / __ddiv_rn / __dsqrt_rn) in the order of the contract in include/te_pool.h, so numpy reproduces
// every bit; left to ptxas, the multiplies and adds would be contracted into FMAs according to the surrounding code.

// upper-triangle read of a symmetric matrix: entry (r, c) with r > c comes from (c, r), which is what the packed kernels keep current
__device__ __forceinline__ int gate_upper(int r, int c, int n) { return r <= c ? r * n + c : c * n + r; }

// per slot: the six entries L00, L10, L20, L11, L21, L22 of the factor of S = C + R[0:3, 0:3] into chol[6 * slot], L00 = NaN when
// the factor does not exist (a radicand <= 0 or NaN), which makes every d^2 of the slot NaN.  use_t1 == 0: C = P[0:3, 0:3].
// use_t1 != 0: C = the position block of A(tau) P A(tau)^T + Q with tau = t1 - t, evaluated like predict_kinematic (rows, then
// columns) over the position-derivative offsets: (0, 3) UV, (0, 3, 6) UA, (0, 6, 12) AR, (0, 6) AV -- the position rows of
// predict_av's Jacobian are [I 0 tau*I 0], so the position block of F P F^T depends on those rows only.  One thread per slot: the
// 32 lanes of a warp read one tile, each field of it one 256 B segment.
template <int TYPE>
__global__ void __launch_bounds__(256) gate_prep_kernel(int n, const double* __restrict__ tiles, const uint16_t* __restrict__ cls,
                                                        const double* __restrict__ Qtab, const double* __restrict__ Rtab, int use_t1,
                                                        double t1, double* __restrict__ chol) {
  using MT = Model<TYPE>;
  using LY = Layout<TYPE>;
  constexpr int N = MT::N, M = MT::M;
  constexpr int NO = (TYPE == UNIFORM_VELOCITY || TYPE == ANGULAR_VELOCITIES) ? 2 : 3;   // offsets
  constexpr int OS = (TYPE == UNIFORM_VELOCITY || TYPE == UNIFORM_ACCELERATION) ? 3 : 6;  // offset stride
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  const double* rec = tiles + (size_t)(s / TILE) * LY::TILE_DOUBLES + (s % TILE);
  const int c = (int)cls[s];
  const double* Q = Qtab + (size_t)c * N * N;
  const double* R = Rtab + (size_t)c * M * M;
  double tau = 0.0, h = 0.0;
  if (use_t1) {
    tau = __dsub_rn(t1, rec[LY::F_T * TILE]);
    h = __dmul_rn(__dmul_rn(0.5, tau), tau);
  }
  auto P = [&](int r, int cc) { return rec[(LY::F_P + gate_upper(r, cc, N)) * TILE]; };
  double S[3][3];   // the lower triangle (a >= b) is what the factor reads
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int b = 0; b <= a; ++b) {
      double C;
      if (!use_t1) {
        C = P(a, b);
      } else {
        double r[NO];
#pragma unroll
        for (int v = 0; v < NO; ++v) {
          r[v] = __dadd_rn(P(a, v * OS + b), __dmul_rn(tau, P(OS + a, v * OS + b)));
          if constexpr (NO == 3) r[v] = __dadd_rn(r[v], __dmul_rn(h, P(2 * OS + a, v * OS + b)));
        }
        C = __dadd_rn(r[0], __dmul_rn(tau, r[1]));
        if constexpr (NO == 3) C = __dadd_rn(C, __dmul_rn(h, r[NO - 1]));
        C = __dadd_rn(C, __ldg(&Q[gate_upper(a, b, N)]));
      }
      S[a][b] = __dadd_rn(C, __ldg(&R[gate_upper(a, b, M)]));
    }
  const double l00 = __dsqrt_rn(S[0][0]);
  const double l10 = __ddiv_rn(S[1][0], l00);
  const double l20 = __ddiv_rn(S[2][0], l00);
  const double rad1 = __dsub_rn(S[1][1], __dmul_rn(l10, l10));
  const double l11 = __dsqrt_rn(rad1);
  const double l21 = __ddiv_rn(__dsub_rn(S[2][1], __dmul_rn(l20, l10)), l11);
  const double rad2 = __dsub_rn(__dsub_rn(S[2][2], __dmul_rn(l20, l20)), __dmul_rn(l21, l21));
  const double l22 = __dsqrt_rn(rad2);
  const bool ok = S[0][0] > 0.0 && rad1 > 0.0 && rad2 > 0.0;   // false for NaN too
  double* o = chol + 6 * (size_t)s;
  o[0] = ok ? l00 : __longlong_as_double(0x7ff8000000000000ll);
  o[1] = l10;
  o[2] = l20;
  o[3] = l11;
  o[4] = l21;
  o[5] = l22;
}

// d^2 = (w0^2 + w1^2) + w2^2 of slot s for the measured position z, w = L^-1 (p - z) by forward substitution over the slot's position
// (pose7 as in near_key_kernel) and factor (gate_prep_kernel): steps 4 and 5 of the gating contract in include/te_pool.h, in one
// place for gate_key_kernel and the association's candidate search (te_assoc.cuh).  NaN when the slot has no factor.
__device__ __forceinline__ double gate_d2(const double* __restrict__ pose7, const double* __restrict__ chol, size_t s, double zx, double zy,
                                          double zz) {
  const double* L = chol + 6 * s;
  const double d0 = __dsub_rn(pose7[7 * s], zx);
  const double d1 = __dsub_rn(pose7[7 * s + 1], zy);
  const double d2 = __dsub_rn(pose7[7 * s + 2], zz);
  const double w0 = __ddiv_rn(d0, L[0]);
  const double w1 = __ddiv_rn(__dsub_rn(d1, __dmul_rn(L[1], w0)), L[3]);
  const double w2 = __ddiv_rn(__dsub_rn(__dsub_rn(d2, __dmul_rn(L[2], w0)), __dmul_rn(L[4], w1)), L[5]);
  return __dadd_rn(__dadd_rn(__dmul_rn(w0, w0), __dmul_rn(w1, w1)), __dmul_rn(w2, w2));
}

// position and factor -> key: the bits of d^2 (gate_d2) for a target inside the gate (d^2 <= gate; NaN -- no factor -- never is),
// SWEEP_MISS otherwise; inside targets counted.  d^2 >= +0 always, so its bits order like its value.
static __global__ void gate_key_kernel(int n, const double* __restrict__ pose7, const double* __restrict__ chol, double zx, double zy,
                                       double zz, double gate, unsigned long long* __restrict__ keys,
                                       unsigned long long* __restrict__ inside) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  bool in = false;
  if (s < n) {
    const double m2 = gate_d2(pose7, chol, (size_t)s, zx, zy, zz);
    in = m2 <= gate;
    keys[s] = in ? (unsigned long long)__double_as_longlong(m2) : SWEEP_MISS;
  }
  const unsigned b = __ballot_sync(0xffffffffu, in);
  if ((threadIdx.x & 31) == 0 && b) atomicAdd(inside, (unsigned long long)__popc(b));
}

// per sphere: rows to return and the state of the selection.  Nothing to select when every hit is returned (hits <= k: the empty
// prefix matches them all) or none is.
static __global__ void sweep_init_kernel(int nq, unsigned k, const unsigned long long* __restrict__ hits, SweepSel* __restrict__ sel,
                                         unsigned* __restrict__ count) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nq) return;
  const unsigned long long h = hits[c];
  const unsigned take = h < k ? (unsigned)h : k;
  sel[c] = SweepSel{0ull, 0ull, 0u, 0u, take, take, (take == 0 || h <= k) ? 1 : 0};
  count[c] = 0;
}

// histogram of digit `sh` over the hits of sphere blockIdx.y that match the selected prefix
static __global__ void __launch_bounds__(256) sweep_hist_kernel(const unsigned long long* __restrict__ keys, int n,
                                                                const SweepSel* __restrict__ sel, int sh, unsigned* __restrict__ hist) {
  const int c = blockIdx.y;
  const SweepSel S = sel[c];
  if (S.done) return;
  __shared__ unsigned h[SWEEP_BINS];
  for (int i = threadIdx.x; i < SWEEP_BINS; i += blockDim.x) h[i] = 0;
  __syncthreads();
  const unsigned long long* kc = keys + (size_t)c * n;
  const int lane = threadIdx.x & 31;
  for (long long base = (long long)blockIdx.x * blockDim.x; base < n; base += (long long)gridDim.x * blockDim.x) {   // uniform trip count
    const int s = (int)base + threadIdx.x;
    const unsigned long long key = s < n ? kc[s] : SWEEP_MISS;
    const unsigned long long r = sweep_rank(key);
    const bool m = key != SWEEP_MISS && (r & S.mk) == S.pk && ((unsigned)s & S.ms) == S.ps;
    const unsigned act = __ballot_sync(0xffffffffu, m);
    if (m) {   // one shared atomic per distinct digit of the warp: the first digits of the keys are few
      const unsigned dg = sweep_digit(r, (unsigned)s, sh);
      const unsigned peers = __match_any_sync(act, dg);
      if (lane == __ffs(peers) - 1) atomicAdd(&h[dg], (unsigned)__popc(peers));
    }
  }
  __syncthreads();
  unsigned* hc = hist + (size_t)c * SWEEP_BINS;
  for (int i = threadIdx.x; i < SWEEP_BINS; i += blockDim.x)
    if (h[i]) atomicAdd(&hc[i], h[i]);
}

// the digit bucket of sphere blockIdx.x that holds its kk-th matching key; the histogram is left zeroed for the next digit
static __global__ void __launch_bounds__(1024) sweep_select_kernel(unsigned* __restrict__ hist, SweepSel* __restrict__ sel, int sh) {
  const int c = blockIdx.x;
  if (sel[c].done) return;
  const unsigned kk = sel[c].kk;
  unsigned* hc = hist + (size_t)c * SWEEP_BINS;
  const int b0 = 4 * threadIdx.x;
  unsigned v[4], sum = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) { v[j] = hc[b0 + j]; sum += v[j]; }
  typedef cub::BlockScan<unsigned, 1024> Scan;
  __shared__ typename Scan::TempStorage tmp;
  unsigned pre;
  Scan(tmp).ExclusiveSum(sum, pre);   // (its barrier orders every thread's read of sel[c] before the one write below)
  if (pre < kk && kk <= pre + sum) {
    unsigned acc = pre;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (kk <= acc + v[j]) {
        SweepSel S = sel[c];
        sweep_set_digit(S, (unsigned)(b0 + j), sh);
        S.kk = kk - acc;
        S.done = (v[j] <= SWEEP_SLACK || v[j] == S.kk) ? 1 : 0;   // small enough, or taken whole
        sel[c] = S;
        break;
      }
      acc += v[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) hc[b0 + j] = 0;
}

// the candidates of sphere blockIdx.y: every hit whose composite is at or below the boundary bucket, at [c * cap, c * cap + count[c])
static __global__ void __launch_bounds__(256) sweep_collect_kernel(const unsigned long long* __restrict__ keys, int n,
                                                                   const SweepSel* __restrict__ sel, unsigned cap,
                                                                   unsigned* __restrict__ count, unsigned long long* __restrict__ cand_rank,
                                                                   unsigned* __restrict__ cand_slot) {
  const int c = blockIdx.y;
  const SweepSel S = sel[c];
  if (S.take == 0) return;
  const unsigned long long* kc = keys + (size_t)c * n;
  const int lane = threadIdx.x & 31;
  for (long long base = (long long)blockIdx.x * blockDim.x; base < n; base += (long long)gridDim.x * blockDim.x) {
    const int s = (int)base + threadIdx.x;
    const unsigned long long key = s < n ? kc[s] : SWEEP_MISS;
    const unsigned long long r = sweep_rank(key), rm = r & S.mk;
    const unsigned sm = (unsigned)s & S.ms;
    const bool m = key != SWEEP_MISS && (rm < S.pk || (rm == S.pk && sm <= S.ps));
    const unsigned b = __ballot_sync(0xffffffffu, m);
    if (!b) continue;
    unsigned at = 0;
    if (lane == 0) at = atomicAdd(&count[c], (unsigned)__popc(b));
    at = __shfl_sync(0xffffffffu, at, 0) + __popc(b & ((1u << lane) - 1));
    if (m && at < cap) {
      cand_rank[(size_t)c * cap + at] = r;
      cand_slot[(size_t)c * cap + at] = (unsigned)s;
    }
  }
}

// segment c of the sort = sphere c's candidates; more than cap would mean a broken selection: flagged, never read past
static __global__ void sweep_segments_kernel(int nq, unsigned cap, const unsigned* __restrict__ count, int* __restrict__ seg_begin,
                                             int* __restrict__ seg_end, int* __restrict__ overflow) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nq) return;
  seg_begin[c] = (int)(c * cap);
  seg_end[c] = (int)(c * cap + (count[c] < cap ? count[c] : cap));
  if (count[c] > cap) *overflow = 1;
}

// rows of sphere blockIdx.y: the first `take` sorted candidates (id through the pool's cold ids, delta as the sweep computed it), then
// the sentinel rows
static __global__ void sweep_output_kernel(int k, const SweepSel* __restrict__ sel, const unsigned* __restrict__ slot_sorted, unsigned cap,
                                           const unsigned long long* __restrict__ keys, int n, const uint32_t* __restrict__ ids,
                                           uint32_t* __restrict__ ids_out, double* __restrict__ delta_out) {
  const int c = blockIdx.y;
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= k) return;
  const size_t o = (size_t)c * k + r;
  if ((unsigned)r < sel[c].take) {
    const unsigned s = slot_sorted[(size_t)c * cap + r];
    ids_out[o] = ids[s];
    delta_out[o] = __longlong_as_double((long long)keys[(size_t)c * n + s]);
  } else {
    ids_out[o] = 0xFFFFFFFFu;
    delta_out[o] = -1.0;
  }
}

}  // namespace te
