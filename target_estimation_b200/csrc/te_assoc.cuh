// te_assoc.cuh -- sm_100a kernels of the association of unlabelled detections (te_assoc.cu; contract in include/te_pool.h).
//   candidates   a multi-level uniform grid over every slot's gate box, built per call: assoc_box_kernel (which slots take part,
//                and the extent the grid is sized from), assoc_grid_kernel (origin, level-0 edge, level cap), assoc_cell_kernel
//                (one key per cell a box overlaps, at most 8, or the everywhere list), a radix sort of the keys, then
//                assoc_lookup_kernel: one warp per detection, one cell per non-empty level plus the everywhere list, the K best
//                candidates by (d^2, slot) kept across the warp's lanes and every candidate counted.  d^2 is gate_d2 (te_sweep.cuh),
//                the gating query's arithmetic, so candidate rows are gatedTargets' rows bit for bit.
//   matching     greedy on the edges sorted by (d^2, id, j), run as rounds of mutual best edges: assoc_edge_*_kernel sort the
//                edges per target by (d^2, j) and give every target a dense index, assoc_propose_kernel moves every unmatched
//                detection and target to its best edge to an unmatched partner, assoc_match_kernel takes the mutual pairs.
//   update       assoc_dt_kernel: dt = t1 - t of each named slot, then the scatter and step launch of te_pool_step_ids.
// The exactness argument of the index (why a target with computed d^2 <= gate is never missed) is in DESIGN.md section 4.10.
#pragma once
#include "te_sweep.cuh"

namespace te {

constexpr int ASSOC_CELL_BITS = 19;                       // cell coordinates per axis and level: [0, 2^19)
constexpr long long ASSOC_CELLS = 1LL << ASSOC_CELL_BITS;
constexpr int ASSOC_MAX_LEVELS = 32;                      // 5 bits of the key
constexpr int ASSOC_CELLS_PER_SLOT = 8;
constexpr unsigned long long ASSOC_NO_KEY = ~0ull;
enum { ASSOC_OUT = 0, ASSOC_GRID = 1, ASSOC_EVERYWHERE = 2 };   // per-slot kind

// the grid of one call, computed on the device: ordered-bits extremes of the boxes, then the parameters
struct AssocGrid {
  unsigned long long lo_min[3], hi_max[3], w_min, w_max;   // ordered bits (assoc_ord) of min lo, max hi, min / max box width
  double o[3];                                              // origin: min lo per axis
  double inv[ASSOC_MAX_LEVELS];                             // 1 / edge of level l = 2^-(e0 + l), exact
  int levels;                                               // level cap
  unsigned level_mask;                                      // levels that hold a key
  unsigned n_every;                                         // slots on the everywhere list
};

// a double's bits mapped so that unsigned order is numeric order (NaN excluded by the callers)
__device__ __forceinline__ unsigned long long assoc_ord(double v) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double assoc_unord(unsigned long long k) {
  return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

// The gate box of a slot: lo / hi per axis, true when every bound is finite.  Half-width h_a = ((sqrt(S_aa) + 2^-530) *
// (sqrt(gate) + 2^-530)) * (1 + 2^-40) with S_aa = row a of L times itself; each operation rounded on its own.  The two 2^-530
// terms cover underflow in the forward substitution and the squares, the factor every rounding (DESIGN.md 4.10).
__device__ __forceinline__ bool assoc_box(const double* __restrict__ pose7, const double* __restrict__ chol, size_t s, double sg,
                                          double lo[3], double hi[3]) {
  const double* L = chol + 6 * s;
  double S[3];
  S[0] = __dmul_rn(L[0], L[0]);
  S[1] = __dadd_rn(__dmul_rn(L[1], L[1]), __dmul_rn(L[3], L[3]));
  S[2] = __dadd_rn(__dadd_rn(__dmul_rn(L[2], L[2]), __dmul_rn(L[4], L[4])), __dmul_rn(L[5], L[5]));
  const double tiny = 0x1p-530;
  bool fin = true;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const double h = __dmul_rn(__dmul_rn(__dadd_rn(__dsqrt_rn(S[a]), tiny), __dadd_rn(sg, tiny)), 1.0 + 0x1p-40);
    const double p = pose7[7 * s + a];
    lo[a] = __dsub_rn(p, h);
    hi[a] = __dadd_rn(p, h);
    fin = fin && isfinite(lo[a]) && isfinite(hi[a]);
  }
  return fin;
}

// cell coordinate of x at the level of inverse edge inv: floor((x - o) * inv), each operation rounded, so that it is monotone in x
// (the argument of DESIGN.md 4.10 rests on that); -1 below the grid, ASSOC_CELLS above it or for a non-finite value
__device__ __forceinline__ long long assoc_cell(double x, double o, double inv) {
  const double c = floor(__dmul_rn(__dsub_rn(x, o), inv));
  if (!(c >= 0.0)) return -1;
  return c < (double)ASSOC_CELLS ? (long long)c : ASSOC_CELLS;
}
__device__ __forceinline__ unsigned long long assoc_key(int level, long long ix, long long iy, long long iz) {
  return ((unsigned long long)level << (3 * ASSOC_CELL_BITS)) | ((unsigned long long)ix << (2 * ASSOC_CELL_BITS)) |
         ((unsigned long long)iy << ASSOC_CELL_BITS) | (unsigned long long)iz;
}

// per slot: kind (out: no factor, a NaN position or t > t1 -- never a candidate; everywhere: a non-finite box; grid otherwise),
// and the extremes of the grid slots' boxes, reduced over the warp first (a million slots' atomics on eight words would queue)
template <int TYPE>
__global__ void __launch_bounds__(256) assoc_box_kernel(int n, const double* __restrict__ tiles, const double* __restrict__ pose7,
                                                        const double* __restrict__ chol, double t1, double sg, uint8_t* __restrict__ kind,
                                                        AssocGrid* __restrict__ g) {
  using LY = Layout<TYPE>;
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long lo_k[3] = {~0ull, ~0ull, ~0ull}, hi_k[3] = {0ull, 0ull, 0ull}, wmin = ~0ull, wmax = 0ull;
  if (s < n) {
    const double t = tiles[(size_t)(s / TILE) * LY::TILE_DOUBLES + LY::F_T * TILE + (s % TILE)];
    const double* p = pose7 + 7 * (size_t)s;
    uint8_t k = ASSOC_OUT;
    if (t <= t1 && !isnan(chol[6 * (size_t)s]) && !isnan(p[0]) && !isnan(p[1]) && !isnan(p[2])) {
      double lo[3], hi[3];
      if (!assoc_box(pose7, chol, (size_t)s, sg, lo, hi)) {
        k = ASSOC_EVERYWHERE;
      } else {
        k = ASSOC_GRID;
        double w = 0.0;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          lo_k[a] = assoc_ord(lo[a]);
          hi_k[a] = assoc_ord(hi[a]);
          w = fmax(w, __dsub_rn(hi[a], lo[a]));
        }
        wmin = wmax = assoc_ord(w);
      }
    }
    kind[s] = k;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      lo_k[a] = min(lo_k[a], __shfl_xor_sync(0xffffffffu, lo_k[a], o));
      hi_k[a] = max(hi_k[a], __shfl_xor_sync(0xffffffffu, hi_k[a], o));
    }
    wmin = min(wmin, __shfl_xor_sync(0xffffffffu, wmin, o));
    wmax = max(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
  }
  if ((threadIdx.x & 31) == 0 && wmax != 0ull) {   // (wmax > 0: the warp holds a grid slot)
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      atomicMin(&g->lo_min[a], lo_k[a]);
      atomicMax(&g->hi_max[a], hi_k[a]);
    }
    atomicMin(&g->w_min, wmin);
    atomicMax(&g->w_max, wmax);
  }
}

// the grid from the extremes (one thread): origin = min lo; level-0 edge = the power of two at or above max(min width,
// extent * 2^-18), so level 0 spans the extent in fewer than 2^19 cells; levels up to the first whose edge covers the widest box
static __global__ void assoc_grid_kernel(AssocGrid* __restrict__ g) {
  if (g->hi_max[0] == 0ull) {   // no grid slot
    g->levels = 0;
    return;
  }
  double ext = 0.0;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    g->o[a] = assoc_unord(g->lo_min[a]);
    ext = fmax(ext, assoc_unord(g->hi_max[a]) - g->o[a]);
  }
  const double want = fmax(fmax(assoc_unord(g->w_min), ext * 0x1p-18), 0x1p-1000);
  int e0;
  frexp(want, &e0);   // want = m * 2^e0, 0.5 <= m < 1: 2^e0 >= want
  const double wmax = assoc_unord(g->w_max);
  int levels = 1;
  while (levels < ASSOC_MAX_LEVELS && ldexp(1.0, e0 + levels - 1) < wmax) ++levels;
  g->levels = levels;
  for (int l = 0; l < ASSOC_MAX_LEVELS; ++l) g->inv[l] = ldexp(1.0, -(e0 + l));
}

// per slot: the keys of the cells its box overlaps at the lowest level whose cells it spans at most two of per axis (up to 8
// keys, ASSOC_NO_KEY for the rest), or the everywhere list when no level fits or a cell lies outside the grid
static __global__ void __launch_bounds__(256) assoc_cell_kernel(int n, const double* __restrict__ pose7, const double* __restrict__ chol,
                                                                double sg, const uint8_t* __restrict__ kind, AssocGrid* __restrict__ g,
                                                                unsigned long long* __restrict__ keys, unsigned* __restrict__ vals,
                                                                unsigned* __restrict__ every) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned level_bit = 0;
  if (s < n) {
    unsigned long long* ks = keys + (size_t)ASSOC_CELLS_PER_SLOT * s;
    unsigned* vs = vals + (size_t)ASSOC_CELLS_PER_SLOT * s;
#pragma unroll
    for (int c = 0; c < ASSOC_CELLS_PER_SLOT; ++c) {
      ks[c] = ASSOC_NO_KEY;
      vs[c] = (unsigned)s;
    }
    if (kind[s] != ASSOC_OUT) {
      if (kind[s] == ASSOC_GRID) {
        double lo[3], hi[3];
        assoc_box(pose7, chol, (size_t)s, sg, lo, hi);
        for (int l = 0; l < g->levels && !level_bit; ++l) {
          long long c0[3], c1[3];
          bool fits = true;
#pragma unroll
          for (int a = 0; a < 3; ++a) {
            c0[a] = assoc_cell(lo[a], g->o[a], g->inv[l]);
            c1[a] = assoc_cell(hi[a], g->o[a], g->inv[l]);
            fits = fits && c0[a] >= 0 && c1[a] < ASSOC_CELLS && c1[a] - c0[a] <= 1;
          }
          if (!fits) continue;
          int c = 0;
          for (long long x = c0[0]; x <= c1[0]; ++x)
            for (long long y = c0[1]; y <= c1[1]; ++y)
              for (long long z = c0[2]; z <= c1[2]; ++z) ks[c++] = assoc_key(l, x, y, z);
          level_bit = 1u << l;
        }
      }
      if (!level_bit) every[atomicAdd(&g->n_every, 1u)] = (unsigned)s;
    }
  }
  const unsigned mask = __reduce_or_sync(0xffffffffu, level_bit);   // one atomic per warp
  if ((threadIdx.x & 31) == 0 && mask) atomicOr(&g->level_mask, mask);
}

// (d^2 bits, slot) order
__device__ __forceinline__ bool assoc_better(unsigned long long d, unsigned s, unsigned long long bd, unsigned bs) {
  return d < bd || (d == bd && s < bs);
}

// one batch of up to 32 slots of a warp's detection, lane l holding slot s (ok = it holds one): test, count, and insert the
// candidates into the warp's sorted list (lane r = the r-th best by (d^2, slot); only the first K are kept)
__device__ __forceinline__ void assoc_offer(bool ok, unsigned s, const double* __restrict__ pose7, const double* __restrict__ chol, double zx,
                                            double zy, double zz, double gate, int K, int lane, unsigned& found, unsigned long long& bd,
                                            unsigned& bs) {
  double d2 = 0.0;
  bool cand = false;
  if (ok) {
    d2 = gate_d2(pose7, chol, (size_t)s, zx, zy, zz);
    cand = d2 <= gate;
  }
  found += cand ? 1u : 0u;
  unsigned m = __ballot_sync(0xffffffffu, cand);
  const unsigned long long my = (unsigned long long)__double_as_longlong(d2);
  while (m) {
    const int src = __ffs(m) - 1;
    m &= m - 1;
    const unsigned long long cd = __shfl_sync(0xffffffffu, my, src);
    const unsigned cs = __shfl_sync(0xffffffffu, s, src);
    const unsigned worse = __ballot_sync(0xffffffffu, assoc_better(cd, cs, bd, bs));   // lanes [pos, 32): a suffix
    if (!((worse >> (K - 1)) & 1u)) continue;                                          // not among the K best
    const int pos = __ffs(worse) - 1;
    const unsigned long long ud = __shfl_up_sync(0xffffffffu, bd, 1);
    const unsigned us = __shfl_up_sync(0xffffffffu, bs, 1);
    if (lane == pos) { bd = cd; bs = cs; }
    else if (lane > pos) { bd = ud; bs = us; }
  }
}

// One warp per detection j (position det[j * stride + 0 .. 2]): every slot in the detection's cell of each non-empty level and
// every slot of the everywhere list is met once; a candidate has d^2 <= gate.  Lane r keeps the r-th best candidate by (d^2,
// slot); rows 0 .. K - 1 of the detection receive slot and d^2 (ASSOC_NO_KEY-slot / -1 after the candidates), count[j] the
// number of candidates.
static __global__ void __launch_bounds__(256) assoc_lookup_kernel(int q, const double* __restrict__ det, int stride, double gate, int K,
                                                                  const double* __restrict__ pose7, const double* __restrict__ chol,
                                                                  const AssocGrid* __restrict__ g, const unsigned long long* __restrict__ keys,
                                                                  const unsigned* __restrict__ vals, long long n_keys,
                                                                  const unsigned* __restrict__ every, unsigned* __restrict__ slot_out,
                                                                  double* __restrict__ d2_out, long long* __restrict__ count) {
  const unsigned j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;   // (unsigned: a sign word would be kept live across gate_d2's calls)
  const int lane = threadIdx.x & 31;
  if (j >= (unsigned)q) return;   // (whole warps)
  const double zx = det[(size_t)j * stride], zy = det[(size_t)j * stride + 1], zz = det[(size_t)j * stride + 2];
  unsigned long long bd = ~0ull;   // this lane's entry of the sorted best list
  unsigned bs = ~0u;
  unsigned found = 0;
  const unsigned mask = g->levels > 0 ? g->level_mask : 0u;
  for (int l = 0; l < ASSOC_MAX_LEVELS; ++l) {
    if (!((mask >> l) & 1u)) continue;
    const long long cx = assoc_cell(zx, g->o[0], g->inv[l]), cy = assoc_cell(zy, g->o[1], g->inv[l]), cz = assoc_cell(zz, g->o[2], g->inv[l]);
    if (cx < 0 || cy < 0 || cz < 0 || cx >= ASSOC_CELLS || cy >= ASSOC_CELLS || cz >= ASSOC_CELLS) continue;   // no box reaches it
    const unsigned long long key = assoc_key(l, cx, cy, cz);
    long long lo = 0, hi = n_keys;   // lower bound of key (every lane the same search: broadcast loads)
    while (lo < hi) {
      const long long mid = (lo + hi) >> 1;
      if (keys[mid] < key) lo = mid + 1; else hi = mid;
    }
    for (long long base = lo;; base += 32) {
      const long long i = base + lane;
      const bool ok = i < n_keys && keys[i] == key;
      assoc_offer(ok, ok ? vals[i] : 0u, pose7, chol, zx, zy, zz, gate, K, lane, found, bd, bs);
      if (__ballot_sync(0xffffffffu, ok) != 0xffffffffu) break;
    }
  }
  const unsigned n_every = g->n_every;
  for (unsigned base = 0; base < n_every; base += 32) {
    const bool ok = base + lane < n_every;
    assoc_offer(ok, ok ? every[base + lane] : 0u, pose7, chol, zx, zy, zz, gate, K, lane, found, bd, bs);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) found += __shfl_xor_sync(0xffffffffu, found, o);   // (< 2^32 slots)
  if (lane < K) {
    const bool has = bs != ~0u;
    slot_out[(size_t)j * K + lane] = has ? bs : ~0u;
    d2_out[(size_t)j * K + lane] = has ? __longlong_as_double((long long)bd) : -1.0;
  }
  if (lane == 0) count[j] = found;
}

// candidate rows: slot -> id (0xFFFFFFFF after the candidates)
static __global__ void assoc_slot_ids_kernel(long long n, const unsigned* __restrict__ slot, const uint32_t* __restrict__ ids,
                                             uint32_t* __restrict__ out) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n) out[i] = slot[i] == ~0u ? 0xFFFFFFFFu : ids[slot[i]];
}

// ---- matching -------------------------------------------------------------------------------------------------------------
// edge e = row e of the q x K rows (detection e / K); a row with d^2 < 0 (the -1 of an empty row) is no edge.  Sort keys: the bits
// of d^2 (a non-negative double's bits order like its value; no edge: ~0), then the target key (no edge: 2^32).
static __global__ void assoc_edge_init_kernel(long long E, const double* __restrict__ d2, unsigned long long* __restrict__ dkey,
                                              unsigned* __restrict__ idx) {
  const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (e >= E) return;
  dkey[e] = d2[e] >= 0.0 ? (unsigned long long)__double_as_longlong(d2[e]) : ~0ull;
  idx[e] = (unsigned)e;
}
static __global__ void assoc_edge_tkey_kernel(long long E, const unsigned* __restrict__ idx, const double* __restrict__ d2,
                                              const unsigned* __restrict__ tgt, unsigned long long* __restrict__ tkey) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= E) return;
  const unsigned e = idx[i];
  tkey[i] = d2[e] >= 0.0 ? (unsigned long long)tgt[e] : (1ull << 32);
}
// edges in (target, d^2, j) order: head[i] = 1 where a target's run starts
static __global__ void assoc_edge_head_kernel(long long E, const unsigned long long* __restrict__ tkey, int* __restrict__ head) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= E) return;
  head[i] = (tkey[i] < (1ull << 32) && (i == 0 || tkey[i - 1] != tkey[i])) ? 1 : 0;
}
// tix[i] = inclusive sum of head: target t = tix[i] - 1 owns edges [seg_begin[t], seg_end[t]); row_tgt[e] = t (-1: no edge)
static __global__ void assoc_edge_seg_kernel(long long E, int K, const unsigned long long* __restrict__ tkey, const int* __restrict__ tix,
                                             const unsigned* __restrict__ idx, int* __restrict__ seg_begin, int* __restrict__ seg_end,
                                             int* __restrict__ tgt_ptr, int* __restrict__ tgt_match, int* __restrict__ row_tgt) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= E) return;
  if (tkey[i] >= (1ull << 32)) {
    row_tgt[idx[i]] = -1;
    return;
  }
  const int t = tix[i] - 1;
  row_tgt[idx[i]] = t;
  if (i == 0 || tkey[i - 1] != tkey[i]) {
    seg_begin[t] = (int)i;
    tgt_ptr[t] = (int)i;
    tgt_match[t] = -1;
  }
  if (i == E - 1 || tkey[i + 1] != tkey[i]) seg_end[t] = (int)(i + 1);
}
// every unmatched detection: its first row whose target is unmatched (det_best = that target, -1 when none is left); every
// unmatched target: its first edge whose detection is unmatched (tgt_best = that detection, -1 when none)
static __global__ void assoc_propose_kernel(int q, int K, long long E, const int* __restrict__ tix_last, const int* __restrict__ row_tgt,
                                            const unsigned* __restrict__ idx, const int* __restrict__ seg_end, const int* __restrict__ det_match,
                                            const int* __restrict__ tgt_match, int* __restrict__ det_ptr, int* __restrict__ det_best,
                                            int* __restrict__ tgt_ptr, int* __restrict__ tgt_best) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < q && det_match[i] < 0) {
    int r = det_ptr[i], t = -1;
    for (; r < K; ++r) {
      const int u = row_tgt[i * K + r];
      if (u < 0) { r = K; break; }
      if (tgt_match[u] < 0) { t = u; break; }
    }
    det_ptr[i] = r;
    det_best[i] = t;
  }
  if (E > 0 && i < *tix_last && tgt_match[i] < 0) {
    int e = tgt_ptr[i], jb = -1;
    const int end = seg_end[i];
    for (; e < end; ++e) {
      const int jj = (int)(idx[e] / (unsigned)K);
      if (det_match[jj] < 0) { jb = jj; break; }
    }
    tgt_ptr[i] = e;
    tgt_best[i] = jb;
  }
}
static __global__ void assoc_match_kernel(int q, const int* __restrict__ det_ptr, const int* __restrict__ det_best,
                                          const int* __restrict__ tgt_best, int* __restrict__ det_match, int* __restrict__ tgt_match,
                                          unsigned long long* __restrict__ matched) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  bool m = false;
  if (j < q && det_match[j] < 0) {
    const int t = det_best[j];
    if (t >= 0 && tgt_best[t] == j) {
      det_match[j] = det_ptr[j];
      tgt_match[t] = j;
      m = true;
    }
  }
  const unsigned b = __ballot_sync(0xffffffffu, m);
  if ((threadIdx.x & 31) == 0 && b) atomicAdd(matched, (unsigned long long)__popc(b));
}
// detection j's assigned row: target key (mapped through map when given: slot -> id) and d^2, else 0xFFFFFFFF / -1; action byte
// of the update (UPDATE for an assigned detection) when act is given
static __global__ void assoc_out_kernel(int q, int K, const int* __restrict__ det_match, const unsigned* __restrict__ tgt, const double* __restrict__ d2,
                                        const uint32_t* __restrict__ map, uint32_t* __restrict__ id_out, double* __restrict__ d2_out,
                                        uint8_t* __restrict__ act) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= q) return;
  const int r = det_match[j];
  if (r >= 0) {
    const unsigned k = tgt[(size_t)j * K + r];
    id_out[j] = map ? map[k] : k;
    d2_out[j] = d2[(size_t)j * K + r];
  } else {
    id_out[j] = 0xFFFFFFFFu;
    d2_out[j] = -1.0;
  }
  if (act) act[j] = r >= 0 ? (uint8_t)ACT_UPDATE : (uint8_t)ACT_NONE;
}

// ---- update at t1 -----------------------------------------------------------------------------------------------------------
// op k (action UPDATE, or every op when act is NULL) on a known id: dt[k] = t1 - t of its slot, rounded once; bad counts the ops
// whose dt is not >= 0 (t > t1 or NaN)
template <int TYPE>
__global__ void assoc_dt_kernel(const double* __restrict__ tiles, const uint32_t* __restrict__ ids_sorted, int n_slots, long long n,
                                const uint32_t* __restrict__ ids, const uint8_t* __restrict__ act, double t1, double* __restrict__ dt,
                                int* __restrict__ bad) {
  using LY = Layout<TYPE>;
  const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= n) return;
  dt[k] = 0.0;
  if (act && act[k] == ACT_NONE) return;
  const int s = lower_bound_u32(ids_sorted, n_slots, ids[k]);
  if (s >= n_slots || ids_sorted[s] != ids[k]) return;
  const double d = __dsub_rn(t1, tiles[(size_t)(s / TILE) * LY::TILE_DOUBLES + LY::F_T * TILE + (s % TILE)]);
  dt[k] = d;
  if (!(d >= 0.0)) atomicAdd(bad, 1);
}

}  // namespace te
