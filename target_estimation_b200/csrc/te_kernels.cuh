// te_kernels.cuh -- sm_100a kernels of the device-resident target pool.
//   kf_step_kernel     : the hot path (one tick of predict [+ update] for every staged tile)
//   init/rebuild/...   : add / erase by stable stream compaction, read-back gathers
//   isolver_kernel     : batched IntersectionSolver
#pragma once
#include "te_device.cuh"
#include "te_quartic.h"
#include "te_av_sym.cuh"

namespace te {

// -------------------------------------------------------------------------------------
// kf_step_kernel: persistent, one CTA per SM, WARPS warps per CTA, each warp owns STAGES
// shared-memory stages.  A stage holds one pool tile (32 targets x NF fields, contiguous
// in HBM) plus the tile's 32 x meas_stride measurement block, both fetched with one-
// dimensional TMA bulk copies (cp.async.bulk, completion on an mbarrier) and written back
// with a bulk store, so the state streams HBM -> smem -> registers -> smem -> HBM exactly
// once per tick without occupying registers while in flight.
// Algorithmic traffic per target-step: SURVEY.md 8(d) (UA: 1496 B).
// -------------------------------------------------------------------------------------
struct StepArgs {
  double* tiles;            // [n_tiles][NF][32]
  int n_slots;
  int n_tiles;               // tiles to process in dense mode: [tile_begin, tile_begin + n_tiles)
  int tile_begin;
  double* pos_out;           // optional [n_slots][3]: estimated position after the tick (publish record)
  const int* tile_list;     // sparse mode: tiles to process (device), else nullptr
  const int* d_nwork;       // sparse mode: number of entries in tile_list (device)
  double dt;
  const double* dt_slot;    // per-slot dt (sparse mode) or nullptr
  const double* meas;       // [n_slots][meas_stride] slot-order AoS, or nullptr
  int meas_stride;
  int meas_tma;             // 1: full tiles fetch their measurement block by TMA
  uint8_t* action;          // [n_slots] TE_ACT_* or nullptr
  int default_action;
  int clear_action;         // sparse mode: reset action[] and tile flags after use
  uint8_t* tile_flag;       // sparse mode tile flags (cleared with the actions)
  const uint16_t* cls;      // [n_slots] model class
  const double* Qtab;       // [n_classes][N*N] row-major
  const double* Rtab;       // [n_classes][M*M]
  // Q / R of one class (normally the pool's only one) travel in the kernel-parameter constant bank: a tile whose
  // lanes all use that class reads them as c[0][..] operands / LDC instead of 50+ global loads per target through an
  // L1 that the staged tiles leave almost no room for (AV with two CTAs per SM: < 4 KB)
  // multi-tick ("replay") launches: tick k reads meas + k * meas_tick_stride and action + k * action_tick_stride; a tile
  // stays on chip for all n_ticks ticks (temporal blocking: targets are independent)
  int n_ticks;
  long long meas_tick_stride;     // doubles
  long long action_tick_stride;   // bytes
  // compacting tick (te_pool_step_dense_expire): the tile is read from `tiles` as usual, but every surviving target's
  // column goes to slot dst_pos[slot] of `dst_tiles` (the pool's other buffer) instead of back in place, so the stable
  // compaction after an expiry costs no pass of its own.  nullptr = in place.
  double* dst_tiles;
  const int* dst_alive;     // [n_slots] 1 = survives
  const int* dst_pos;       // [n_slots] exclusive scan of dst_alive
  // live launch (te_pool_live_*): a replay launch whose ticks are released one by one.  tick_gate[0] = number of ticks released so
  // far, tick_gate[1] != 0 = stop (unreleased ticks are skipped); tick_done[k] counts the warps that have applied tick k;
  // pos_tick_stride > 0: the positions after tick k go to pos_out + k * pos_tick_stride
  const int* tick_gate;        // device words written by the copy engine (te_pool_live_push): [0] released ticks, [1] stop
  const int* tick_gate_host;   // page-locked, device-mapped words written by the host (te_pool_live_release / _end): [0] released, [1] stop
  int* tick_gate_eff;          // device words every warp watches: [0] = max of the two sources, [1] stop; kept by the warp of tile 0
  int* tick_done;
  int* tick_done_host;         // page-locked, device-mapped: the warp that completes tick k stores k + 1 here
  int tick_warps;              // warps that count themselves done per tick (= tiles of the pool)
  long long pos_tick_stride;   // doubles
  int packed;               // direct symmetric kernels: write the upper triangle of P only (pool flag lower_stale)
  int cls_c;                // class held in Qc / Rc, -1 = none
  double Rc[36];
  double Qc[324];
  const double* Ttab;       // [n_classes][M*M] row-major lower triangular: T = L^-1, R = L L^T (te_av_sym.cuh av_update_seq)
  double Tc[36];            // the same for class cls_c
};

constexpr int MEAS_DOUBLES = 7 * TILE;   // measurement block of a stage (max stride 7)

template <int TYPE> __host__ __device__ constexpr int stage_doubles() { return Layout<TYPE>::TILE_DOUBLES + MEAS_DOUBLES; }
template <int TYPE> __host__ __device__ constexpr size_t step_smem_bytes(int warps, int stages) {
  return 1024 + (size_t)warps * stages * stage_doubles<TYPE>() * 8;
}

// IMPL = 1 (AV only): step_lane_av_sym, the register-resident symmetric-covariance step of te_av_sym.cuh
template <int TYPE, int WARPS, int STAGES, bool MULTI = false, int IMPL = 0>
__global__ void __launch_bounds__(WARPS * 32, 1) kf_step_kernel(const StepArgs a) {
  using MT = Model<TYPE>;
  using LY = Layout<TYPE>;
  constexpr int STAGE_DOUBLES = stage_doubles<TYPE>();
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);
  double* stage0 = reinterpret_cast<double*>(smem_raw + 1024);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint64_t* mybar = bars + warp * STAGES;
  double* mystage = stage0 + (size_t)warp * STAGES * STAGE_DOUBLES;

  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < STAGES; ++s) mbar_init(&mybar[s], 1);
    fence_mbar_init();
  }
  __syncwarp();

  const int n_work = a.d_nwork ? *a.d_nwork : a.n_tiles;
  const int gw = blockIdx.x * WARPS + warp, GW = gridDim.x * WARPS;
  const int n_my = (n_work > gw) ? (n_work - gw + GW - 1) / GW : 0;

  auto tile_of = [&](int it) -> int {
    const int w = gw + it * GW;
    return a.tile_list ? a.tile_list[w] : a.tile_begin + w;
  };
  auto use_meas_tma = [&](int tile) -> bool { return a.meas_tma && (tile * TILE + TILE <= a.n_slots); };
  // lane 0: fetch tile `it` into its stage
  auto issue = [&](int it) {
    const int tile = tile_of(it);
    const int s = it % STAGES;
    double* st = mystage + (size_t)s * STAGE_DOUBLES;
    const bool mt = use_meas_tma(tile);
    const uint32_t mbytes = mt ? (uint32_t)a.meas_stride * TILE * 8u : 0u;
    mbar_expect_tx(&mybar[s], (uint32_t)LY::TILE_BYTES + mbytes);
    bulk_g2s(st, a.tiles + (size_t)tile * LY::TILE_DOUBLES, LY::TILE_BYTES, &mybar[s]);
    if (mt) bulk_g2s(st + LY::TILE_DOUBLES, a.meas + (size_t)tile * TILE * a.meas_stride, mbytes, &mybar[s]);
  };

  if (lane == 0) {
    for (int pre = 0; pre < STAGES - 1 && pre < n_my; ++pre) issue(pre);
  }

  for (int it = 0; it < n_my; ++it) {
    const int s = it % STAGES;
    const uint32_t parity = (uint32_t)(it / STAGES) & 1u;
    const int tile = tile_of(it);
    const int slot = tile * TILE + lane;
    const bool valid = slot < a.n_slots;

    // per-lane control words: issued before waiting on the tile so their latency overlaps
    int act = ACT_NONE;
    double dt = a.dt;
    int cls = 0;
    int dst = -1;   // compacting tick: destination slot, -1 = erased
    if (valid) {
      act = a.action ? (int)a.action[slot] : a.default_action;
      if (a.dt_slot) dt = a.dt_slot[slot];
      cls = (int)a.cls[slot];
      if (a.dst_tiles && a.dst_alive[slot]) dst = a.dst_pos[slot];
    }
    if (a.dst_tiles && dst < 0) act = ACT_NONE;   // erased at the end of this tick: its step is unobservable
    const bool mt = use_meas_tma(tile);
    double meas[7];
    if (!mt && act == ACT_UPDATE) {
      const double* mp = a.meas + (size_t)slot * a.meas_stride;
#pragma unroll
      for (int k = 0; k < 3; ++k) meas[k] = __ldg(mp + k);
      if (MT::M == 6) {
#pragma unroll
        for (int k = 3; k < 7; ++k) meas[k] = __ldg(mp + k);
      }
    }

    // refill the stage freed by the previous iteration's store (its smem must have been read)
    if (lane == 0 && it + STAGES - 1 < n_my) {
      bulk_wait_read<0>();
      issue(it + STAGES - 1);
    }

    double* st = mystage + (size_t)s * STAGE_DOUBLES;
    mbar_wait(&mybar[s], parity);

    if (MULTI) {
      // replay: all n_ticks ticks of this tile while it is staged; the next tick's control word and measurement are
      // fetched while the current one is computed (they are the only global traffic per tick: <= 57 B per target)
      unsigned any_tile = 0u;
      int act_t = act;
      double meas_t[7];
#pragma unroll
      for (int k = 0; k < 7; ++k) meas_t[k] = meas[k];
      const double* __restrict__ Qc = a.Qtab + (size_t)cls * MT::N * MT::N;
      const double* __restrict__ Rc = a.Rtab + (size_t)cls * MT::M * MT::M;
      // register-resident models (UV / UA): state and covariance stay in registers across the ticks
      constexpr int NR = MT::REGS ? MT::N : 1;
      RegP<NR> Preg;
      double xreg[NR];
      double t_reg = 0.0;
      long long nm_reg = 0;
      if (MT::REGS) {
#pragma unroll
        for (int i = 0; i < NR; ++i) xreg[i] = st[(LY::F_X + i) * TILE + lane];
#pragma unroll
        for (int k = 0; k < NR * NR; ++k) Preg.v[k] = st[(LY::F_P + k) * TILE + lane];
        t_reg = st[LY::F_T * TILE + lane];
        nm_reg = reinterpret_cast<const long long*>(st)[LY::F_NMEAS * TILE + lane];
      }
      for (int tick = 0; tick < a.n_ticks; ++tick) {
        int act_nx = ACT_NONE;
        double meas_nx[7];
#pragma unroll
        for (int k = 0; k < 7; ++k) meas_nx[k] = 0.0;
        if (tick + 1 < a.n_ticks && valid) {
          act_nx = a.action ? (int)a.action[(size_t)(tick + 1) * a.action_tick_stride + slot] : a.default_action;
          if (a.meas) {
            const double* mp = a.meas + (size_t)(tick + 1) * a.meas_tick_stride + (size_t)slot * a.meas_stride;
#pragma unroll
            for (int k = 0; k < 3; ++k) meas_nx[k] = __ldg(mp + k);
            if (MT::M == 6) {
#pragma unroll
              for (int k = 3; k < 7; ++k) meas_nx[k] = __ldg(mp + k);
            }
          }
        }
        any_tile |= __ballot_sync(0xffffffffu, act_t != ACT_NONE);
        if (act_t != ACT_NONE) {
          if constexpr (MT::REGS) {   // same calls, in the same order, as step_lane()
            predict_kinematic<NR, MT::B, MT::NB>(Preg, xreg, dt, Qc);
            if (act_t == ACT_UPDATE) {
              kf_update<NR, MT::M>(Preg, xreg, meas_t, Rc);
              nm_reg += 1;
            }
            t_reg = t_reg + dt;
          } else {
            step_lane<TYPE>(st, lane, act_t, dt, meas_t, Qc, Rc);
          }
        }
        act_t = act_nx;
#pragma unroll
        for (int k = 0; k < 7; ++k) meas_t[k] = meas_nx[k];
      }
      if (MT::REGS) {
#pragma unroll
        for (int i = 0; i < NR; ++i) st[(LY::F_X + i) * TILE + lane] = xreg[i];
#pragma unroll
        for (int k = 0; k < NR * NR; ++k) st[(LY::F_P + k) * TILE + lane] = Preg.v[k];
        st[LY::F_T * TILE + lane] = t_reg;
        reinterpret_cast<long long*>(st)[LY::F_NMEAS * TILE + lane] = nm_reg;
      }
      if (a.pos_out && valid) {
#pragma unroll
        for (int k = 0; k < 3; ++k) a.pos_out[(size_t)slot * 3 + k] = st[(LY::F_X + k) * TILE + lane];
      }
      if (any_tile) {
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          bulk_s2g(a.tiles + (size_t)tile * LY::TILE_DOUBLES, st, LY::TILE_BYTES);
          bulk_commit();
        }
      } else {
        __syncwarp();
      }
      continue;
    }

    const unsigned any = __ballot_sync(0xffffffffu, act != ACT_NONE);
    if (any) {
      if (mt && act == ACT_UPDATE) {
        const double* mp = st + LY::TILE_DOUBLES + lane * a.meas_stride;
#pragma unroll
        for (int k = 0; k < 3; ++k) meas[k] = mp[k];
        if (MT::M == 6) {
#pragma unroll
          for (int k = 3; k < 7; ++k) meas[k] = mp[k];
        }
      }
      if (act != ACT_NONE) {
        if constexpr (IMPL == 1) step_lane_av_sym<LY::F_PREV, false>(st + lane, st + lane, st + lane, act, dt, meas, a.Qtab + (size_t)cls * MT::N * MT::N, a.Rtab + (size_t)cls * MT::M * MT::M);
        else step_lane<TYPE>(st, lane, act, dt, meas, a.Qtab + (size_t)cls * MT::N * MT::N, a.Rtab + (size_t)cls * MT::M * MT::M);
        if (a.clear_action) a.action[slot] = 0;
      }
    }
    if (a.pos_out && valid) {
#pragma unroll
      for (int k = 0; k < 3; ++k) a.pos_out[(size_t)slot * 3 + k] = st[(LY::F_X + k) * TILE + lane];
    }
    if (a.dst_tiles) {
      // compacting tick: every lane moves its own column (the only one it wrote) to its destination slot; consecutive
      // survivors are consecutive there, so each field is one or two coalesced segments per warp
      if (dst >= 0) {
        double* dr = a.dst_tiles + (size_t)(dst / TILE) * LY::TILE_DOUBLES + (dst % TILE);
#pragma unroll 8
        for (int f = 0; f < LY::NF; ++f) __stcs(dr + (size_t)f * TILE, st[f * TILE + lane]);
      }
      __syncwarp();   // all columns read before lane 0 refills this stage in the next iteration
    } else if (any) {
      fence_proxy_async();   // generic-proxy writes of the stage -> visible to the bulk store
      __syncwarp();
      if (lane == 0) {
        bulk_s2g(a.tiles + (size_t)tile * LY::TILE_DOUBLES, st, LY::TILE_BYTES);
        bulk_commit();
        if (a.clear_action) a.tile_flag[tile] = 0;
      }
    } else {
      __syncwarp();
    }
  }
  if (lane == 0) bulk_wait<0>();
}

// -------------------------------------------------------------------------------------
// pool maintenance kernels
// -------------------------------------------------------------------------------------
__device__ __forceinline__ int lower_bound_u32(const uint32_t* __restrict__ a, int n, uint32_t key) {
  int lo = 0, hi = n;
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (a[mid] < key) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// ids -> slots (-1 if absent)
static __global__ void lookup_slots_kernel(const uint32_t* __restrict__ ids_sorted, int n_slots, const uint32_t* __restrict__ q,
                                    long long n, int* __restrict__ slots) {
  long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= n) return;
  int s = lower_bound_u32(ids_sorted, n_slots, q[k]);
  slots[k] = (s < n_slots && ids_sorted[s] == q[k]) ? s : -1;
}

// initial state of one new target (constructors of src/types/*.cpp + KalmanFilterInterface::init,
// src/kalman.cpp:16-21): x0 from (p0,v0,a0), P = scale*P0[cls], t = t0, n_meas = 0, prev_rpy = 0 (H3).
struct AddData {
  const uint32_t* ids;
  const uint16_t* cls;
  const double* t0;
  const double* p0;      // [n][7]
  const double* v0;      // [n][6] or nullptr
  const double* a0;      // [n][6] or nullptr
  const double* scale;   // [n] or nullptr
};

struct ColdArrays {
  uint32_t* ids;
  uint16_t* cls;
  double* last_meas;   // last measurement stamp [s], 0 = never (Measurement::last_meas_time_)
  double* meas;        // [slot][7] last measurement (TargetInterface::measured_pose_)
};

template <int TYPE>
__device__ __forceinline__ void init_slot(double* tiles, const ColdArrays& cold, int slot, const AddData& ad, long long k,
                                          const double* __restrict__ P0tab) {
  using MT = Model<TYPE>;
  using LY = Layout<TYPE>;
  constexpr int N = MT::N;
  double* rec = tiles + (size_t)(slot / TILE) * LY::TILE_DOUBLES + (slot % TILE);
  const double* p0 = ad.p0 + 7 * k;
  double x[N];
#pragma unroll
  for (int i = 0; i < N; ++i) x[i] = 0.0;
  if (TYPE == UNIFORM_VELOCITY || TYPE == UNIFORM_ACCELERATION) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      x[i] = p0[i];
      x[3 + i] = ad.v0 ? ad.v0[6 * k + i] : 0.0;
      if (TYPE == UNIFORM_ACCELERATION) x[6 + i] = ad.a0 ? ad.a0[6 * k + i] : 0.0;
    }
  } else {
    // pose7dToPose6d (geometry.hpp:619-628)
    Quat q{p0[3], p0[4], p0[5], p0[6]};
    quat_normalize(q);
    double rpy[3];
    quat_to_rpy(q, rpy);
#pragma unroll
    for (int i = 0; i < 3; ++i) { x[i] = p0[i]; x[3 + i] = rpy[i]; }
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      x[6 + i] = ad.v0 ? ad.v0[6 * k + i] : 0.0;
      if (TYPE == ANGULAR_RATES) x[12 + i] = ad.a0 ? ad.a0[6 * k + i] : 0.0;
    }
  }
#pragma unroll
  for (int i = 0; i < N; ++i) rec[(LY::F_X + i) * TILE] = x[i];
  const int c = ad.cls ? (int)ad.cls[k] : 0;
  const double sc = ad.scale ? ad.scale[k] : 1.0;
  const double* P0 = P0tab + (size_t)c * N * N;
  for (int e = 0; e < N * N; ++e) rec[(LY::F_P + e) * TILE] = ad.scale ? sc * P0[e] : P0[e];
  rec[LY::F_T * TILE] = ad.t0 ? ad.t0[k] : 0.0;
  reinterpret_cast<long long*>(rec)[LY::F_NMEAS * TILE] = 0;
  for (int e = 0; e < MT::NPREV; ++e) rec[(LY::F_PREV + e) * TILE] = 0.0;
  cold.ids[slot] = ad.ids[k];
  cold.cls[slot] = (uint16_t)c;
  cold.last_meas[slot] = 0.0;
  // initPose(measured_pose_) (src/target_interface.cpp:25)
  for (int e = 0; e < 7; ++e) cold.meas[(size_t)slot * 7 + e] = (e == 6) ? 1.0 : 0.0;
}

// append path: new targets occupy slots [base, base+n)
template <int TYPE>
__global__ void init_append_kernel(double* tiles, ColdArrays cold, int base, AddData ad, long long n, const double* P0tab) {
  long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= n) return;
  init_slot<TYPE>(tiles, cold, base + (int)k, ad, k, P0tab);
}

// alive[s] = 1 for all, then 0 for listed slots
static __global__ void fill_i32_kernel(int* a, int n, int v) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) a[i] = v;
}
static __global__ void clear_listed_kernel(int* alive, const int* slots, long long n) {
  long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k < n && slots[k] >= 0) alive[slots[k]] = 0;
}

// merge ranks: surviving old slot s -> dest = pos[s] + #(new ids < id[s])
static __global__ void map_existing_kernel(int n_old, const int* __restrict__ alive, const int* __restrict__ pos,
                                    const uint32_t* __restrict__ old_ids, const uint32_t* __restrict__ add_ids, int n_add,
                                    int* __restrict__ srcmap) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_old || !alive[s]) return;
  int d = pos[s] + (n_add ? lower_bound_u32(add_ids, n_add, old_ids[s]) : 0);
  srcmap[d] = s;
}
// new id k -> dest = k + #(surviving old ids < new id)
static __global__ void map_new_kernel(int n_add, const uint32_t* __restrict__ add_ids, const uint32_t* __restrict__ old_ids, int n_old,
                               const int* __restrict__ pos, int total_alive, int* __restrict__ srcmap) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_add) return;
  int e = lower_bound_u32(old_ids, n_old, add_ids[k]);
  int before = (e < n_old) ? pos[e] : total_alive;
  srcmap[k + before] = -1 - k;
}

// stable gather of every field of every surviving target into the other buffer + init of new ones.  blockIdx.y selects a
// chunk of REBUILD_FPT fields, all of whose loads are issued before the first store (a single thread walking the 347
// fields of an AR slot one after the other keeps too few bytes in flight: 2.0 TB/s; chunked: see DESIGN.md section 7);
// chunk 0 also moves the cold arrays and initialises the new slots.
constexpr int REBUILD_FPT = 16;
template <int TYPE>
__global__ void rebuild_kernel(int n_new, const int* __restrict__ srcmap, const double* __restrict__ old_tiles, ColdArrays old_cold,
                               double* __restrict__ new_tiles, ColdArrays new_cold, AddData ad, const double* P0tab) {
  using LY = Layout<TYPE>;
  int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= n_new) return;
  int s = srcmap[d];
  const int f0 = blockIdx.y * REBUILD_FPT;
  if (s >= 0) {
    const double* src = old_tiles + (size_t)(s / TILE) * LY::TILE_DOUBLES + (s % TILE);
    double* dst = new_tiles + (size_t)(d / TILE) * LY::TILE_DOUBLES + (d % TILE);
    double v[REBUILD_FPT];
#pragma unroll
    for (int k = 0; k < REBUILD_FPT; ++k) if (f0 + k < LY::NF) v[k] = __ldcs(src + (size_t)(f0 + k) * TILE);
#pragma unroll
    for (int k = 0; k < REBUILD_FPT; ++k) if (f0 + k < LY::NF) __stcs(dst + (size_t)(f0 + k) * TILE, v[k]);
    if (blockIdx.y == 0) {
      new_cold.ids[d] = old_cold.ids[s];
      new_cold.cls[d] = old_cold.cls[s];
      new_cold.last_meas[d] = old_cold.last_meas[s];
#pragma unroll
      for (int e = 0; e < 7; ++e) new_cold.meas[(size_t)d * 7 + e] = old_cold.meas[(size_t)s * 7 + e];
    }
  } else if (blockIdx.y == 0) {
    init_slot<TYPE>(new_tiles, new_cold, d, ad, (long long)(-1 - s), P0tab);
  }
}

// sparse tick: op k -> per-slot action / dt / measurement; tiles touched for the first time are
// appended to tile_list (counters[0] = #tiles, counters[1] = #ops applied).  One op per id per call.
static __global__ void scatter_ops_kernel(const uint32_t* __restrict__ ids_sorted, int n_slots, long long n, const uint32_t* __restrict__ q,
                                   const double* __restrict__ dt, double dt_scalar, const double* __restrict__ meas,
                                   const uint8_t* __restrict__ action, uint8_t* act_slot, double* dt_slot, double* meas_slot,
                                   uint8_t* tile_flag, int* tile_list, int* counters, int* claim) {
  long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= n) return;
  int a = action ? (int)action[k] : ACT_UPDATE;
  if (a == ACT_NONE) return;
  int s = lower_bound_u32(ids_sorted, n_slots, q[k]);
  if (s >= n_slots || ids_sorted[s] != q[k]) return;
  // one op per slot and launch: a second op on the same slot (an id named twice) would race with the first one's record --
  // counted here, and the host then applies nothing and splits the batch (counters[2]; claim is zeroed per call)
  if (atomicAdd(&claim[s], 1) > 0) {
    atomicAdd(&counters[2], 1);
    return;
  }
  act_slot[s] = (uint8_t)a;
  dt_slot[s] = dt ? dt[k] : dt_scalar;
  if (a == ACT_UPDATE) {
#pragma unroll
    for (int e = 0; e < 7; ++e) meas_slot[(size_t)s * 7 + e] = meas[(size_t)k * 7 + e];
  }
  // byte flags packed four to a word: claim the tile with an atomicOr on its byte
  const int tile = s / TILE;
  unsigned* w = reinterpret_cast<unsigned*>(tile_flag) + (tile >> 2);
  const unsigned bit = 1u << ((tile & 3) * 8);
  const unsigned old = atomicOr(w, bit);
  if (!(old & bit)) tile_list[atomicAdd(&counters[0], 1)] = tile;
  atomicAdd(&counters[1], 1);
}

// measured_pose_ refresh of a masked dense host tick (src/target_interface.cpp:142-146)
static __global__ void copy_meas_masked_kernel(double* __restrict__ dst, const double* __restrict__ src, const uint8_t* __restrict__ action, int n) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n || action[s] != ACT_UPDATE) return;
#pragma unroll
  for (int e = 0; e < 7; ++e) dst[(size_t)s * 7 + e] = src[(size_t)s * 7 + e];
}
// initPose (utils.hpp:64-72): [0 0 0 | 0 0 0 1]
static __global__ void init_pose_kernel(double* pose, long long n) {
  long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= n) return;
  for (int e = 0; e < 7; ++e) pose[k * 7 + e] = (e == 6) ? 1.0 : 0.0;
}

// dense host-API tick: remember the applied measurement as measured_pose_ (stride 7 only)
static __global__ void fill_dt_kernel(double* dt_slot, int n, double v) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dt_slot[i] = v;
}

// read-back gathers -------------------------------------------------------------------
template <int TYPE>
__global__ void gather_state_kernel(const double* __restrict__ tiles, const ColdArrays cold, const int* __restrict__ slots, long long n,
                                    double* x, double* P, double* t, long long* n_meas, double* prev, double* mpose, int lower_stale) {
  using MT = Model<TYPE>;
  using LY = Layout<TYPE>;
  long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= n) return;
  int s = slots ? slots[k] : (int)k;
  if (s < 0) return;
  const double* rec = tiles + (size_t)(s / TILE) * LY::TILE_DOUBLES + (s % TILE);
  if (x) for (int i = 0; i < MT::N; ++i) x[k * MT::N + i] = rec[(LY::F_X + i) * TILE];
  if (P) {
    for (int i = 0; i < MT::N; ++i)
      for (int j = 0; j < MT::N; ++j) {
        // lower_stale: the packed symmetric kernels maintain the upper triangle only -- P(i, j) = P(j, i) for i > j
        const int e = (lower_stale && i > j) ? j * MT::N + i : i * MT::N + j;
        P[k * MT::N * MT::N + i * MT::N + j] = rec[(LY::F_P + e) * TILE];
      }
  }
  if (t) t[k] = rec[LY::F_T * TILE];
  if (n_meas) n_meas[k] = reinterpret_cast<const long long*>(rec)[LY::F_NMEAS * TILE];
  if (prev) for (int e = 0; e < 3; ++e) prev[k * 3 + e] = (MT::NPREV ? rec[(LY::F_PREV + (MT::NPREV ? e : 0)) * TILE] : 0.0);
  if (mpose) for (int e = 0; e < 7; ++e) mpose[k * 7 + e] = cold.meas[(size_t)s * 7 + e];
}

template <int TYPE>
__global__ void gather_estimates_kernel(const double* __restrict__ tiles, const int* __restrict__ slots, long long n,
                                        const double* __restrict__ t1, double* pose, double* twist, double* acc, double* pose6,
                                        uint8_t* found, int rec13) {
  using MT = Model<TYPE>;
  using LY = Layout<TYPE>;
  long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= n) return;
  int s = slots ? slots[k] : (int)k;
  if (found) found[k] = (s >= 0);
  if (s < 0) return;
  const double* rec = tiles + (size_t)(s / TILE) * LY::TILE_DOUBLES + (s % TILE);
  double x[MT::N];
#pragma unroll
  for (int i = 0; i < MT::N; ++i) x[i] = rec[(LY::F_X + i) * TILE];
  const double t = rec[LY::F_T * TILE];
  double po[7], tw[6], ac[6], p6[6];
  derive_outputs<TYPE>(x, t, t1 != nullptr, t1 ? t1[k] : 0.0, po, tw, ac, p6);
  if (rec13) {   // [n][13] = pose7 | twist6
    for (int e = 0; e < 7; ++e) pose[k * 13 + e] = po[e];
    for (int e = 0; e < 6; ++e) pose[k * 13 + 7 + e] = tw[e];
    return;
  }
  if (pose) for (int e = 0; e < 7; ++e) pose[k * 7 + e] = po[e];
  if (twist) for (int e = 0; e < 6; ++e) twist[k * 6 + e] = tw[e];
  if (acc) for (int e = 0; e < 6; ++e) acc[k * 6 + e] = ac[e];
  if (pose6) for (int e = 0; e < 6; ++e) pose6[k * 6 + e] = p6[e];
}

// expiry ---------------------------------------------------------------------------------
// toSec (utils.hpp:59-62) with explicit round-to-nearest mul/add: never contracted to FMA (H5)
__device__ __forceinline__ double to_sec_rn(uint32_t sec, uint32_t nsec) {
  return __dadd_rn(__uint2double_rn(sec), __dmul_rn(1e-9, __uint2double_rn(nsec)));
}
static __global__ void set_stamps_kernel(const uint32_t* __restrict__ ids_sorted, int n_slots, long long n, const uint32_t* __restrict__ q,
                                  const uint32_t* __restrict__ sec, const uint32_t* __restrict__ nsec, double* last_meas) {
  long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= n) return;
  int s = lower_bound_u32(ids_sorted, n_slots, q[k]);
  if (s >= n_slots || ids_sorted[s] != q[k]) return;
  last_meas[s] = to_sec_rn(sec[k], nsec[k]);
}
// dense tick: every slot updated this tick gets the tick's stamp as last_meas_time_
static __global__ void stamp_dense_kernel(const uint8_t* __restrict__ action, int default_action, int n_slots, double stamp, double* last_meas) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_slots) return;
  const int a = action ? (int)action[s] : default_action;
  if (a == ACT_UPDATE) last_meas[s] = stamp;
}
// alive[s] = !(last > 0.0 && (now - last) >= timeout)   (src/target_manager_ros.cpp:67)
static __global__ void expire_flags_kernel(const double* __restrict__ last_meas, int n_slots, double now, double timeout, int* alive) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_slots) return;
  const double last = last_meas[s];
  const bool expired = (last > 0.0) && (__dsub_rn(now, last) >= timeout);
  alive[s] = expired ? 0 : 1;
}
static __global__ void collect_erased_kernel(const int* __restrict__ alive, const int* __restrict__ pos, const uint32_t* __restrict__ ids,
                                      int n_slots, uint32_t* erased) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_slots || alive[s]) return;
  erased[s - pos[s]] = ids[s];
}

// device-resident mailboxes ---------------------------------------------------------------
// One Measurement (include/target_estimation/target_manager_ros.hpp:74-134) per slot: tr_'s stamp and pose, new_meas_ kept
// directly as the action byte of the next tick (ACT_UPDATE = readable, ACT_PREDICT = not), last_meas_time_ = cold.last_meas.
// pose [slot][7] and act [slot] ARE the dense step's measurement block and action array: the tick needs no staging pass.
struct MailArrays {
  uint32_t* sec;
  uint32_t* nsec;
  uint8_t* act;
  double* pose;
};
// mailboxes promoted to targets by a tick (index = AddData index; pose = AddData::p0, act = ACT_UPDATE); sec == nullptr:
// targets added outside the tick have NO mailbox (action ACT_NONE: the tick does not touch them, as the reference's loop over
// its mailboxes does not; the first record creates it)
struct MailAdd {
  const uint32_t* sec;
  const uint32_t* nsec;
  const double* last;
};

// record k of a /tf message -> sort key = its slot (unknown ids: key n_slots, listed for the host, which keeps the
// target-less mailboxes)
static __global__ void mb_lookup_kernel(const uint32_t* __restrict__ ids_sorted, int n_slots, const uint32_t* __restrict__ q, int n,
                                 uint32_t* __restrict__ key, int* __restrict__ rec, int* __restrict__ unknown, int* counter) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  int s = n_slots ? lower_bound_u32(ids_sorted, n_slots, q[k]) : 0;
  const bool hit = s < n_slots && ids_sorted[s] == q[k];
  key[k] = hit ? (uint32_t)s : (uint32_t)n_slots;
  rec[k] = k;
  if (!hit) unknown[atomicAdd(counter, 1)] = k;
}
// device-resident messages: the records of unknown ids, packed for the host (which keeps the target-less mailboxes)
static __global__ void mb_pack_unknown_kernel(int n_unknown, const int* __restrict__ list, const uint32_t* __restrict__ ids, const uint32_t* __restrict__ sec,
                                       const uint32_t* __restrict__ nsec, const double* __restrict__ poses, uint32_t* __restrict__ o_ids,
                                       uint32_t* __restrict__ o_sec, uint32_t* __restrict__ o_nsec, double* __restrict__ o_pose) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_unknown) return;
  const int r = list[k];
  o_ids[k] = ids[r];
  o_sec[k] = sec[r];
  o_nsec[k] = nsec[r];
#pragma unroll
  for (int e = 0; e < 7; ++e) o_pose[(size_t)k * 7 + e] = poses[(size_t)r * 7 + e];
}
// records sorted by (slot, arrival order): the first record of each slot's run applies the whole run in arrival order --
// Measurement::update (target_manager_ros.hpp:96-115): a stamp newer than the stored one makes the mailbox readable and
// becomes last_meas_time_, any other stamp makes it unreadable; stamp and pose are stored either way.
static __global__ void mb_apply_kernel(int n, int n_slots, const uint32_t* __restrict__ key, const int* __restrict__ rec, const uint32_t* __restrict__ sec,
                                const uint32_t* __restrict__ nsec, const double* __restrict__ poses, MailArrays mb, double* last_meas) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint32_t s = key[k];
  if (s >= (uint32_t)n_slots || (k > 0 && key[k - 1] == s)) return;
  uint32_t msec = mb.sec[s], mnsec = mb.nsec[s];
  uint8_t act = mb.act[s];
  double last = last_meas[s];
  int r = 0;
  for (int j = k; j < n && key[j] == s; ++j) {
    r = rec[j];
    const double cur = to_sec_rn(sec[r], nsec[r]);
    const double prev = to_sec_rn(msec, mnsec);
    if (cur > prev) { act = (uint8_t)ACT_UPDATE; last = cur; }
    else act = (uint8_t)ACT_PREDICT;
    msec = sec[r];
    mnsec = nsec[r];
  }
  mb.sec[s] = msec;
  mb.nsec[s] = mnsec;
  mb.act[s] = act;
  last_meas[s] = last;
#pragma unroll
  for (int e = 0; e < 7; ++e) mb.pose[(size_t)s * 7 + e] = poses[(size_t)r * 7 + e];
}
// mailboxes follow their slots through a compaction / merge (srcmap of rebuild_kernel); promoted ones are filled in
static __global__ void mb_move_kernel(int n_new, const int* __restrict__ srcmap, MailArrays o, MailArrays nw, MailAdd add, const double* __restrict__ add_p0,
                               double* __restrict__ new_last_meas) {
  int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= n_new) return;
  const int s = srcmap[d];
  if (s >= 0) {
    nw.sec[d] = o.sec[s];
    nw.nsec[d] = o.nsec[s];
    nw.act[d] = o.act[s];
#pragma unroll
    for (int e = 0; e < 7; ++e) nw.pose[(size_t)d * 7 + e] = o.pose[(size_t)s * 7 + e];
  } else {
    const int k = -1 - s;
    nw.sec[d] = add.sec ? add.sec[k] : 0u;
    nw.nsec[d] = add.sec ? add.nsec[k] : 0u;
    nw.act[d] = (uint8_t)(add.sec ? ACT_UPDATE : ACT_NONE);
    if (add.sec) new_last_meas[d] = add.last[k];
#pragma unroll
    for (int e = 0; e < 7; ++e) nw.pose[(size_t)d * 7 + e] = add_p0 ? add_p0[(size_t)k * 7 + e] : (e == 6 ? 1.0 : 0.0);
  }
}
// no mailbox yet for slots [base, base + n) (targets appended outside the tick)
static __global__ void mb_clear_kernel(MailArrays mb, int base, int n) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int d = base + k;
  mb.sec[d] = 0u;
  mb.nsec[d] = 0u;
  mb.act[d] = (uint8_t)ACT_NONE;
#pragma unroll
  for (int e = 0; e < 7; ++e) mb.pose[(size_t)d * 7 + e] = (e == 6 ? 1.0 : 0.0);
}
// ---- fused mailbox tick: the step kernel itself moves the survivors (StepArgs::dst_*), so the merge only needs the
// destination of every old slot and of every new id ----
// new id k -> its slot in the merged order (k + #surviving old ids below it); pos = exclusive scan of alive (unmodified)
static __global__ void merge_new_dst_kernel(int n_add, const uint32_t* __restrict__ add_ids, const uint32_t* __restrict__ old_ids, int n_old,
                                     const int* __restrict__ pos, int total_alive, int* __restrict__ new_dst) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_add) return;
  int e = lower_bound_u32(old_ids, n_old, add_ids[k]);
  new_dst[k] = k + ((e < n_old) ? pos[e] : total_alive);
}
// surviving old slot s -> pos[s] + #new ids below its id (in place; run after merge_new_dst_kernel / collect_erased_kernel)
static __global__ void merge_old_dst_kernel(int n_old, const int* __restrict__ alive, int* __restrict__ pos, const uint32_t* __restrict__ old_ids,
                                     const uint32_t* __restrict__ add_ids, int n_add) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_old || !alive[s]) return;
  pos[s] += lower_bound_u32(add_ids, n_add, old_ids[s]);
}
// mailboxes of the survivors -> their destination slots
static __global__ void mb_compact_kernel(int n_old, const int* __restrict__ alive, const int* __restrict__ pos, MailArrays o, MailArrays nw) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_old || !alive[s]) return;
  const int d = pos[s];
  nw.sec[d] = o.sec[s];
  nw.nsec[d] = o.nsec[s];
  nw.act[d] = o.act[s];
#pragma unroll
  for (int e = 0; e < 7; ++e) nw.pose[(size_t)d * 7 + e] = o.pose[(size_t)s * 7 + e];
}
// promoted mailboxes: init the target in its merged slot (TargetManager::init, v0 = a0 = 0), fill its mailbox, and put it on
// the sparse work list of the follow-up launch that applies its first update (src/target_manager_ros.cpp:54-59)
template <int TYPE>
__global__ void init_promoted_kernel(int n_add, const int* __restrict__ new_dst, double* tiles, ColdArrays cold, AddData ad, MailAdd add, MailArrays mb,
                                     const double* P0tab, uint8_t* act_slot, uint8_t* tile_flag, int* tile_list, int* counters) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_add) return;
  const int d = new_dst[k];
  init_slot<TYPE>(tiles, cold, d, ad, (long long)k, P0tab);
  cold.last_meas[d] = add.last[k];
  mb.sec[d] = add.sec[k];
  mb.nsec[d] = add.nsec[k];
  mb.act[d] = (uint8_t)ACT_UPDATE;
#pragma unroll
  for (int e = 0; e < 7; ++e) {
    const double v = ad.p0[(size_t)k * 7 + e];
    mb.pose[(size_t)d * 7 + e] = v;
    cold.meas[(size_t)d * 7 + e] = v;   // measured_pose_ after the first update
  }
  act_slot[d] = (uint8_t)ACT_UPDATE;
  const int tile = d / TILE;
  unsigned* w = reinterpret_cast<unsigned*>(tile_flag) + (tile >> 2);
  const unsigned bit = 1u << ((tile & 3) * 8);
  const unsigned old = atomicOr(w, bit);
  if (!(old & bit)) tile_list[atomicAdd(&counters[0], 1)] = tile;
}
// number of slots that have a mailbox (action != ACT_NONE)
static __global__ void mb_count_kernel(const uint8_t* __restrict__ act, int n, int* counter) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned m = __ballot_sync(0xFFFFFFFFu, s < n && act[s] != (uint8_t)ACT_NONE);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd(counter, __popc(m));
}
// mailboxes of listed slots -> packed records (sec, nsec, act, last, pose) for the host (a target erased by hand keeps its
// mailbox in the reference: it moves to the host's target-less map)
static __global__ void mb_gather_kernel(int n, const int* __restrict__ slots, MailArrays mb, const double* __restrict__ last_meas, uint32_t* __restrict__ sec,
                                 uint32_t* __restrict__ nsec, uint8_t* __restrict__ act, double* __restrict__ last, double* __restrict__ pose) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int s = slots[k];
  if (s < 0) { act[k] = 0xFF; return; }
  sec[k] = mb.sec[s];
  nsec[k] = mb.nsec[s];
  act[k] = mb.act[s];
  last[k] = last_meas[s];
#pragma unroll
  for (int e = 0; e < 7; ++e) pose[(size_t)k * 7 + e] = mb.pose[(size_t)s * 7 + e];
}
// the reverse: host mailboxes attached to the slots of targets that were just created by hand
static __global__ void mb_scatter_kernel(int n, const int* __restrict__ slots, const uint32_t* __restrict__ sec, const uint32_t* __restrict__ nsec,
                                  const uint8_t* __restrict__ act, const double* __restrict__ last, const double* __restrict__ pose, MailArrays mb,
                                  double* __restrict__ last_meas) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int s = slots[k];
  if (s < 0) return;
  mb.sec[s] = sec[k];
  mb.nsec[s] = nsec[k];
  mb.act[s] = act[k];
  last_meas[s] = last[k];
#pragma unroll
  for (int e = 0; e < 7; ++e) mb.pose[(size_t)s * 7 + e] = pose[(size_t)k * 7 + e];
}

// lower triangle <- upper triangle (before a full-matrix kernel runs on a pool whose last steps were packed)
template <int TYPE>
__global__ void mirror_lower_kernel(double* __restrict__ tiles, int n_slots) {
  using MT = Model<TYPE>;
  using LY = Layout<TYPE>;
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_slots) return;
  double* rec = tiles + (size_t)(s / TILE) * LY::TILE_DOUBLES + (s % TILE);
  for (int i = 1; i < MT::N; ++i)
    for (int j = 0; j < i; ++j) rec[(LY::F_P + i * MT::N + j) * TILE] = rec[(LY::F_P + j * MT::N + i) * TILE];
}

// compacting tick: the cold arrays of the survivors move to their destination slots (the tile fields are moved by the step
// kernel itself)
static __global__ void compact_cold_kernel(int n_old, const int* __restrict__ alive, const int* __restrict__ pos, ColdArrays old_cold, ColdArrays new_cold) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_old || !alive[s]) return;
  const int d = pos[s];
  new_cold.ids[d] = old_cold.ids[s];
  new_cold.cls[d] = old_cold.cls[s];
  new_cold.last_meas[d] = old_cold.last_meas[s];
#pragma unroll
  for (int e = 0; e < 7; ++e) new_cold.meas[(size_t)d * 7 + e] = old_cold.meas[(size_t)s * 7 + e];
}

// -------------------------------------------------------------------------------------
// Batched IntersectionSolver (src/intersection_solver.cpp:42-124).
// Roots of the quartic: te_quartic.h (Ferrari split + Newton polish in real FP64, Aberth-Ehrlich fallback; the
// reference uses Eigen's companion-matrix QR; all are backward stable -- they differ only for near-multiple roots,
// SURVEY.md H9), then the reference's selection rule: smallest real part among roots with |imag| < 1e-10, -1 if none /
// leading coefficient 0 / negative.
// -------------------------------------------------------------------------------------
struct IsolverState {
  long long n_streams;
  unsigned L;            // filters_length
  double* prev_pose;     // [n_streams][7]
  double* pos_win;       // [L][n_streams]
  double* ang_win;       // [L][n_streams]
  double* pos_sum;       // [n_streams]
  double* ang_sum;
  unsigned* idx;         // [n_streams] window_idx_
  uint8_t* complete;     // [n_streams] filter_complete_
  double pos_th_all, ang_th_all;   // thresholds of the dense form (per-query arrays absent)
};

// MovingAvgFilter::update (utils.hpp:222-251) without the variance by-product (never read by
// IntersectionSolver).  Returns the filtered value.
__device__ __forceinline__ double mavg_update(double* win, double* sum, unsigned idx, unsigned L, bool complete_after,
                                              long long stream, long long n_streams, double value) {
  double s = *sum;
  double* w = win + (size_t)idx * n_streams + stream;
  s -= *w;
  s += value;
  *w = value;
  *sum = s;
  unsigned num = complete_after ? L : idx + 1;
  return s / num;
}

template <int TYPE>
__global__ void isolver_kernel(const double* __restrict__ tiles, const int* __restrict__ slots, const int* __restrict__ stream, long long n,
                               const double* __restrict__ t1, const double* __restrict__ origin, const double* __restrict__ radius,
                               const double* __restrict__ pos_th, const double* __restrict__ ang_th, IsolverState st, double* delta_out,
                               double* pose_out, uint8_t* conv_out) {
  using MT = Model<TYPE>;
  using LY = Layout<TYPE>;
  long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int s = slots ? slots[k] : (int)k;   // dense form: query k = slot k
  double delta = -1.0;
  double pose[7] = {0, 0, 0, 0, 0, 0, 1};   // initPose(intersection_pose) (:99)
  bool converged = false;
  if (s >= 0) {   // target exists (:44)
    const double* rec = tiles + (size_t)(s / TILE) * LY::TILE_DOUBLES + (s % TILE);
    double x[MT::N];
#pragma unroll
    for (int i = 0; i < MT::N; ++i) x[i] = rec[(LY::F_X + i) * TILE];
    const double t = rec[LY::F_T * TILE];
    const double tq = t1 ? t1[k] : t;           // dense form without t1: the target's own time
    double po[7], tw[6], ac[6];
    derive_outputs<TYPE>(x, t, true, tq, po, tw, ac, nullptr);
    const double px = po[0] - origin[3 * k + 0], py = po[1] - origin[3 * k + 1], pz = po[2] - origin[3 * k + 2];
    const double vx = tw[0], vy = tw[1], vz = tw[2];
    const double ax = ac[0], ay = ac[1], az = ac[2];
    const double Rr = radius[k];
    double c[5];   // :66-70
    c[4] = 0.25 * (ax * ax + ay * ay + az * az);
    c[3] = vx * ax + vy * ay + vz * az;
    c[2] = vx * vx + vy * vy + vz * vz + px * ax + py * ay + pz * az;
    c[1] = 2 * (px * vx + py * vy + pz * vz);
    c[0] = px * px + py * py + pz * pz - Rr * Rr;
    delta = lowest_real_root4(c);
    if (delta < 0) delta = -1.0;
    if (pose_out && delta > -1.0) {   // :102-121
      derive_outputs<TYPE>(x, t, true, delta + tq, pose, nullptr, nullptr, nullptr);
      const long long sidx = stream ? stream[k] : k;
      double* prev = st.prev_pose + sidx * 7;
      const double dx = pose[0] - prev[0], dy = pose[1] - prev[1], dz = pose[2] - prev[2];
      const double pos_error = sqrt(dx * dx + dy * dy + dz * dz);
      Quat q1{pose[3], pose[4], pose[5], pose[6]}, q2{prev[3], prev[4], prev[5], prev[6]};
      quat_normalize(q1);
      quat_normalize(q2);
      // computeQuaternionErrorAngle (geometry.hpp:630-657): q1 * q2^-1, normalise, 2 acos(w)
      const double n2 = q2.x * q2.x + q2.y * q2.y + q2.z * q2.z + q2.w * q2.w;
      Quat qi{-q2.x / n2, -q2.y / n2, -q2.z / n2, q2.w / n2};
      Quat qe = quat_mul(q1, qi);
      quat_normalize(qe);
      const double ang_error = fabs(wrap_min_max(2 * acos(qe.w), -TE_PI, TE_PI));
      const unsigned idx = st.idx[sidx];
      bool complete = st.complete[sidx] != 0;
      if (!complete && idx == st.L - 1) complete = true;
      const double pf = mavg_update(st.pos_win, st.pos_sum + sidx, idx, st.L, complete, sidx, st.n_streams, pos_error);
      const double af = mavg_update(st.ang_win, st.ang_sum + sidx, idx, st.L, complete, sidx, st.n_streams, ang_error);
      st.idx[sidx] = (idx + 1) % st.L;
      st.complete[sidx] = complete ? 1 : 0;
#pragma unroll
      for (int e = 0; e < 7; ++e) prev[e] = pose[e];
      if (pf <= (pos_th ? pos_th[k] : st.pos_th_all) && af <= (ang_th ? ang_th[k] : st.ang_th_all)) converged = true;
    }
  }
  if (delta_out) delta_out[k] = delta;
  if (pose_out) {
#pragma unroll
    for (int e = 0; e < 7; ++e) pose_out[k * 7 + e] = pose[e];
  }
  if (conv_out) conv_out[k] = converged ? 1 : 0;
}

// queries whose id exists (slot >= 0), added to *count
static __global__ void isolver_count_found_kernel(const int* __restrict__ slots, long long n, unsigned long long* count) {
  const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const unsigned found = __ballot_sync(0xffffffffu, k < n && slots[k] >= 0);
  if ((threadIdx.x & 31) == 0 && found) atomicAdd(count, (unsigned long long)__popc(found));
}

// The complete state of n solver streams as one block of ISOLVER_ROWS(L) rows of n doubles, row-major, column j = streams[j]:
// prev_pose (7 rows) | pos_win (L) | ang_win (L) | pos_sum | ang_sum | idx | complete.  idx and complete are small integers,
// exact in a double, so pack + unpack moves every byte of the state unchanged.  Thread i handles row i / n, column i % n: the block
// is written (pack) and read (unpack) coalesced; the window rows are [L][n_streams] on both sides, so consecutive listed streams
// are coalesced there too.
__host__ __device__ inline long long isolver_rows(unsigned L) { return 2 * (long long)L + 11; }

static __global__ void isolver_pack_streams_kernel(IsolverState st, const int* __restrict__ streams, long long n, double* __restrict__ block) {
  const long long L = st.L, total = isolver_rows(st.L) * n;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / n, s = streams[i - row * n];
    double v;
    if (row < 7) v = st.prev_pose[s * 7 + row];
    else if (row < 7 + L) v = st.pos_win[(row - 7) * st.n_streams + s];
    else if (row < 7 + 2 * L) v = st.ang_win[(row - 7 - L) * st.n_streams + s];
    else if (row == 7 + 2 * L) v = st.pos_sum[s];
    else if (row == 8 + 2 * L) v = st.ang_sum[s];
    else if (row == 9 + 2 * L) v = (double)st.idx[s];
    else v = (double)st.complete[s];
    block[i] = v;
  }
}

static __global__ void isolver_unpack_streams_kernel(IsolverState st, const int* __restrict__ streams, long long n, const double* __restrict__ block) {
  const long long L = st.L, total = isolver_rows(st.L) * n;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / n, s = streams[i - row * n];
    const double v = block[i];
    if (row < 7) st.prev_pose[s * 7 + row] = v;
    else if (row < 7 + L) st.pos_win[(row - 7) * st.n_streams + s] = v;
    else if (row < 7 + 2 * L) st.ang_win[(row - 7 - L) * st.n_streams + s] = v;
    else if (row == 7 + 2 * L) st.pos_sum[s] = v;
    else if (row == 8 + 2 * L) st.ang_sum[s] = v;
    else if (row == 9 + 2 * L) st.idx[s] = (unsigned)v;
    else st.complete[s] = (uint8_t)v;
  }
}

}  // namespace te
