// te_direct.cuh -- direct (register-streaming) step kernel of the angular-velocities model.
//
// kf_step_kernel stages whole tiles in shared memory by TMA so that data in flight occupies no registers; that pays when
// a thread's working set is the whole tile (UV / UA).  The symmetric AV step (te_av_sym.cuh) needs only 95 of the tile's 161
// fields as INPUT -- state, upper triangle of the covariance, t, n_meas, previous unwrapped angles -- and keeps them in
// registers from the first instruction to the last, so staging buys nothing and costs 43 KB of shared memory per tile in
// flight (five warps per SM).  Here every lane loads its column of those 95 fields straight from HBM (field-major tiles:
// each field is one coalesced 256 B segment per warp; the lower triangle is never read: 1.26x less read traffic), steps,
// and stores all 161 fields straight back.  Shared memory holds only a 22 KB scratch per warp (Z, x', y), so eight warps
// -- every register of the SM at 255 per thread -- hide each other's load latency and dependent FP64 chains.
// Same arguments and semantics as kf_step_kernel (dense / sparse tile lists, per-slot dt, actions, pos_out, compacting
// destination); replay (n_ticks > 1) stays on the staged kernel.
#pragma once
#include "te_kernels.cuh"
#include "te_kin_sym.cuh"

namespace te {

constexpr int AV_SCRATCH_FIELDS = 12 + 72 + 3;   // x' | Z (6 x 12) | y[3..5]
constexpr int AV_SCRATCH_PREV = 12 + 72;
__host__ __device__ constexpr size_t av_direct_smem_bytes(int warps) { return (size_t)warps * AV_SCRATCH_FIELDS * TILE * 8; }

template <int WARPS, int ZF = 2>
__global__ void __launch_bounds__(WARPS * 32, 1) kf_step_av_direct_kernel(const StepArgs a) {
  using LY = Layout<ANGULAR_VELOCITIES>;
  constexpr int N = 12, M = 6;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* sc = reinterpret_cast<double*>(smem_raw) + (size_t)warp * AV_SCRATCH_FIELDS * TILE + lane;
  const int n_work = a.d_nwork ? *a.d_nwork : a.n_tiles;
  const int gw = blockIdx.x * WARPS + warp, GW = gridDim.x * WARPS;
  for (int w = gw; w < n_work; w += GW) {
    const int tile = a.tile_list ? a.tile_list[w] : a.tile_begin + w;
    const int slot = tile * TILE + lane;
    const bool valid = slot < a.n_slots;
    int act = ACT_NONE, cls = 0, dst = -1;
    double dt = a.dt;
    if (valid) {
      act = a.action ? (int)a.action[slot] : a.default_action;
      if (a.dt_slot) dt = a.dt_slot[slot];
      cls = (int)a.cls[slot];
      if (a.dst_tiles) {
        if (a.dst_alive[slot]) dst = a.dst_pos[slot];
        else act = ACT_NONE;   // erased at the end of this tick: its step is unobservable
      }
    }
    // (an L2 prefetch of the warp's next tile -- cp.async.bulk.prefetch.L2 of the field ranges the step reads -- was
    //  measured SLOWER: 0.83 -> 0.71 of the HBM peak; eight warps per SM already keep enough loads in flight)
    const double* in = a.tiles + (size_t)tile * LY::TILE_DOUBLES + lane;
    double* out = a.dst_tiles ? (dst >= 0 ? a.dst_tiles + (size_t)(dst / TILE) * LY::TILE_DOUBLES + (dst % TILE) : nullptr)
                              : a.tiles + (size_t)tile * LY::TILE_DOUBLES + lane;
    if (act != ACT_NONE) {
      double meas[7];
      if (act == ACT_UPDATE) {
        const double* mp = a.meas + (size_t)slot * a.meas_stride;
#pragma unroll
        for (int k = 0; k < 7; ++k) meas[k] = __ldg(mp + k);
      }
      step_lane_av_sym<AV_SCRATCH_PREV, true, ZF>(in, out, sc, act, dt, meas, a.Qtab + (size_t)cls * N * N, a.Rtab + (size_t)cls * M * M, a.packed != 0);
      if (a.clear_action) a.action[slot] = 0;
      if (a.pos_out) {
#pragma unroll
        for (int k = 0; k < 3; ++k) a.pos_out[(size_t)slot * 3 + k] = sc[(LY::F_X + k) * TILE];
      }
    } else if (valid) {
      if (a.dst_tiles && dst >= 0) {   // compacting tick: an untouched survivor still moves to its new slot
#pragma unroll 8
        for (int f = 0; f < LY::NF; ++f) __stcs(out + (size_t)f * TILE, __ldcs(in + (size_t)f * TILE));
      }
      if (a.pos_out) {
#pragma unroll
        for (int k = 0; k < 3; ++k) a.pos_out[(size_t)slot * 3 + k] = in[(LY::F_X + k) * TILE];
      }
    }
    if (a.clear_action && lane == 0) a.tile_flag[tile] = 0;
  }
}

// The same for the linear models (UV / UA): no shared memory at all, everything lives in registers.  n_ticks > 1 = replay
// launch (te_pool_step_dense_ticks): the target stays in registers for all its ticks.
// MULTI: the replay / live instantiation (n_ticks > 1 or a tick gate); the single-tick instantiation carries none of its code (its
// registers cost the dense tick a spill).
// AXIS: the axis-blocked step (te_kin_sym.cuh) of a packed pool in which no class couples the axes: UA moves 29 of its 56 packed
// fields, UV 17 of 29.
template <int TYPE, int WARPS, int MIN_CTAS, bool MULTI = false, bool AXIS = false>
__global__ void __launch_bounds__(WARPS * 32, MIN_CTAS) kf_step_kin_direct_kernel(const StepArgs a) {
  using MT = Model<TYPE>;
  using LY = Layout<TYPE>;
  constexpr int N = MT::N, M = MT::M;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // Programmatic dependent launch (small pools are launched with programmatic stream serialization; without the launch
  // attribute the two griddepcontrol instructions are no-ops): the next tick's
  // grid may be scheduled while this one runs, and this one may have been scheduled while the previous kernel on the
  // stream was still running -- everything above griddepcontrol.wait touches only launch parameters; the wait returns
  // once all earlier work on the stream has completed and flushed.  Hides the launch latency between the ticks of a
  // small pool (BASELINE configs[1]: 10 000 targets, where a tick is a few microseconds).
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int gw = blockIdx.x * WARPS + warp, GW = gridDim.x * WARPS;
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const int n_work = a.d_nwork ? *a.d_nwork : a.n_tiles;
  for (int w = gw; w < n_work; w += GW) {
    const int tile = a.tile_list ? a.tile_list[w] : a.tile_begin + w;
    const int slot = tile * TILE + lane;
    const bool valid = slot < a.n_slots;
    int act = ACT_NONE, cls = 0, dst = -1;
    double dt = a.dt;
    if (valid) {
      act = a.action ? (int)a.action[slot] : a.default_action;
      if (a.dt_slot) dt = a.dt_slot[slot];
      cls = (int)a.cls[slot];
      if (a.dst_tiles) {
        if (a.dst_alive[slot]) dst = a.dst_pos[slot];
        else act = ACT_NONE;   // erased at the end of this tick: its step is unobservable
      }
    }
    const double* in = a.tiles + (size_t)tile * LY::TILE_DOUBLES + lane;
    double* out = a.dst_tiles ? (dst >= 0 ? a.dst_tiles + (size_t)(dst / TILE) * LY::TILE_DOUBLES + (dst % TILE) : nullptr)
                              : a.tiles + (size_t)tile * LY::TILE_DOUBLES + lane;
    const double* __restrict__ Q = a.Qtab + (size_t)cls * N * N;
    const double* __restrict__ R = a.Rtab + (size_t)cls * M * M;
    if (MULTI) {
      if (!valid) continue;
      // a lane whose actions are all ACT_NONE still goes through load / store: cheaper than a second pass to find out
      KinSym<TYPE, AXIS> ks;
      ks.load(in);
      if (a.tick_gate) {
        // live launch: the target stays in registers while its ticks arrive one by one -- a tick costs neither a launch nor a
        // trip of the state through L2.  Lane 0 watches the gate (released-tick count; the measurement block of a released tick is
        // complete), the warp applies the tick, publishes the positions and counts itself done.  Every warp owns ONE tile here
        // (the host sizes the grid so), so no tile waits behind another one's ticks.
        const unsigned m = __activemask();
        const int first = __ffs(m) - 1;
        int pub_released = 0, pub_stop = 0;
        int known = 0;          // lane `first`: ticks known to be released (a gate read shows all of them: a burst costs one read)
        int pending = 0;        // lane `first`: the completion count of the previous tick is still in flight
        int before = 0;
        auto resolve = [&]() {  // lane `first`: the previous tick's count has come back -- the last warp of a tick tells the host
          if (pending && before == a.tick_warps - 1 && a.tick_done_host) {
            // one posted 4-byte write over PCIe per tick.  No system-scope fence in front of it: the positions it announces are in
            // device memory, ordered at GPU scope by the acq_rel count, and whoever reads them (a copy engine, a kernel) reads
            // through the same L2 -- a __threadfence_system() here cost the announcing warp ~3 us per tick, and that warp then
            // arrived last at the next tick as well: the whole launch ran at tick + fence.
            asm volatile("st.relaxed.sys.global.s32 [%0], %1;" ::"l"(a.tick_done_host), "r"(pending) : "memory");
          }
          pending = 0;
        };
        auto count_done = [&](int tk) {   // lane `first`
          resolve();            // (one count in flight at a time: `before` is its return value)
          asm volatile("atom.add.acq_rel.gpu.global.s32 %0, [%1], 1;" : "=r"(before) : "l"(a.tick_done + tk) : "memory");
          pending = tk + 1;
        };
        int at_n = ACT_NONE;                      // inputs of the next tick, requested a tick ahead when it is already released
        double meas_n[3] = {0.0, 0.0, 0.0};
        bool have_n = false;
        for (int tick = 0; tick < a.n_ticks; ++tick) {
          int at = ACT_NONE;
          double meas[3] = {0.0, 0.0, 0.0};
          auto fetch = [&](int tk, int& at_o, double* meas_o) {   // a tick's inputs (written while this kernel runs: not through the read-only path)
            // (the measurement is requested whatever the action byte says: behind a branch on the byte the two L2 round trips would
            //  run one after the other)
            at_o = a.action ? (int)__ldcg(a.action + (size_t)tk * a.action_tick_stride + slot) : a.default_action;
            if (a.meas) {
              const double* mp = a.meas + (size_t)tk * a.meas_tick_stride + (size_t)slot * a.meas_stride;
#pragma unroll
              for (int k = 0; k < 3; ++k) meas_o[k] = __ldcg(mp + k);
            }
          };
          if (have_n) {
            // requested under the previous tick's arithmetic: a burst of released ticks costs no L2 round trip per tick
            at = at_n;
#pragma unroll
            for (int k = 0; k < 3; ++k) meas[k] = meas_n[k];
            // (no resolve() here: the count in flight was issued a moment ago, reading its return value now would wait for the whole
            //  L2 round trip; it is resolved in front of the next count, a tick of arithmetic later)
          } else {
            // a tick already known to be released: its inputs are requested before the previous tick's count is waited for, so the
            // two L2 round trips overlap
            const int ahead = __shfl_sync(m, known > tick ? 1 : 0, first);
            if (ahead) fetch(tick, at, meas);
            if (lane == first) resolve();
            if (!ahead) {
              int go = 1;
              if (lane == first) {
                // Two sources open the gate: the copy engine (a pushed tick: its block and then the count travel in order on the copy
                // stream) and the host itself (a released tick: one store to a page-locked word, no CUDA call).  The warp of tile 0
                // reads both -- the host word across PCIe -- and republishes their maximum in device memory for everybody else.
                for (;;) {
                  int released, stop;
                  if (gw == 0) {
                    int hr, hs, dr, ds;
                    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(hr) : "l"(a.tick_gate_host) : "memory");
                    asm volatile("ld.relaxed.sys.global.s32 %0, [%1];" : "=r"(hs) : "l"(a.tick_gate_host + 1) : "memory");
                    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(dr) : "l"(a.tick_gate) : "memory");
                    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(ds) : "l"(a.tick_gate + 1) : "memory");
                    released = hr > dr ? hr : dr;
                    stop = hs | ds;
                    if (released > pub_released || stop != pub_stop) {
                      if (stop != pub_stop) asm volatile("st.relaxed.gpu.global.s32 [%0], %1;" ::"l"(a.tick_gate_eff + 1), "r"(stop) : "memory");
                      asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(a.tick_gate_eff), "r"(released) : "memory");
                      pub_released = released;
                      pub_stop = stop;
                    }
                  } else {
                    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(released) : "l"(a.tick_gate_eff) : "memory");
                    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(stop) : "l"(a.tick_gate_eff + 1) : "memory");
                  }
                  known = released;
                  if (released > tick) break;
                  if (stop) { go = 0; break; }
                  __nanosleep(20);
                }
              }
              go = __shfl_sync(m, go, first);
              if (!go) break;
              fetch(tick, at, meas);
            }
          }
          // the next tick, if the gate read above has already shown it released: its inputs travel under this tick's arithmetic
          // (the acquire that showed the count orders them; the warp of tile 0 keeps republishing through its own reads)
          have_n = tick + 1 < a.n_ticks && __shfl_sync(m, known > tick + 1 ? 1 : 0, first) != 0;
          if (have_n) fetch(tick + 1, at_n, meas_n);
          if (at != ACT_NONE) ks.tick(at, dt, meas, Q, R);
          if (a.pos_out && a.pos_tick_stride > 0) {
#pragma unroll
            for (int k = 0; k < 3; ++k) __stcg(a.pos_out + (size_t)tick * a.pos_tick_stride + (size_t)slot * 3 + k, ks.x[k]);
          }
          // completion count: the warp barrier orders every lane's position stores before lane `first`'s acq_rel increment
          // (release patterns are cumulative), so whoever sees the full count -- the last warp -- has every warp's stores behind it.
          // A tick whose successor is already here (a burst) is NOT counted: a warp applies its ticks in order, so the count of the
          // burst's last tick announces all of them, and the release fence in front of every count -- an L2 round trip with the whole
          // warp waiting behind lane `first` -- is paid once per burst.  A tick released alone is counted at once, as before.
          __syncwarp(m);
          if (lane == first && !have_n) count_done(tick);
        }
        if (lane == first) resolve();
        ks.store(out, a.packed != 0);
        if (a.pos_out && a.pos_tick_stride == 0) {
#pragma unroll
          for (int k = 0; k < 3; ++k) a.pos_out[(size_t)slot * 3 + k] = ks.x[k];
        }
        continue;
      }
      // replay: the inputs of tick k + 1 are requested before tick k is applied (and the measurement whatever the action byte says),
      // so no tick waits for an L2 round trip
      auto fetch_replay = [&](int tk, int& at_o, double* meas_o) {
        at_o = a.action ? (int)a.action[(size_t)tk * a.action_tick_stride + slot] : a.default_action;
        if (a.meas) {
          const double* mp = a.meas + (size_t)tk * a.meas_tick_stride + (size_t)slot * a.meas_stride;
#pragma unroll
          for (int k = 0; k < 3; ++k) meas_o[k] = __ldg(mp + k);
        }
      };
      int at_n = ACT_NONE;
      double meas_n[3] = {0.0, 0.0, 0.0};
      fetch_replay(0, at_n, meas_n);
      for (int tick = 0; tick < a.n_ticks; ++tick) {
        const int at = at_n;
        const double meas[3] = {meas_n[0], meas_n[1], meas_n[2]};
        if (tick + 1 < a.n_ticks) fetch_replay(tick + 1, at_n, meas_n);
        if (at == ACT_NONE) continue;
        ks.tick(at, dt, meas, Q, R);
      }
      ks.store(out, a.packed != 0);
      if (a.pos_out) {
#pragma unroll
        for (int k = 0; k < 3; ++k) a.pos_out[(size_t)slot * 3 + k] = ks.x[k];
      }
      continue;
    }
    if (act != ACT_NONE) {
      double meas[3];
      if (act == ACT_UPDATE) {
        const double* mp = a.meas + (size_t)slot * a.meas_stride;
#pragma unroll
        for (int k = 0; k < 3; ++k) meas[k] = __ldg(mp + k);
      }
      KinSym<TYPE, AXIS> ks;
      ks.load(in);
      ks.tick(act, dt, meas, Q, R);
      ks.store(out, a.packed != 0, AXIS && a.dst_tiles);
      if (a.pos_out) {
#pragma unroll
        for (int k = 0; k < 3; ++k) a.pos_out[(size_t)slot * 3 + k] = ks.x[k];
      }
      if (a.clear_action) a.action[slot] = 0;
    } else if (valid) {
      if (a.dst_tiles && dst >= 0) {   // compacting tick: an untouched survivor still moves to its new slot
#pragma unroll 8
        for (int f = 0; f < LY::NF; ++f) __stcs(out + (size_t)f * TILE, __ldcs(in + (size_t)f * TILE));
      }
      if (a.pos_out) {
#pragma unroll
        for (int k = 0; k < 3; ++k) a.pos_out[(size_t)slot * 3 + k] = in[(LY::F_X + k) * TILE];
      }
    }
    if (a.clear_action && lane == 0) a.tile_flag[tile] = 0;
  }
}

}  // namespace te
