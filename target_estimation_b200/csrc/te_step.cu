// te_step.cu -- launch policy of the step kernels (which kernel shape serves which model / pool size / variant) and the stepping
// entry points of include/te_pool.h: dense tick, replay launch, host-buffer ticks, sparse tick by id, the fused churn tick.
#include <cub/device/device_scan.cuh>

#include "te_pool_internal.cuh"
#include "te_split.cuh"
#include "te_direct.cuh"
#include "te_av_stream.cuh"

namespace tehost {

// te_pool_set_grid_cap: a small pool under a capped grid walks the same persistent loops (grid-stride tiles, the STAGES ring of
// the split kernel with its mbarrier phase flips) that a bench-size pool walks on the full machine
inline int capped(const te_pool* p, int grid) { return p->grid_cap > 0 ? std::min(grid, p->grid_cap) : grid; }
template <int TYPE, int WARPS, int STAGES, bool MULTI = false, int IMPL = 0>
void launch_step_t(te_pool* p, const te::StepArgs& a, int n_work_hint) {
  auto kern = te::kf_step_kernel<TYPE, WARPS, STAGES, MULTI, IMPL>;
  const size_t smem = te::step_smem_bytes<TYPE>(WARPS, STAGES);
  static thread_local int configured_dev = -1;
  static bool configured[64] = {false};
  (void)configured_dev;
  if (!configured[p->device & 63]) {
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured[p->device & 63] = true;
  }
  int grid = capped(p, std::min(p->n_sm, std::max(1, cdiv(n_work_hint, WARPS))));
  kern<<<grid, WARPS * 32, smem, p->stream>>>(a);
  CK(cudaGetLastError());
}

// row/column-split kernel (te_split.cuh): one CTA of 6*CS warps per tile, STAGES stages per CTA, CTAS CTAs per SM
template <int TYPE, int CS, int STAGES, int CTAS, bool COMPACT>
void launch_split_k(te_pool* p, const te::StepArgs& a, int n_work_hint) {
  auto kern = te::kf_step_split_kernel<TYPE, CS, STAGES, CTAS, COMPACT>;
  const size_t smem = te::split_smem_bytes<TYPE>(STAGES);
  static bool configured[64] = {false};
  if (!configured[p->device & 63]) {
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured[p->device & 63] = true;
  }
  int grid = capped(p, std::min(p->n_sm * CTAS, std::max(1, n_work_hint)));
  kern<<<grid, (te::SPLIT_RS * CS + te::split_nt<TYPE>()) * 32, smem, p->stream>>>(a);
  CK(cudaGetLastError());
}
template <int TYPE, int CS, int STAGES, int CTAS>
void launch_split_t(te_pool* p, const te::StepArgs& a, int n_work_hint) { launch_split_k<TYPE, CS, STAGES, CTAS, false>(p, a, n_work_hint); }

bool uses_direct(const te_pool* p);
void ensure_full(te_pool* p);
void launch_kin(te_pool* p, const te::StepArgs& a, int n_work_hint);
void launch_step_multi(te_pool* p, const te::StepArgs& a_in, int n_work_hint) {
  te::StepArgs a = a_in;
  if (uses_direct(p) && p->model != te::ANGULAR_VELOCITIES) {   // UV / UA: the direct kernel keeps the target in registers for all ticks
    a.packed = (p->all_sym && p->variant != 12) ? 1 : 0;
    if (a.packed) p->lower_stale = true;
    launch_kin(p, a, n_work_hint);
    return;
  }
  ensure_full(p);
  switch (p->model) {
    case te::UNIFORM_VELOCITY: launch_step_t<te::UNIFORM_VELOCITY, 8, 2, true>(p, a, n_work_hint); break;
    case te::UNIFORM_ACCELERATION: launch_step_t<te::UNIFORM_ACCELERATION, 4, 2, true>(p, a, n_work_hint); break;
    case te::ANGULAR_VELOCITIES: launch_step_t<te::ANGULAR_VELOCITIES, 5, 1, true>(p, a, n_work_hint); break;
    default: launch_step_t<te::ANGULAR_RATES, 2, 1, true>(p, a, n_work_hint); break;
  }
}

template <int WARPS, int ZF = 2>
void launch_av_direct(te_pool* p, const te::StepArgs& a, int n_work_hint) {
  auto kern = te::kf_step_av_direct_kernel<WARPS, ZF>;
  const size_t smem = te::av_direct_smem_bytes(WARPS);
  static bool configured[64] = {false};
  if (!configured[p->device & 63]) {
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured[p->device & 63] = true;
  }
  int grid = capped(p, std::min(p->n_sm, std::max(1, cdiv(n_work_hint, WARPS))));
  kern<<<grid, WARPS * 32, smem, p->stream>>>(a);
  CK(cudaGetLastError());
}

// dense in-place packed tick of an AV pool: the TMA-streamed kernel (te_av_stream.cuh)
bool av_stream_serves(const te_pool* p, const te::StepArgs& a) {
  if (p->variant != 0 || !a.packed || !p->whiten_ok) return false;   // 13 = the direct kernel for every launch
  if (a.tile_list || a.d_nwork || a.dt_slot || a.clear_action || a.n_ticks != 1 || a.tick_gate) return false;
  if (a.meas && (a.meas_stride != 7 || (reinterpret_cast<uintptr_t>(a.meas) & 15) != 0)) return false;
  if (!a.meas && (a.action || a.default_action == te::ACT_UPDATE)) return false;
  return true;
}
template <bool QC, bool COMPACT>
void launch_av_stream_k(te_pool* p, const te::StepArgs& a, int n_work_hint) {
  constexpr int WARPS = 8;
  auto kern = te::kf_step_av_stream_kernel<WARPS, QC, COMPACT>;
  const size_t smem = te::av_stream_smem_bytes(WARPS);
  static bool configured[64] = {false};
  if (!configured[p->device & 63]) {
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured[p->device & 63] = true;
  }
  int grid = capped(p, std::min(p->n_sm, std::max(1, cdiv(n_work_hint, WARPS))));
  kern<<<grid, WARPS * 32, smem, p->stream>>>(a);
  CK(cudaGetLastError());
}
template <bool QC>
void launch_av_stream(te_pool* p, const te::StepArgs& a, int n_work_hint) {
  if (a.dst_tiles) launch_av_stream_k<QC, true>(p, a, n_work_hint);
  else launch_av_stream_k<QC, false>(p, a, n_work_hint);
}

template <int TYPE, int WARPS, int CTAS, bool AXIS>
void launch_kin_direct_k(te_pool* p, const te::StepArgs& a, int n_work_hint) {
  const bool multi = a.n_ticks > 1 || a.tick_gate != nullptr;   // replay / live launches: an instantiation of their own
  auto kern = multi ? te::kf_step_kin_direct_kernel<TYPE, WARPS, CTAS, true, AXIS> : te::kf_step_kin_direct_kernel<TYPE, WARPS, CTAS, false, AXIS>;
  int grid = capped(p, std::min(p->n_sm * CTAS, std::max(1, cdiv(n_work_hint, WARPS))));
  // programmatic stream serialization: see the kernel's griddepcontrol.wait
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(WARPS * 32);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = p->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  // Only for small pools, where a tick is a few microseconds and the launch latency matters.  For big pools it buys nothing,
  // and in a process with an NCCL communicator it was measured to cost 37 % (4 Mi UA targets: 0.64 -> 0.86 ms per tick under
  // torchrun, 0.63 either way in a plain process) -- the early-scheduled grid and the running one compete for the SMs.
  static const bool no_pdl = std::getenv("TE_NO_PDL") != nullptr;   // debugging switch
  cfg.attrs = attr;
  cfg.numAttrs = (no_pdl || n_work_hint > 4 * p->n_sm) ? 0 : 1;
  CK(cudaLaunchKernelEx(&cfg, kern, a));
}
// small pools (fewer tiles than the SMs have scheduler partitions) spread over more, smaller CTAs: one warp per partition has
// the FP64 pipe to itself, which is what bounds a tick of a few hundred tiles
template <int TYPE, int WARPS, int CTAS, bool AXIS>
void launch_kin_direct(te_pool* p, const te::StepArgs& a, int n_work_hint) {
  if (n_work_hint <= 2 * p->n_sm) launch_kin_direct_k<TYPE, 2, 1, AXIS>(p, a, n_work_hint);
  else if (n_work_hint <= 4 * p->n_sm) launch_kin_direct_k<TYPE, 4, 1, AXIS>(p, a, n_work_hint);
  else launch_kin_direct_k<TYPE, WARPS, CTAS, AXIS>(p, a, n_work_hint);
}
// The axis-blocked form at its large-pool shape.  TE_AXIS_SHAPE ("WARPSxCTAS", read per call) is the tuning knob with which
// tools/bench_axis_blocks.py measures the other shapes against it.
template <int TYPE, int WARPS, int CTAS>
void launch_kin_axis(te_pool* p, const te::StepArgs& a, int n_work_hint) {
  const char* shape = std::getenv("TE_AXIS_SHAPE");
  if (shape && n_work_hint > 4 * p->n_sm) {
    if (!std::strcmp(shape, "8x1")) return launch_kin_direct_k<TYPE, 8, 1, true>(p, a, n_work_hint);
    if (!std::strcmp(shape, "8x2")) return launch_kin_direct_k<TYPE, 8, 2, true>(p, a, n_work_hint);
    if (!std::strcmp(shape, "4x3")) return launch_kin_direct_k<TYPE, 4, 3, true>(p, a, n_work_hint);
    if (!std::strcmp(shape, "4x4")) return launch_kin_direct_k<TYPE, 4, 4, true>(p, a, n_work_hint);
  }
  launch_kin_direct<TYPE, WARPS, CTAS, true>(p, a, n_work_hint);
}
// UV / UA on the direct kernels (variants 0 / 12 / 13): the axis-blocked form when the pool is packed and no class couples the axes
void launch_kin(te_pool* p, const te::StepArgs& a, int n_work_hint) {
  const bool axis = a.packed && p->all_axis;
  if (p->model == te::UNIFORM_VELOCITY) {
    // measured, packed, 4 Mi targets: <4,3> (12 warps per SM) 1.17e10, <4,4> 1.11e10, <8,1> 1.09e10 steps/s.  Axis-blocked (80 registers
    // against 128; tools/bench_axis_blocks.py, B200 at 1000 W, ms per tick in two runs): <8,2> 0.2285 / 0.2321, <4,4> 0.2299 / 0.2318,
    // <4,3> 0.2349 / 0.2339, <8,1> 0.2823 / 0.2786
    if (axis) launch_kin_axis<te::UNIFORM_VELOCITY, 8, 2>(p, a, n_work_hint);
    else launch_kin_direct<te::UNIFORM_VELOCITY, 4, 3, false>(p, a, n_work_hint);
  } else {
    // axis-blocked (126 registers against 234), 4 Mi targets, ms per tick in two runs: <4,3> 0.3720 / 0.3728, <8,2> 0.3778 / 0.3785,
    // <4,4> 0.3797 / 0.3798, <8,1> 0.3822 / 0.3806
    if (axis) launch_kin_axis<te::UNIFORM_ACCELERATION, 4, 3>(p, a, n_work_hint);
    else launch_kin_direct<te::UNIFORM_ACCELERATION, 8, 1, false>(p, a, n_work_hint);
  }
}

// does the current variant run a direct symmetric-covariance kernel (te_direct.cuh)?
bool uses_direct(const te_pool* p) {
  // variant 0 = the defaults; 12 = the direct kernels writing both halves of the covariance (unpacked); 1 / 10 / 11 = staged forms
  const int v = p->variant;
  if (p->model == te::ANGULAR_RATES) return false;
  return ((v == 0 || v == 13) && p->all_sym) || v == 12;
}
// full-matrix kernels (and anything else that reads both halves) first get the lower triangles back
void ensure_full(te_pool* p) {
  if (!p->lower_stale || p->n == 0) { p->lower_stale = false; return; }
  double* tiles = p->buf[p->cur].tiles;
  const int n = (int)p->n;
  switch (p->model) {
    case te::UNIFORM_VELOCITY: te::mirror_lower_kernel<te::UNIFORM_VELOCITY><<<cdiv(n, 128), 128, 0, p->stream>>>(tiles, n); break;
    case te::UNIFORM_ACCELERATION: te::mirror_lower_kernel<te::UNIFORM_ACCELERATION><<<cdiv(n, 128), 128, 0, p->stream>>>(tiles, n); break;
    case te::ANGULAR_VELOCITIES: te::mirror_lower_kernel<te::ANGULAR_VELOCITIES><<<cdiv(n, 128), 128, 0, p->stream>>>(tiles, n); break;
    default: te::mirror_lower_kernel<te::ANGULAR_RATES><<<cdiv(n, 128), 128, 0, p->stream>>>(tiles, n); break;
  }
  CK(cudaGetLastError());
  p->lower_stale = false;
}

// Stage bytes of the staged kernel: UV 13056, UA 25344, AV 43008, AR 90624.
// Kernel per model and variant.  Variants are what the tests switch between, not tuning shapes:
//   0   default, while every class is bitwise symmetric (packed: upper triangle only): UV / UA direct symmetric-covariance kernels
//       (te_direct.cuh), in their axis-blocked form (per-axis covariance blocks only) while no class couples the axes; AV dense
//       ticks (in place and compacting) the TMA-streamed kernel (te_av_stream.cuh), AV sparse ticks and pools with a class whose R
//       has no Cholesky factor the direct kernel; AR the warp-specialised row-split kernel on the full matrix (te_split.cuh).  A
//       pool with an asymmetric class runs the full-matrix kernels (10).
//   1   the TMA-staged one-warp-per-tile kernel on the full matrix (te_kernels.cuh; also what replay launches of AV / AR run)
//   10  forced full-matrix kernels (UV / UA staged, AV row-split): what a pool with an asymmetric class runs
//   11  AR row-split kernel moving the upper triangle only (44 % fewer bytes, not faster: DESIGN.md section 7)
//   12  UV / UA / AV direct kernels writing both halves of the covariance (never the axis-blocked form)
//   13  as 0, but AV dense ticks on the direct kernel too
// Shape experiments of round 1 (warps x stages sweeps, the AR / AV two-lanes-per-target kernels, thread-per-target AR) were
// measured, lost, and are gone from the tree: DESIGN.md section 7 keeps their numbers.
void launch_step(te_pool* p, const te::StepArgs& a_in, int n_work_hint) {
  const int v = p->variant;
  te::StepArgs a = a_in;
  if (uses_direct(p)) {
    a.packed = (p->all_sym && v != 12) ? 1 : 0;   // (0 / 13)
    if (a.packed) p->lower_stale = true;
    switch (p->model) {
      case te::UNIFORM_VELOCITY:
      case te::UNIFORM_ACCELERATION:
        launch_kin(p, a, n_work_hint);
        return;
      default:
        if (av_stream_serves(p, a)) {
          if (p->hQ.size() == 1 && a.cls_c == 0) launch_av_stream<true>(p, a, n_work_hint);
          else launch_av_stream<false>(p, a, n_work_hint);
        } else {
          launch_av_direct<8>(p, a, n_work_hint);
        }
        return;
    }
  }
  if (p->model == te::ANGULAR_RATES && v == 11 && p->all_sym) {
    a.packed = 1;
    p->lower_stale = true;
  } else {
    ensure_full(p);
  }
  if (a.dst_tiles) {
    // compacting tick: separate instantiations of the default split configurations, so that the in-place kernels carry
    // none of its code (the AV kernel at 128 registers lost 6 % to a few extra runtime branches)
    if (p->model == te::ANGULAR_VELOCITIES) return launch_split_k<te::ANGULAR_VELOCITIES, 1, 2, 2, true>(p, a, n_work_hint);
    if (p->model == te::ANGULAR_RATES) return launch_split_k<te::ANGULAR_RATES, 1, 2, 1, true>(p, a, n_work_hint);
  }
  switch (p->model) {
    case te::UNIFORM_VELOCITY: launch_step_t<te::UNIFORM_VELOCITY, 8, 2>(p, a, n_work_hint); break;
    case te::UNIFORM_ACCELERATION: launch_step_t<te::UNIFORM_ACCELERATION, 4, 2>(p, a, n_work_hint); break;
    case te::ANGULAR_VELOCITIES:
      if (v == 1) launch_step_t<te::ANGULAR_VELOCITIES, 5, 1>(p, a, n_work_hint);
      else launch_split_t<te::ANGULAR_VELOCITIES, 1, 2, 2>(p, a, n_work_hint);
      break;
    default: launch_split_t<te::ANGULAR_RATES, 1, 2, 1>(p, a, n_work_hint); break;
  }
}

te::StepArgs base_args(te_pool* p) {
  te::StepArgs a{};
  Buf& b = p->buf[p->cur];
  a.tiles = b.tiles;
  a.n_slots = (int)p->n;
  a.n_tiles = cdiv(p->n, te::TILE);
  a.cls = b.cold.cls;
  a.Qtab = p->dQ;
  a.Rtab = p->dR;
  a.Ttab = p->dT;
  a.n_ticks = 1;
  a.cls_c = -1;
  if (!p->hQ.empty()) {   // class 0 rides in the parameter constant bank
    a.cls_c = 0;
    std::memcpy(a.Qc, p->hQ[0].data(), sizeof(double) * p->N * p->N);
    std::memcpy(a.Rc, p->hR[0].data(), sizeof(double) * p->M * p->M);
    std::memcpy(a.Tc, p->hT[0].data(), sizeof(double) * p->M * p->M);
  }
  return a;
}

void check_meas_stride(te_pool* p, int stride) {
  if (stride == 7) return;
  if (stride == 3 && p->M == 3) return;
  throw std::invalid_argument("meas_stride must be 7 (pose) or 3 (xyz, UV/UA pools only)");
}

}  // namespace tehost

using namespace tehost;
#define g_err (tehost::last_error())

extern "C" {

int te_pool_step_dense(te_pool* p, double dt, const double* dev_meas, int meas_stride, const uint8_t* dev_action, int default_action) {
  return guarded(p, [&] {
    if (p->n == 0) return 0;
    if (!(dt >= 0.0)) throw std::invalid_argument("dt must be >= 0 (assert of src/target_interface.cpp:150)");
    te::StepArgs a = base_args(p);
    a.dt = dt;
    a.meas = dev_meas;
    a.meas_stride = meas_stride;
    a.action = const_cast<uint8_t*>(dev_action);
    a.default_action = default_action;
    if (dev_meas) {
      check_meas_stride(p, meas_stride);
      a.meas_tma = ((uintptr_t)dev_meas % 16 == 0) ? 1 : 0;
    } else if (dev_action || default_action == TE_ACT_UPDATE) {
      // (an action array may name ACT_UPDATE for any slot: without measurements the kernel would read a null pointer)
      throw std::invalid_argument("update tick without measurements");
    }
    launch_step(p, a, a.n_tiles);
    return 0;
  });
}

int te_pool_step_dense_ticks(te_pool* p, int n_ticks, double dt, const double* dev_meas, int meas_stride, const uint8_t* dev_action,
                             int default_action) {
  return guarded(p, [&] {
    if (p->n == 0 || n_ticks <= 0) return 0;
    if (!(dt >= 0.0)) throw std::invalid_argument("dt must be >= 0");
    if (dev_meas) check_meas_stride(p, meas_stride);
    else if (default_action == TE_ACT_UPDATE || dev_action) throw std::invalid_argument("update ticks without measurements");
    te::StepArgs a = base_args(p);
    a.dt = dt;
    a.meas = dev_meas;
    a.meas_stride = meas_stride;
    a.meas_tma = 0;
    a.action = const_cast<uint8_t*>(dev_action);
    a.default_action = default_action;
    a.n_ticks = n_ticks;
    a.meas_tick_stride = (long long)p->n * meas_stride;
    a.action_tick_stride = p->n;
    launch_step_multi(p, a, a.n_tiles);
    return 0;
  });
}

// ---- live launch: the 250 Hz loop over a small pool without a launch (or a trip of the state through L2) per tick ------------------
namespace {
struct LiveScope {
  LiveScope() { live_call() = true; }
  ~LiveScope() { live_call() = false; }
};
void live_gate_write(te_pool* p, int index, int value) {   // a 4-byte write into the gate block, on the copy stream (the pool's stream is busy)
  te_pool::Live& lv = p->live;
  static thread_local unsigned ring_pos = 0;
  int* src = lv.h_ring + (ring_pos++ & 255);
  *src = value;
  CK(cudaMemcpyAsync(lv.d_gate + index, src, sizeof(int), cudaMemcpyHostToDevice, p->h2d_stream));
}
}  // namespace

int te_pool_live_begin(te_pool* p, int max_ticks, double dt, double* dev_meas, int meas_stride, uint8_t* dev_action, int default_action,
                       double* dev_pos) {
  LiveScope ls;
  return guarded(p, [&] {
    te_pool::Live& lv = p->live;
    if (lv.active) throw std::logic_error("a live launch is already running");
    if (p->n == 0 || max_ticks <= 0) throw std::invalid_argument("empty pool or no ticks");
    if (!(dt >= 0.0)) throw std::invalid_argument("dt must be >= 0");
    if (!(uses_direct(p) && p->model != te::ANGULAR_VELOCITIES)) throw std::invalid_argument("live launches serve uniform-velocity / uniform-acceleration pools");
    if (!dev_meas && (default_action == TE_ACT_UPDATE || dev_action)) throw std::invalid_argument("update ticks without measurements");
    if (dev_meas) check_meas_stride(p, meas_stride);
    const int n_tiles = cdiv(p->n, te::TILE);
    if (n_tiles > p->n_sm * 8) throw std::invalid_argument("pool too large for a live launch: every warp of one resident grid holds one tile in registers");
    if (p->grid_cap > 0) throw std::invalid_argument("live launches need the whole grid (te_pool_set_grid_cap is set)");
    if (!p->h2d_stream) {
      CK(cudaStreamCreateWithFlags(&p->h2d_stream, cudaStreamNonBlocking));
      CK(cudaStreamCreateWithFlags(&p->d2h_stream, cudaStreamNonBlocking));
    }
    if (!lv.h_ring) CK(cudaHostAlloc((void**)&lv.h_ring, 260 * sizeof(int), cudaHostAllocMapped));
    if ((size_t)max_ticks + 4 > lv.d_cap) {
      cudaFree(lv.d_gate);
      lv.d_gate = nullptr;
      CK(cudaMalloc((void**)&lv.d_gate, ((size_t)max_ticks + 4) * sizeof(int)));
      lv.d_cap = (size_t)max_ticks + 4;
    }
    CK(cudaMemsetAsync(lv.d_gate, 0, ((size_t)max_ticks + 4) * sizeof(int), p->stream));
    lv.h_ring[256] = lv.h_ring[257] = lv.h_ring[258] = 0;
    void* done_dev = nullptr;
    CK(cudaHostGetDevicePointer(&done_dev, lv.h_ring + 256, 0));
    te::StepArgs a = base_args(p);
    a.dt = dt;
    a.meas = dev_meas;
    a.meas_stride = meas_stride;
    a.meas_tma = 0;
    a.action = dev_action;
    a.default_action = default_action;
    a.n_ticks = max_ticks;
    a.meas_tick_stride = (long long)p->n * meas_stride;
    a.action_tick_stride = p->n;
    a.pos_out = dev_pos;
    a.pos_tick_stride = dev_pos ? (long long)p->n * 3 : 0;
    a.tick_gate = lv.d_gate;
    a.tick_gate_eff = lv.d_gate + 2;
    a.tick_done = lv.d_gate + 4;
    a.tick_done_host = (int*)done_dev;
    a.tick_gate_host = (int*)done_dev + 1;
    a.tick_warps = n_tiles;
    launch_step_multi(p, a, a.n_tiles);
    lv.active = true;
    lv.max_ticks = max_ticks;
    lv.released = 0;
    lv.stride = meas_stride;
    lv.d_meas = dev_meas;
    lv.d_action = dev_action;
    return 0;
  });
}

int te_pool_live_release(te_pool* p, int upto) {
  LiveScope ls;
  return guarded(p, [&] {
    te_pool::Live& lv = p->live;
    if (!lv.active) throw std::logic_error("no live launch");
    if (upto > lv.max_ticks) throw std::invalid_argument("more ticks than the launch holds");
    if (upto <= lv.released) return lv.released;
    // the caller's blocks are complete (its contract): one store to the page-locked gate word, no CUDA call; the launch's
    // gate-keeping warp reads it across PCIe
    __atomic_store_n(lv.h_ring + 257, upto, __ATOMIC_RELEASE);
    lv.released = upto;
    return upto;
  });
}

int te_pool_live_push(te_pool* p, const double* meas, const uint8_t* action) {
  LiveScope ls;
  return guarded(p, [&] {
    te_pool::Live& lv = p->live;
    if (!lv.active) throw std::logic_error("no live launch");
    if (lv.released >= lv.max_ticks) throw std::invalid_argument("the launch holds no more ticks");
    const int k = lv.released;
    // the tick's block, then the gate, in order on the copy stream: the kernel sees a released tick only with its data complete
    if (meas && lv.d_meas) CK(cudaMemcpyAsync(lv.d_meas + (size_t)k * p->n * lv.stride, meas, (size_t)p->n * lv.stride * 8, cudaMemcpyHostToDevice, p->h2d_stream));
    if (action && lv.d_action) CK(cudaMemcpyAsync(lv.d_action + (size_t)k * p->n, action, (size_t)p->n, cudaMemcpyHostToDevice, p->h2d_stream));
    live_gate_write(p, 0, k + 1);
    lv.released = k + 1;
    return k + 1;
  });
}

int te_pool_live_wait(te_pool* p, int ticks) {
  LiveScope ls;
  return guarded(p, [&] {
    te_pool::Live& lv = p->live;
    if (!lv.active) throw std::logic_error("no live launch");
    if (ticks > lv.released) throw std::invalid_argument("waiting for a tick that has not been released");
    volatile int* done = lv.h_ring + 256;
    const auto t0 = std::chrono::steady_clock::now();
    long long spins = 0;
    while (*done < ticks) {
      if ((++spins & 0xFFFF) == 0) {
        if (cudaStreamQuery(p->stream) != cudaErrorNotReady) break;   // the launch ended (an error, or all ticks done)
        if (std::chrono::steady_clock::now() - t0 > std::chrono::seconds(20)) throw std::runtime_error("live tick timed out");
      }
    }
    return (int)*done;
  });
}

int te_pool_live_end(te_pool* p) {
  LiveScope ls;
  return guarded(p, [&] {
    te_pool::Live& lv = p->live;
    if (!lv.active) return 0;
    CK(cudaStreamSynchronize(p->h2d_stream));               // pushed ticks have reached the device
    __atomic_store_n(lv.h_ring + 258, 1, __ATOMIC_RELEASE);   // stop: ticks not released by now are skipped
    const cudaError_t e = cudaStreamSynchronize(p->stream);
    lv.active = false;
    if (e != cudaSuccess) throw CudaError(std::string("live launch: ") + cudaGetErrorString(e));
    return (int)lv.h_ring[256];
  });
}

int te_pool_step_dense_host(te_pool* p, double dt, const double* meas, int meas_stride, const uint8_t* action, int default_action) {
  return guarded(p, [&] {
    if (p->n == 0) return 0;
    if (!(dt >= 0.0)) throw std::invalid_argument("dt must be >= 0");
    te::StepArgs a = base_args(p);
    a.dt = dt;
    a.default_action = default_action;
    if (meas) {
      check_meas_stride(p, meas_stride);
      if (meas_stride == 7) {
        // measured_pose_ = meas (src/target_interface.cpp:142-146): land the batch in the pool's own record
        // for UPDATE slots only -> stage, then the kernel-side copy would cost a pass; instead keep the
        // staged batch as this tick's measurement block and refresh measured_pose_ with one D2D copy
        // when every slot is updated.
        double* d = to_dev(p, meas, (size_t)p->n * 7);
        a.meas = d;
        if (!action && default_action == TE_ACT_UPDATE)
          CK(cudaMemcpyAsync(p->buf[p->cur].cold.meas, d, (size_t)p->n * 7 * 8, cudaMemcpyDeviceToDevice, p->stream));
      } else {
        a.meas = to_dev(p, meas, (size_t)p->n * meas_stride);
      }
      a.meas_stride = meas_stride;
      a.meas_tma = 1;
    } else if (!action && default_action == TE_ACT_UPDATE) {
      throw std::invalid_argument("update tick without measurements");
    }
    if (action) a.action = to_dev(p, action, (size_t)p->n);
    launch_step(p, a, a.n_tiles);
    if (action && meas && meas_stride == 7) {
      // masked refresh of measured_pose_ for the UPDATE slots
      te::copy_meas_masked_kernel<<<cdiv(p->n, 256), 256, 0, p->stream>>>(p->buf[p->cur].cold.meas, a.meas, a.action, (int)p->n);
      CK(cudaGetLastError());
    }
    CK(cudaStreamSynchronize(p->stream));
    return 0;
  });
}

namespace {

void tick_set_reserve(te_pool* p, te_pool::TickSet& ts, size_t meas_bytes, size_t act_bytes, size_t pos_bytes) {
  auto grow = [&](void** ptr, size_t& cap, size_t need) {
    if (need <= cap) return;
    CK(cudaStreamSynchronize(p->stream));
    CK(cudaStreamSynchronize(p->h2d_stream));
    CK(cudaStreamSynchronize(p->d2h_stream));
    cudaFree(*ptr);
    *ptr = nullptr;
    cap = 0;
    const size_t c = need + need / 8 + 256;
    CK(cudaMalloc(ptr, c));
    cap = c;
  };
  grow((void**)&ts.meas, ts.meas_cap, meas_bytes);
  grow((void**)&ts.act, ts.act_cap, act_bytes);
  grow((void**)&ts.pos, ts.pos_cap, pos_bytes);
  if (!ts.step_done) {
    CK(cudaEventCreateWithFlags(&ts.step_done, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ts.d2h_done, cudaEventDisableTiming));
  }
}

// one dense tick from host buffers, enqueued on the pool's three streams; nothing here waits on the host
void tick_host_enqueue(te_pool* p, double dt, const double* meas, int meas_stride, const uint8_t* action, int default_action, double* est_pos_out,
                       bool pipelined) {
  if (!(dt >= 0.0)) throw std::invalid_argument("dt must be >= 0");
  if (meas) check_meas_stride(p, meas_stride);
  else if (!action && default_action == TE_ACT_UPDATE) throw std::invalid_argument("update tick without measurements");
  if (!p->h2d_stream) {
    CK(cudaStreamCreateWithFlags(&p->h2d_stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&p->d2h_stream, cudaStreamNonBlocking));
  }
  const long long n = p->n;
  const int n_tiles = cdiv(n, te::TILE);
  // Chunk of the copy / step / read-back pipeline.  Measured (tools/e2e_probe.py, 4 Mi UA targets, xyz in / positions out, ms per
  // tick, one tick at a time | two ticks in flight): 2048 tiles 4.09 | 4.05, 8192 tiles 3.14 | 3.03, 32768 tiles 2.99 | 2.61,
  // 131072 tiles 4.31 | 2.47 -- many small copies in both directions at once cost the link a third of its rate; with two ticks in
  // flight the overlap comes from the neighbouring tick, so the chunks can be the whole pool.
  const char* chunk_str = std::getenv("TE_TICK_CHUNK_TILES");   // tuning / test knob, read per call
  const int chunk_env = chunk_str ? std::atoi(chunk_str) : 0;
  const int chunk_tiles = std::max(256, std::min(n_tiles, chunk_env > 0 ? chunk_env : (pipelined ? 131072 : 32768)));
  const int n_chunks = cdiv(n_tiles, chunk_tiles);
  te_pool::TickSet& ts = p->tick_set[p->ticks_issued % te_pool::TICK_SETS];
  if (ts.busy) {   // the tick that used this set three ticks ago must have left it (its results are in the caller's buffer by then)
    CK(cudaEventSynchronize(ts.d2h_done));
    ts.busy = false;
  }
  tick_set_reserve(p, ts, meas ? (size_t)n * meas_stride * 8 : 0, action ? (size_t)n : 0, est_pos_out ? (size_t)n * 24 : 0);
  while ((int)ts.ev.size() < 2 * n_chunks) {
    cudaEvent_t e;
    CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    ts.ev.push_back(e);
  }
  double* d_meas = meas ? ts.meas : nullptr;
  uint8_t* d_act = action ? ts.act : nullptr;
  double* d_pos = est_pos_out ? ts.pos : nullptr;
  // the copies of this tick may start as soon as the kernels that last read this set's staging are done (three ticks ago: already
  // waited for above through d2h_done, which follows them) and whatever the caller queued on the pool's stream before this call
  // that could touch the pool -- nothing reads the staging but the step kernels, so the copy stream needs no further wait
  te::StepArgs a = base_args(p);
  a.dt = dt;
  a.meas = d_meas;
  a.meas_stride = meas_stride;
  a.meas_tma = d_meas ? 1 : 0;
  a.action = d_act;
  a.default_action = default_action;
  a.pos_out = d_pos;
  for (int c = 0; c < n_chunks; ++c) {
    const long long s0 = (long long)c * chunk_tiles * te::TILE;
    const long long s1 = std::min<long long>(n, s0 + (long long)chunk_tiles * te::TILE);
    if (d_meas) CK(cudaMemcpyAsync(d_meas + s0 * meas_stride, meas + s0 * meas_stride, (size_t)(s1 - s0) * meas_stride * 8, cudaMemcpyHostToDevice, p->h2d_stream));
    if (d_act) CK(cudaMemcpyAsync(d_act + s0, action + s0, (size_t)(s1 - s0), cudaMemcpyHostToDevice, p->h2d_stream));
    CK(cudaEventRecord(ts.ev[2 * c], p->h2d_stream));
    CK(cudaStreamWaitEvent(p->stream, ts.ev[2 * c], 0));
    a.tile_begin = c * chunk_tiles;
    a.n_tiles = std::min(chunk_tiles, n_tiles - c * chunk_tiles);
    launch_step(p, a, a.n_tiles);
    if (d_pos) {
      CK(cudaEventRecord(ts.ev[2 * c + 1], p->stream));
      CK(cudaStreamWaitEvent(p->d2h_stream, ts.ev[2 * c + 1], 0));
      CK(cudaMemcpyAsync(est_pos_out + s0 * 3, d_pos + s0 * 3, (size_t)(s1 - s0) * 24, cudaMemcpyDeviceToHost, p->d2h_stream));
    }
  }
  if (d_meas && meas_stride == 7) {   // measured_pose_ = meas for the updated slots (src/target_interface.cpp:142-146)
    if (d_act) te::copy_meas_masked_kernel<<<cdiv(n, 256), 256, 0, p->stream>>>(p->buf[p->cur].cold.meas, d_meas, d_act, (int)n);
    else if (default_action == TE_ACT_UPDATE)
      CK(cudaMemcpyAsync(p->buf[p->cur].cold.meas, d_meas, (size_t)n * 56, cudaMemcpyDeviceToDevice, p->stream));
    CK(cudaGetLastError());
  }
  // the tick has left this set when its kernels AND its read-backs are done
  CK(cudaEventRecord(ts.step_done, p->stream));
  CK(cudaStreamWaitEvent(p->d2h_stream, ts.step_done, 0));
  CK(cudaEventRecord(ts.d2h_done, p->d2h_stream));
  ts.busy = true;
  ++p->ticks_issued;
}

void tick_host_wait(te_pool* p, int lag) {
  // ticks are numbered by issue; tick i used set i % TICK_SETS.  lag 0: everything done; lag k: all but the newest k ticks done
  for (int back = te_pool::TICK_SETS - 1; back >= 0; --back) {
    if (back < lag) continue;
    const long long i = p->ticks_issued - 1 - back;
    if (i < 0) continue;
    te_pool::TickSet& ts = p->tick_set[i % te_pool::TICK_SETS];
    if (ts.busy) {
      CK(cudaEventSynchronize(ts.d2h_done));
      ts.busy = false;
    }
  }
}

}  // namespace

int te_pool_tick_host(te_pool* p, double dt, const double* meas, int meas_stride, const uint8_t* action, int default_action,
                      double* est_pos_out) {
  return guarded(p, [&] {
    if (p->n == 0) return 0;
    tick_host_enqueue(p, dt, meas, meas_stride, action, default_action, est_pos_out, false);
    tick_host_wait(p, 0);
    return 0;
  });
}

int te_pool_tick_host_async(te_pool* p, double dt, const double* meas, int meas_stride, const uint8_t* action, int default_action,
                            double* est_pos_out) {
  return guarded(p, [&] {
    if (p->n == 0) return 0;
    tick_host_enqueue(p, dt, meas, meas_stride, action, default_action, est_pos_out, true);
    return 0;
  });
}

int te_pool_tick_host_wait(te_pool* p, int lag) {
  return guarded(p, [&] {
    if (lag < 0 || lag >= te_pool::TICK_SETS) throw std::invalid_argument("lag must be 0, 1 or 2");
    tick_host_wait(p, lag);
    return 0;
  });
}

}  // extern "C"

namespace tehost {
long long step_ops(te_pool* p, long long n, const uint32_t* d_ids, const double* d_dt, double dt_scalar, const double* d_meas,
                   const uint8_t* d_act) {
  ensure_work(p, (size_t)p->n);
  Buf& b = p->buf[p->cur];
  CK(cudaMemsetAsync(p->d_counters, 0, 3 * sizeof(int), p->stream));
  CK(cudaMemsetAsync(p->alive, 0, (size_t)p->n * sizeof(int), p->stream));   // per-slot claim counts of this call (alive[] is scratch between compactions)
  te::scatter_ops_kernel<<<cdiv(n, 256), 256, 0, p->stream>>>(b.cold.ids, (int)p->n, n, d_ids, d_dt, dt_scalar, d_meas, d_act, p->action,
                                                               p->dt_slot, b.cold.meas, p->tile_flag, p->tile_list, p->d_counters, p->alive);
  CK(cudaGetLastError());
  if (n > 1) {   // a repeated id?  (checked before anything is stepped)
    int dups = 0;
    CK(cudaMemcpyAsync(&dups, p->d_counters + 2, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    if (dups > 0) {
      CK(cudaMemsetAsync(p->action, 0, (size_t)p->n, p->stream));
      CK(cudaMemsetAsync(p->tile_flag, 0, (size_t)cdiv(p->n, te::TILE) + 4, p->stream));
      CK(cudaStreamSynchronize(p->stream));
      last_error() = "an id appears more than once in the batch: nothing applied";
      return -2;
    }
  }
  te::StepArgs a = base_args(p);
  a.tile_list = p->tile_list;
  a.d_nwork = p->d_counters;
  a.dt = dt_scalar;
  a.dt_slot = p->dt_slot;
  a.meas = b.cold.meas;
  a.meas_stride = 7;
  a.meas_tma = 1;
  a.action = p->action;
  a.default_action = TE_ACT_NONE;
  a.clear_action = 1;
  a.tile_flag = p->tile_flag;
  launch_step(p, a, (int)std::min<long long>(n, a.n_tiles));
  int applied = 0;
  CK(cudaMemcpyAsync(&applied, p->d_counters + 1, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
  CK(cudaStreamSynchronize(p->stream));
  return applied;
}
}  // namespace tehost

extern "C" {

long long te_pool_step_ids(te_pool* p, long long n, const uint32_t* ids, const double* dt, double dt_scalar, const double* meas,
                           const uint8_t* action) {
  return guarded_ll(p, [&]() -> long long {
    if (n <= 0 || p->n == 0) return 0;
    if (!ids) throw std::invalid_argument("null ids");
    if (!dt && !(dt_scalar >= 0.0)) throw std::invalid_argument("dt must be >= 0");
    uint32_t* d_ids = to_dev(p, ids, n);
    double* d_dt = to_dev(p, dt, n);
    double* d_meas = to_dev(p, meas, n * 7);
    uint8_t* d_act = to_dev(p, action, n);
    if (!meas) {
      bool needs = !action;
      if (action) for (long long k = 0; k < n && !needs; ++k) needs = action[k] == TE_ACT_UPDATE;
      if (needs) throw std::invalid_argument("update ops without measurements");
    }
    return step_ops(p, n, d_ids, d_dt, dt_scalar, d_meas, d_act);
  });
}

int te_pool_predict_all(te_pool* p, double dt) { return te_pool_step_dense(p, dt, nullptr, 7, nullptr, TE_ACT_PREDICT); }

long long te_pool_step_dense_expire(te_pool* p, double dt, const double* dev_meas, int meas_stride, const uint8_t* dev_action,
                                    int default_action, uint32_t stamp_sec, uint32_t stamp_nsec, uint32_t now_sec, uint32_t now_nsec,
                                    double timeout, uint32_t* erased_out, long long cap) {
  return guarded_ll(p, [&]() -> long long {
    if (p->n == 0) return 0;
    if (p->mb_on) throw std::logic_error("this pool keeps device mailboxes: its ticks go through te_pool_mailbox_tick");
    if (!(dt >= 0.0)) throw std::invalid_argument("dt must be >= 0 (assert of src/target_interface.cpp:150)");
    if (dev_meas) check_meas_stride(p, meas_stride);
    else if (dev_action || default_action == TE_ACT_UPDATE) throw std::invalid_argument("update tick without measurements");
    const int n_old = (int)p->n;
    ensure_work(p, (size_t)n_old);
    Buf& ob = p->buf[p->cur];
    // 1. this tick's stamps, then the expiry predicate (both as in te_pool_stamp_dense / te_pool_expire)
    volatile double sns = 1e-9 * (double)stamp_nsec;
    const double stamp = (double)stamp_sec + sns;
    volatile double nns = 1e-9 * (double)now_nsec;
    const double now = (double)now_sec + nns;
    te::stamp_dense_kernel<<<cdiv(n_old, 256), 256, 0, p->stream>>>(dev_action, default_action, n_old, stamp, ob.cold.last_meas);
    CK(cudaGetLastError());
    te::expire_flags_kernel<<<cdiv(n_old, 256), 256, 0, p->stream>>>(ob.cold.last_meas, n_old, now, timeout, p->alive);
    CK(cudaGetLastError());
    size_t tmp = p->cub_bytes;
    CK(cub::DeviceScan::ExclusiveSum(p->cub_tmp, tmp, p->alive, p->pos, n_old, p->stream));
    int last_pos = 0, last_alive = 0;
    CK(cudaMemcpyAsync(&last_pos, p->pos + n_old - 1, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaMemcpyAsync(&last_alive, p->alive + n_old - 1, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    const int n_alive = last_pos + last_alive;
    const long long n_er = n_old - n_alive;
    // 2. the step: in place when nobody expired, else into the compacted slots of the other buffer
    te::StepArgs a = base_args(p);
    a.dt = dt;
    a.meas = dev_meas;
    a.meas_stride = meas_stride;
    a.meas_tma = (dev_meas && (uintptr_t)dev_meas % 16 == 0) ? 1 : 0;
    a.action = const_cast<uint8_t*>(dev_action);
    a.default_action = default_action;
    if (n_er == 0) {
      launch_step(p, a, a.n_tiles);
      return 0;
    }
    uint32_t* d_erased = p->arena.get_n<uint32_t>((size_t)n_er);
    te::collect_erased_kernel<<<cdiv(n_old, 256), 256, 0, p->stream>>>(p->alive, p->pos, ob.cold.ids, n_old, d_erased);
    CK(cudaGetLastError());
    if (n_alive > 0) {
      ensure_other_capacity(p, (size_t)n_alive);
      Buf& nb = p->buf[1 - p->cur];
      te::compact_cold_kernel<<<cdiv(n_old, 256), 256, 0, p->stream>>>(n_old, p->alive, p->pos, p->buf[p->cur].cold, nb.cold);
      CK(cudaGetLastError());
      a.dst_tiles = nb.tiles;
      a.dst_alive = p->alive;
      a.dst_pos = p->pos;
      launch_step(p, a, a.n_tiles);
    }
    p->cur = 1 - p->cur;
    p->n = n_alive;
    p->h_ids_valid = false;
    fetch_last_id(p);
    if (erased_out && cap > 0)
      CK(cudaMemcpyAsync(erased_out, d_erased, (size_t)std::min(cap, n_er) * sizeof(uint32_t), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    return n_er;
  });
}
}  // extern "C"


#ifdef TE_TIMELINE
// debug build only (tools/timeline.py): phase timestamps of CTA 0 recorded by kf_step_split_kernel
extern "C" int te_debug_timeline(long long* out) {
  return (int)cudaMemcpyFromSymbol(out, te::g_timeline, sizeof(long long) * 2 * 64 * 12);
}
#endif