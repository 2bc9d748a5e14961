// te_pool_internal.cuh -- what the translation units of libte_pool.so share: the pool object, its scratch arena, the error
// channel, and the host helpers each unit calls in the others.  Not installed; the public surface is include/te_pool.h.
//   te_pool.cu     lifecycle, model classes, add / erase (stream compaction), read-back, expiry
//   te_step.cu     step-kernel launch policy and the stepping entry points (dense / replay / host / by id / fused expiry)
//   te_mailbox.cu  device-resident mailboxes (the node loop)
//   te_isolver.cu  batched IntersectionSolver
//   te_sweep.cu    the k earliest sphere intercepts, the k nearest targets and the k gated targets over every target of a pool
//                  (te_pool_earliest_intersections, te_pool_nearest_targets, te_pool_gated_targets)
//   te_assoc.cu    association of unlabelled detections: grid-indexed gate candidates, device greedy matching, update at t1
//                  (te_pool_associate, te_pool_gated_candidates, te_assign_greedy, te_pool_update_at)
//   te_group.cu    several pools on several devices: the NCCL all-gather of estimate records
#pragma once
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <numeric>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/te_pool.h"
#include "te_kernels.cuh"

namespace tehost {

std::string& last_error();   // thread-local message behind te_last_error()

struct CudaError : std::runtime_error {
  using std::runtime_error::runtime_error;
};
#define CK(call)                                                                                       \
  do {                                                                                                 \
    cudaError_t e__ = (call);                                                                          \
    if (e__ != cudaSuccess)                                                                            \
      throw CudaError(std::string(#call) + ": " + cudaGetErrorString(e__) + " (" __FILE__ ":" + std::to_string(__LINE__) + ")"); \
  } while (0)

inline int cdiv(long long a, int b) { return (int)((a + b - 1) / b); }

// grow-only device scratch, bump-allocated per call: one main block sized by the previous call's demand,
// overflow goes to one-off blocks that are folded into the main block at the next reset
struct Arena {
  char* main = nullptr;
  size_t main_cap = 0, off = 0, want = 0;
  std::vector<void*> extra;
  void reset() {
    for (void* c : extra) cudaFree(c);
    extra.clear();
    if (want > main_cap) {
      cudaFree(main);
      main = nullptr;
      main_cap = 0;
      const size_t cap = want + want / 2;
      CK(cudaMalloc((void**)&main, cap));
      main_cap = cap;
    }
    off = 0;
    want = 0;
  }
  void* get(size_t bytes) {
    bytes = (bytes + 255) & ~(size_t)255;
    if (bytes == 0) bytes = 256;
    want += bytes;
    if (off + bytes <= main_cap) {
      void* p = main + off;
      off += bytes;
      return p;
    }
    void* p = nullptr;
    CK(cudaMalloc(&p, bytes));
    extra.push_back(p);
    return p;
  }
  template <class T> T* get_n(size_t n) { return (T*)get(n * sizeof(T)); }
  void destroy() {
    for (void* c : extra) cudaFree(c);
    extra.clear();
    cudaFree(main);
    main = nullptr;
    main_cap = 0;
  }
};

struct Buf {   // one generation of the pool's per-slot storage
  double* tiles = nullptr;
  te::ColdArrays cold{nullptr, nullptr, nullptr, nullptr};
  size_t cap = 0;   // slots (multiple of 32)
};

struct MailBuf {   // one generation of the per-slot mailboxes (te_pool_mailbox_*)
  te::MailArrays a{nullptr, nullptr, nullptr, nullptr};
  size_t cap = 0;
};

// A mailbox whose id has no target yet (Measurement of target_manager_ros.hpp:74-134 on the host): the message carried a
// stamp that is not newer than the initial one, or a newer record was followed by an older one before the tick.  Rare, so
// these stay in a host map; the tick promotes the readable ones to targets and expires the others by the same predicate.
struct HostMail {
  uint32_t sec = 0, nsec = 0;
  double last = 0.0;
  bool fresh = true;   // Measurement(): new_meas_ = true
  double pose[7] = {0, 0, 0, 0, 0, 0, 0};
};
inline double host_to_sec(uint32_t sec, uint32_t nsec) {   // utils.hpp:59-62, never contracted
  volatile double ns = 1e-9 * (double)nsec;
  return (double)sec + ns;
}
// a /tf record whose id has no target: kept in arrival order until the next tick folds it into a mailbox (the common case --
// an id seen for the first time, promoted by that tick -- then never touches the std::map)
struct PendingRec {
  uint32_t id, sec, nsec;
  double pose[7];
};
inline void apply_record(HostMail& m, const PendingRec& r) {   // Measurement::update (target_manager_ros.hpp:96-115)
  const double cur = host_to_sec(r.sec, r.nsec), prev = host_to_sec(m.sec, m.nsec);
  if (cur > prev) { m.fresh = true; m.last = cur; }
  else m.fresh = false;
  m.sec = r.sec;
  m.nsec = r.nsec;
  std::memcpy(m.pose, r.pose, sizeof(m.pose));
}


}  // namespace tehost

struct te_pool {
  int model = 0, device = 0;
  int N = 0, M = 0, NF = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int n_sm = 148;
  int variant = 0;
  int grid_cap = 0;      // test hook (te_pool_set_grid_cap): upper bound on the CTAs of a step launch, 0 = none
  bool all_sym = true;   // every registered class has bitwise-symmetric Q, R, P0 (symmetric-covariance kernels are legal)
  // UV / UA: no registered class couples the x / y / z axes (Q, P0 zero between axes, R diagonal), so every cross-axis covariance
  // entry in HBM stays +-0 and the packed direct kernels move the per-axis blocks only (te_kin_sym.cuh AXIS).  Always false for
  // AV / AR.  Like all_sym, it only ever goes from true to false.
  bool all_axis = true;
  // The direct symmetric kernels maintain the UPPER triangle of every covariance only ("packed": 36 of UA's 92 fields are
  // neither read nor written per step).  lower_stale = the lower triangles in HBM are out of date; whoever needs the full
  // matrix (a full-matrix kernel, a state read-back) mirrors it first / on the fly.
  bool lower_stale = false;
  long long n = 0;   // live targets
  long long assoc_stats[4] = {0, 0, 0, 0};   // te_pool_assoc_stats: of the last association call
  tehost::Buf buf[2];
  int cur = 0;
  // per-slot work arrays (capacity wcap slots)
  size_t wcap = 0;
  uint8_t* action = nullptr;
  double* dt_slot = nullptr;
  uint8_t* tile_flag = nullptr;
  int* tile_list = nullptr;
  int* alive = nullptr;
  int* pos = nullptr;
  int* srcmap = nullptr;
  int* d_counters = nullptr;   // [0] = n_work, [1] = applied
  void* cub_tmp = nullptr;
  size_t cub_bytes = 0;
  // model classes
  std::vector<std::vector<double>> hQ, hR, hP0;
  double *dQ = nullptr, *dR = nullptr, *dP0 = nullptr;
  // per class: T = L^-1 with R = L L^T (lower triangular, row-major M x M): the whitening of the measurement that lets a kernel apply
  // an update as M scalar updates (te_av_sym.cuh av_update_seq).  whiten_ok = every class's R has a Cholesky factor.
  double* dT = nullptr;
  std::vector<std::vector<double>> hT;
  bool whiten_ok = true;
  int cls_cap = 0;
  // host mirror of the sorted ids (lazy)
  std::vector<uint32_t> h_ids;
  bool h_ids_valid = true;
  // largest live id, kept across compactions: enough to recognise an append-only add batch (monotonically increasing
  // track ids, the common case) without downloading the whole id array again
  uint32_t h_last_id = 0;
  bool h_last_valid = false;
  tehost::Arena arena;
  // device-resident mailboxes (te_pool_mailbox_*): allocated on first use, then carried through every compaction
  bool mb_on = false;
  tehost::MailBuf mb[2];
  int mb_cur = 0;
  te::MailAdd mb_add{nullptr, nullptr, nullptr};   // set by the mailbox tick around its merge
  std::map<uint32_t, tehost::HostMail> orphans;            // mailboxes without a target that outlived a tick (unreadable ones)
  std::vector<tehost::PendingRec> pending;                 // records of unknown ids since the last tick, arrival order
  char* h_stage = nullptr;                         // pinned staging for the tick's add arrays / the ingest's read-backs (grow-only)
  size_t h_stage_cap = 0;
  // chunk pipeline of te_pool_tick_host / te_pool_tick_host_async: TICK_SETS sets of device staging (measurements, actions,
  // positions) so that the copies of tick k + 1 run under the kernels of tick k and the read-back of tick k - 1.  Three, not two:
  // a tick is in flight for copy-in + kernel + copy-out (2.1 + 0.6 + 2.0 ms at 4 Mi UA targets), and with two sets the copy-in of
  // tick k + 1 waits for the read-back of tick k - 1 to leave its set -- the link idles a tenth of the time (2.37 ms per tick by
  // that arithmetic, 2.48 measured); with three the copy-in engine never waits
  cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
  struct TickSet {
    double* meas = nullptr;
    uint8_t* act = nullptr;
    double* pos = nullptr;
    size_t meas_cap = 0, act_cap = 0, pos_cap = 0;   // bytes
    std::vector<cudaEvent_t> ev;                     // [2 * chunk] h2d done, [2 * chunk + 1] step done
    cudaEvent_t step_done = nullptr, d2h_done = nullptr;
    bool busy = false;
  } tick_set[3];
  static constexpr int TICK_SETS = 3;
  long long ticks_issued = 0;
  // live launch (te_pool_live_*): one resident replay launch whose ticks are released one by one
  struct Live {
    bool active = false;
    int max_ticks = 0, released = 0, stride = 0;
    int* d_gate = nullptr;      // [0] released ticks (copy engine), [1] stop, [2] / [3] the gate every warp watches, [4 ..] done counts per tick
    size_t d_cap = 0;           // ints
    int* h_ring = nullptr;      // page-locked, mapped: staging of the pushed gate writes [0 .. 255], done flag (kernel writes) [256], host gate [257], host stop [258]
    double* d_meas = nullptr;   // the caller's rings
    uint8_t* d_action = nullptr;
  } live;
  // a /tf message on its way to the device under the running tick (te_pool_mailbox_prefetch)
  struct Prefetch {
    char* dev = nullptr;
    size_t cap = 0;
    long long n = 0;
    const uint32_t *ids = nullptr, *sec = nullptr, *nsec = nullptr;
    const double* poses = nullptr;
    cudaEvent_t keys_done = nullptr, done = nullptr;   // ids / stamps on the device; everything on the device
    bool pending = false;   // a message is registered
    bool started = false;   // its copies are in the copy stream's queue
  } prefetch;
};

struct te_isolver {
  te_pool* pool = nullptr;
  te::IsolverState st{};
  // te_isolver_move_streams: the packed streams and their indices on this solver's device (grow-only)
  double* move_block = nullptr;
  int* move_streams = nullptr;
  size_t move_cap = 0;   // streams
  unsigned long long* d_found = nullptr;   // te_isolver_query's count of existing ids
};

namespace tehost {

struct DeviceGuard {
  int prev = 0;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) CK(cudaSetDevice(dev));
  }
  ~DeviceGuard() { cudaSetDevice(prev); }
};

// ---- te_pool.cu ----
size_t tile_doubles(const te_pool* p);
void free_buf(Buf& b);
void alloc_buf(te_pool* p, Buf& b, size_t slots);
void ensure_work(te_pool* p, size_t slots);
void ensure_cur_capacity(te_pool* p, size_t slots);
void ensure_other_capacity(te_pool* p, size_t slots);
char* pinned_stage(te_pool* p, size_t bytes);
void free_mail(MailBuf& m);
void alloc_mail(MailBuf& m, size_t slots);
void ensure_mail_cur(te_pool* p, size_t slots);
void ensure_mail_other(te_pool* p, size_t slots);
void enable_mail(te_pool* p);
void sync_host_ids(te_pool* p);
void upload_classes(te_pool* p);
void rebuild(te_pool* p, int n_new, const te::AddData& ad);
void init_append(te_pool* p, int base, const te::AddData& ad, long long n);
void init_promoted(te_pool* p, int n_add, const int* new_dst, const Buf& nb, const te::AddData& ad, const te::MailArrays& mb);
void fetch_last_id(te_pool* p);
int compact_and_merge(te_pool* p, const te::AddData& ad, const uint32_t* d_add_ids, int n_add, uint32_t* d_erased /*or null*/);
int* lookup_slots(te_pool* p, const uint32_t* d_ids, long long n);
// gather_estimates_kernel on the pool's stream: query k reads slot slots[k] (slots NULL = slot k), at d_t1[k] (NULL = now)
void launch_gather_estimates(te_pool* p, const int* slots, long long n, const double* d_t1, double* pose, double* twist, double* acc,
                             double* pose6, uint8_t* found, int rec13);
void fold_pending(te_pool* p);
void demote_mailboxes(te_pool* p, const uint32_t* ids, const int* d_slots, long long n);
void attach_mailboxes(te_pool* p, const uint32_t* ids, long long n);
// ---- te_sweep.cu ----
// gate_prep_kernel of the pool's model over every slot: the factor of S into chol[6 * slot]; t1 NULL = no predict
void launch_gate_prep(te_pool* p, int n, const double* t1, double* chol);
// ---- te_mailbox.cu ----
void prefetch_start(te_pool* p);   // put the registered message's copies into the copy stream's queue (no-op if none / started)
// ---- te_step.cu ----
bool uses_direct(const te_pool* p);
void ensure_full(te_pool* p);
void launch_step(te_pool* p, const te::StepArgs& a_in, int n_work_hint);
void launch_step_multi(te_pool* p, const te::StepArgs& a_in, int n_work_hint);
te::StepArgs base_args(te_pool* p);
void check_meas_stride(te_pool* p, int stride);
// te_pool_step_ids over device arrays (d_dt NULL = dt_scalar, d_meas NULL only without UPDATE ops, d_act NULL = UPDATE): the scatter,
// the duplicate check (-2, nothing applied) and the step launch.  Returns #applied.
long long step_ops(te_pool* p, long long n, const uint32_t* d_ids, const double* d_dt, double dt_scalar, const double* d_meas,
                   const uint8_t* d_act);

template <class T> T* to_dev(te_pool* p, const T* host, size_t n) {
  if (!host || !n) return nullptr;
  T* d = p->arena.get_n<T>(n);
  CK(cudaMemcpyAsync(d, host, n * sizeof(T), cudaMemcpyHostToDevice, p->stream));
  return d;
}

// ---- step kernel launch -----------------------------------------------------------------

inline bool& live_call() {   // set by the te_pool_live_* entry points: every other call is refused while a live launch holds the pool
  static thread_local bool f = false;
  return f;
}
template <class F> int guarded(te_pool* p, F&& f) {
  try {
    if (!p) throw std::invalid_argument("null pool");
    if (p->live.active && !live_call()) throw std::logic_error("the pool is held by a live launch: call te_pool_live_end first");
    DeviceGuard g(p->device);
    p->arena.reset();
    return f();
  } catch (const std::exception& e) {
    last_error() = e.what();
    return -1;
  }
}
template <class F> long long guarded_ll(te_pool* p, F&& f) {
  try {
    if (!p) throw std::invalid_argument("null pool");
    if (p->live.active && !live_call()) throw std::logic_error("the pool is held by a live launch: call te_pool_live_end first");
    DeviceGuard g(p->device);
    p->arena.reset();
    return f();
  } catch (const std::exception& e) {
    last_error() = e.what();
    return -1;
  }
}

}  // namespace tehost
