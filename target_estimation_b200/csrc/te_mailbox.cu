// te_mailbox.cu -- device-resident mailboxes: measurementCallBack + update(dt) of RosTargetManager
// (/root/reference/src/target_manager_ros.cpp:26-92, include/target_estimation/target_manager_ros.hpp:74-134) for pools too large
// for a host loop.  Entry points: te_pool_mailbox_* of include/te_pool.h.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "te_pool_internal.cuh"

using namespace tehost;
#define g_err (tehost::last_error())

// ---- device-resident mailboxes: measurementCallBack + update(dt) of RosTargetManager ----------------
namespace {
// one /tf message into the mailboxes.  Host source (ids .. poses non-null): the arrays are staged here; device source (d_* given,
// host pointers null): the records are used in place and the few records of unknown ids are read back for the host's queue.
int mailbox_ingest_impl(te_pool* p, long long n, const uint32_t* ids, const uint32_t* sec, const uint32_t* nsec, const double* poses,
                        const uint32_t* d_ids, const uint32_t* d_sec, const uint32_t* d_nsec, const double* d_pose,
                        cudaEvent_t payload_ready = nullptr /* d_sec / d_nsec / d_pose are complete once this event has fired */) {
  if (n <= 0) return 0;
  if (n > 0x7FFFFFFF) throw std::invalid_argument("too many records in one message");
  const bool host_src = ids != nullptr;
  enable_mail(p);
  const int nr = (int)n;
  static const bool dbg = std::getenv("TE_MB_DEBUG") != nullptr;   // phase times of the call on stderr (each mark synchronises: debugging only)
  auto wall = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  double tw[5] = {0, 0, 0, 0, 0};
  auto mark = [&](int i, bool sync) { if (dbg) { if (sync) cudaStreamSynchronize(p->stream); tw[i] = wall(); } };
  mark(0, true);
  auto queue = [&](uint32_t id, uint32_t s, uint32_t ns, const double* pose) {   // unknown id: queued in arrival order for the next tick
    PendingRec r;
    r.id = id;
    r.sec = s;
    r.nsec = ns;
    std::memcpy(r.pose, pose, sizeof(r.pose));
    p->pending.push_back(r);
  };
  if (p->n == 0 && host_src) {   // no targets yet: every record belongs to a target-less mailbox
    for (long long k = 0; k < n; ++k) queue(ids[k], sec[k], nsec[k], poses + 7 * k);
    return 0;
  }
  if (host_src && !d_ids) {
    d_ids = to_dev(p, ids, (size_t)n);
    d_sec = to_dev(p, sec, (size_t)n);
    d_nsec = to_dev(p, nsec, (size_t)n);
    d_pose = to_dev(p, poses, (size_t)n * 7);
  }
  uint32_t* key_in = p->arena.get_n<uint32_t>((size_t)n);
  uint32_t* key_out = p->arena.get_n<uint32_t>((size_t)n);
  int* rec_in = p->arena.get_n<int>((size_t)n);
  int* rec_out = p->arena.get_n<int>((size_t)n);
  int* unknown = p->arena.get_n<int>((size_t)n);
  int* counter = p->arena.get_n<int>(1);
  CK(cudaMemsetAsync(counter, 0, sizeof(int), p->stream));
  Buf& b = p->buf[p->cur];
  te::mb_lookup_kernel<<<cdiv(n, 256), 256, 0, p->stream>>>(b.cold.ids, (int)p->n, d_ids, nr, key_in, rec_in, unknown, counter);
  CK(cudaGetLastError());
  if (p->n > 0) {
    // stable sort by slot: the records of one id stay in arrival order (a message may name an id more than once, and several
    // messages may be ingested between two ticks)
    int bits = 1;
    while (bits < 32 && (1ll << bits) <= p->n) ++bits;   // keys are slots < n, or n for unknown ids: 2^bits > n
    size_t tmp_bytes = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, key_in, key_out, rec_in, rec_out, nr, 0, bits, p->stream));
    void* tmp = p->arena.get(tmp_bytes);
    CK(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, key_in, key_out, rec_in, rec_out, nr, 0, bits, p->stream));
    mark(1, true);
    if (payload_ready) CK(cudaStreamWaitEvent(p->stream, payload_ready, 0));   // lookup and sort ran under the tail of the copy
    mark(2, true);
    te::mb_apply_kernel<<<cdiv(n, 256), 256, 0, p->stream>>>(nr, (int)p->n, key_out, rec_out, d_sec, d_nsec, d_pose, p->mb[p->mb_cur].a, b.cold.last_meas);
    CK(cudaGetLastError());
  }
  int n_unknown = 0;
  // Host source with targets in the pool: the stable sort has left the records of unknown ids (key = n, the largest) at the END of
  // rec_out, in arrival order -- the count and the last TAIL entries come back in one pinned read (a second one only when more
  // ids are unknown than that), and nothing is sorted on the host (std::sort of the 10 k first-sight records of a 1 Mi-target
  // message cost 0.2 ms of every ingest).
  constexpr int TAIL = 16384;
  const int tail_n = (host_src && p->n > 0) ? std::min(nr, TAIL) : 0;
  int* h_tail = nullptr;
  if (tail_n > 0) {
    h_tail = reinterpret_cast<int*>(pinned_stage(p, (size_t)(TAIL + 1) * sizeof(int)));
    CK(cudaMemcpyAsync(h_tail, counter, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaMemcpyAsync(h_tail + 1, rec_out + (nr - tail_n), (size_t)tail_n * sizeof(int), cudaMemcpyDeviceToHost, p->stream));
  } else {
    CK(cudaMemcpyAsync(&n_unknown, counter, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
  }
  CK(cudaStreamSynchronize(p->stream));   // also: a host caller's record arrays are free again
  if (tail_n > 0) n_unknown = h_tail[0];
  mark(3, false);
  if (n_unknown == 0) return 0;
  if (host_src) {
    p->pending.reserve(p->pending.size() + (size_t)n_unknown);
    if (tail_n > 0 && n_unknown <= tail_n) {
      const int* list = h_tail + 1 + (tail_n - n_unknown);
      for (int i = 0; i < n_unknown; ++i) {
        const int k = list[i];
        queue(ids[k], sec[k], nsec[k], poses + 7 * (size_t)k);
      }
    } else {
      std::vector<int> list((size_t)n_unknown);
      if (tail_n > 0) {   // more unknown ids than the tail read: the whole run, still in arrival order
        CK(cudaMemcpy(list.data(), rec_out + (nr - n_unknown), (size_t)n_unknown * sizeof(int), cudaMemcpyDeviceToHost));
      } else {
        CK(cudaMemcpy(list.data(), unknown, (size_t)n_unknown * sizeof(int), cudaMemcpyDeviceToHost));
        std::sort(list.begin(), list.end());   // arrival order
      }
      for (int k : list) queue(ids[k], sec[k], nsec[k], poses + 7 * (size_t)k);
    }
    mark(4, false);
    if (dbg) std::fprintf(stderr, "[te mailbox ingest] lookup + sort %.3f ms, wait for the payload %.3f ms, apply %.3f ms, unknown ids to the host queue %.3f ms (%d)\n",
                          tw[1] - tw[0], tw[2] - tw[1], tw[3] - tw[2], tw[4] - tw[3], n_unknown);
    return 0;
  }
  // device source: pack the unknown records into one block [pose 7 | index | id | sec | nsec] x n_unknown, read it back in one copy
  // to pinned memory, queue the records in arrival order.  With targets in the pool the stable sort has left the unknown records at
  // the end of rec_out in arrival order already; otherwise the lookup's list is in completion order and is sorted here
  const size_t nu = (size_t)n_unknown;
  const int* list = p->n > 0 ? rec_out + (nr - n_unknown) : unknown;
  char* d_blk = (char*)p->arena.get(nu * 72);
  double* o_pose = (double*)d_blk;
  int* o_idx = (int*)(o_pose + 7 * nu);
  uint32_t* o_ids = (uint32_t*)(o_idx + nu);
  uint32_t* o_sec = o_ids + nu;
  uint32_t* o_nsec = o_sec + nu;
  te::mb_pack_unknown_kernel<<<cdiv(n_unknown, 256), 256, 0, p->stream>>>(n_unknown, list, d_ids, d_sec, d_nsec, d_pose, o_ids, o_sec, o_nsec, o_pose);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(o_idx, list, nu * sizeof(int), cudaMemcpyDeviceToDevice, p->stream));
  char* h_blk = pinned_stage(p, nu * 72);
  CK(cudaMemcpyAsync(h_blk, d_blk, nu * 72, cudaMemcpyDeviceToHost, p->stream));
  CK(cudaStreamSynchronize(p->stream));
  const double* h_pose = (const double*)h_blk;
  const int* h_idx = (const int*)(h_pose + 7 * nu);
  const uint32_t* h_ids = (const uint32_t*)(h_idx + nu);
  const uint32_t* h_sec = h_ids + nu;
  const uint32_t* h_nsec = h_sec + nu;
  bool in_order = true;
  for (size_t k = 1; k < nu && in_order; ++k) in_order = h_idx[k - 1] < h_idx[k];
  if (in_order) {
    for (size_t k = 0; k < nu; ++k) queue(h_ids[k], h_sec[k], h_nsec[k], h_pose + 7 * k);
  } else {
    std::vector<int> order(nu);
    std::iota(order.begin(), order.end(), 0);
    std::sort(order.begin(), order.end(), [&](int a, int c) { return h_idx[a] < h_idx[c]; });
    for (int k : order) queue(h_ids[(size_t)k], h_sec[(size_t)k], h_nsec[(size_t)k], h_pose + 7 * (size_t)k);
  }
  return 0;
}
}  // namespace

namespace tehost {
void prefetch_start(te_pool* p) {
  te_pool::Prefetch& pf = p->prefetch;
  if (!pf.pending || pf.started) return;
  pf.started = true;
  if (!p->h2d_stream) {
    CK(cudaStreamCreateWithFlags(&p->h2d_stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&p->d2h_stream, cudaStreamNonBlocking));
  }
  if (!pf.done) {
    CK(cudaEventCreateWithFlags(&pf.done, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&pf.keys_done, cudaEventDisableTiming));
  }
  const size_t nn = (size_t)pf.n, need = nn * 68 + 1024;
  if (need > pf.cap) {   // (the previous message's consumers ran on the pool's stream)
    CK(cudaStreamSynchronize(p->stream));
    cudaFree(pf.dev);
    pf.dev = nullptr;
    pf.cap = 0;
    const size_t cap = need + need / 8;
    CK(cudaMalloc((void**)&pf.dev, cap));
    pf.cap = cap;
  } else {
    // the kernels that read the previous message out of this staging must be done before the copies overwrite it
    CK(cudaEventRecord(pf.done, p->stream));
    CK(cudaStreamWaitEvent(p->h2d_stream, pf.done, 0));
  }
  if (nn > 0) {
    // ids and stamps first: the lookup and the sort of the records need nothing else and run under the copy of the poses
    uint32_t* d_ids = (uint32_t*)pf.dev;
    double* d_pose = (double*)(pf.dev + ((nn * 12 + 255) & ~(size_t)255));
    CK(cudaMemcpyAsync(d_ids, pf.ids, nn * 4, cudaMemcpyHostToDevice, p->h2d_stream));
    CK(cudaEventRecord(pf.keys_done, p->h2d_stream));
    CK(cudaMemcpyAsync(d_ids + nn, pf.sec, nn * 4, cudaMemcpyHostToDevice, p->h2d_stream));
    CK(cudaMemcpyAsync(d_ids + 2 * nn, pf.nsec, nn * 4, cudaMemcpyHostToDevice, p->h2d_stream));
    CK(cudaMemcpyAsync(d_pose, pf.poses, nn * 56, cudaMemcpyHostToDevice, p->h2d_stream));
  } else {
    CK(cudaEventRecord(pf.keys_done, p->h2d_stream));
  }
  CK(cudaEventRecord(pf.done, p->h2d_stream));
}
}  // namespace tehost

extern "C" {

int te_pool_mailbox_ingest(te_pool* p, long long n, const uint32_t* ids, const uint32_t* sec, const uint32_t* nsec, const double* poses) {
  return guarded(p, [&] {
    if (n <= 0) return 0;
    if (!ids || !sec || !nsec || !poses) throw std::invalid_argument("null record arrays");
    return mailbox_ingest_impl(p, n, ids, sec, nsec, poses, nullptr, nullptr, nullptr, nullptr);
  });
}

/* the message is registered; its copies go into the copy stream's queue when the next tick has queued its own small uploads (or at
   te_pool_mailbox_ingest_prefetched, whichever comes first) and run under whatever the pool's stream is doing */
int te_pool_mailbox_prefetch(te_pool* p, long long n, const uint32_t* ids, const uint32_t* sec, const uint32_t* nsec, const double* poses) {
  return guarded(p, [&] {
    te_pool::Prefetch& pf = p->prefetch;
    if (pf.pending) throw std::logic_error("a prefetched message is waiting: call te_pool_mailbox_ingest_prefetched first");
    if (n < 0 || n > 0x7FFFFFFF) throw std::invalid_argument("bad record count");
    if (n > 0 && (!ids || !sec || !nsec || !poses)) throw std::invalid_argument("null record array");
    pf.n = n; pf.ids = ids; pf.sec = sec; pf.nsec = nsec; pf.poses = poses;
    pf.pending = true;
    pf.started = false;
    return 0;
  });
}

int te_pool_mailbox_ingest_prefetched(te_pool* p) {
  return guarded(p, [&] {
    te_pool::Prefetch& pf = p->prefetch;
    if (!pf.pending) throw std::logic_error("no prefetched message");
    prefetch_start(p);
    pf.pending = false;
    pf.started = false;
    if (pf.n == 0) return 0;
    const size_t nn = (size_t)pf.n;
    const uint32_t* d_ids = (const uint32_t*)pf.dev;
    const double* d_pose = (const double*)(pf.dev + ((nn * 12 + 255) & ~(size_t)255));
    CK(cudaStreamWaitEvent(p->stream, pf.keys_done, 0));
    return mailbox_ingest_impl(p, pf.n, pf.ids, pf.sec, pf.nsec, pf.poses, d_ids, d_ids + nn, d_ids + 2 * nn, d_pose, pf.done);
  });
}

int te_pool_mailbox_ingest_dev(te_pool* p, long long n, const uint32_t* dev_ids, const uint32_t* dev_sec, const uint32_t* dev_nsec,
                               const double* dev_poses) {
  return guarded(p, [&] {
    if (n <= 0) return 0;
    if (!dev_ids || !dev_sec || !dev_nsec || !dev_poses) throw std::invalid_argument("null record arrays");
    return mailbox_ingest_impl(p, n, nullptr, nullptr, nullptr, nullptr, dev_ids, dev_sec, dev_nsec, dev_poses);
  });
}

long long te_pool_mailbox_tick(te_pool* p, double dt, double t0_new, int cls_new, uint32_t now_sec, uint32_t now_nsec, double timeout,
                               uint32_t* erased_out, long long cap, uint32_t* added_out, long long added_cap, long long* n_added_out) {
  return guarded_ll(p, [&]() -> long long {
    if (!(dt >= 0.0)) throw std::invalid_argument("dt must be >= 0 (assert of src/target_interface.cpp:150)");
    if (p->hQ.empty()) throw std::runtime_error("no model class registered");
    if (cls_new < 0 || cls_new >= (int)p->hQ.size()) throw std::invalid_argument("unknown model class for the new targets");
    enable_mail(p);
    static const bool dbg = std::getenv("TE_MB_DEBUG") != nullptr;
    auto wall = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double tw[6] = {0, 0, 0, 0, 0, 0};
    auto mark = [&](int i) { if (dbg) { cudaStreamSynchronize(p->stream); tw[i] = wall(); } };
    mark(0);
    const double now = host_to_sec(now_sec, now_nsec);
    // 1. target-less mailboxes, ascending id: readable -> init on first sight (src/target_manager_ros.cpp:54-58) unless the
    //    same tick would erase it again (:67-72; init + update + erase is unobservable); unreadable -> stays, or expires
    // the add arrays are written straight into ONE pinned block [pose 7 | t0 | last | id | sec | nsec] x max_add and go to the
    // device in one copy
    std::vector<uint32_t> host_erased;
    const size_t max_add = p->pending.size() + p->orphans.size();
    char* stage = max_add ? pinned_stage(p, max_add * 84) : nullptr;
    double* add_pose = (double*)stage;
    double* add_t0 = add_pose + 7 * max_add;
    double* add_last = add_t0 + max_add;
    uint32_t* add_ids = (uint32_t*)(add_last + max_add);
    uint32_t* add_sec = add_ids + max_add;
    uint32_t* add_nsec = add_sec + max_add;
    size_t n_promoted = 0;
    auto promote = [&](uint32_t id, const HostMail& m) {
      const size_t k = n_promoted++;
      add_ids[k] = id;
      add_sec[k] = m.sec;
      add_nsec[k] = m.nsec;
      add_last[k] = m.last;
      add_t0[k] = t0_new;
      std::memcpy(add_pose + 7 * k, m.pose, 56);
    };
    bool fast = p->orphans.empty();   // common case: every queued record is the first sight of a new id, ids ascending
    for (size_t k = 1; fast && k < p->pending.size(); ++k) fast = p->pending[k - 1].id < p->pending[k].id;
    if (fast) {
      for (const PendingRec& r : p->pending) {
        HostMail m;   // Measurement(): readable, stamp 0
        apply_record(m, r);
        if (m.last > 0.0 && (now - m.last) >= timeout) host_erased.push_back(r.id);
        else if (m.fresh) promote(r.id, m);
        else p->orphans.emplace_hint(p->orphans.end(), r.id, m);   // "Target(id) does not exist!" (src/target_manager.cpp:209)
      }
      p->pending.clear();
    } else {
      fold_pending(p);
      for (auto it = p->orphans.begin(); it != p->orphans.end();) {
        const HostMail& m = it->second;
        const bool expired = m.last > 0.0 && (now - m.last) >= timeout;
        if (expired) {
          host_erased.push_back(it->first);
          it = p->orphans.erase(it);
        } else if (m.fresh) {
          promote(it->first, m);
          it = p->orphans.erase(it);
        } else {
          ++it;
        }
      }
    }
    const int n_add = (int)n_promoted;
    const int n_old = (int)p->n;
    if (n_added_out) *n_added_out = n_add;
    if (added_out && added_cap > 0 && n_add > 0) std::memcpy(added_out, add_ids, (size_t)std::min<long long>(added_cap, n_add) * sizeof(uint32_t));
    mark(1);
    // 2. expiry flags of the existing targets, then ONE stable rebuild: survivors compacted, promoted mailboxes merged in by id
    ensure_work(p, (size_t)n_old + (size_t)n_add);
    uint32_t* d_erased = nullptr;
    long long n_dev_erased = 0;
    if (n_old > 0) {
      te::expire_flags_kernel<<<cdiv(n_old, 256), 256, 0, p->stream>>>(p->buf[p->cur].cold.last_meas, n_old, now, timeout, p->alive);
      CK(cudaGetLastError());
      d_erased = p->arena.get_n<uint32_t>((size_t)n_old);
    }
    te::AddData ad{};
    std::vector<uint16_t> add_cls;
    if (n_add > 0) {
      char* d_stage = (char*)p->arena.get(max_add * 84);
      CK(cudaMemcpyAsync(d_stage, stage, max_add * 84, cudaMemcpyHostToDevice, p->stream));   // (pinned: the final sync of the tick covers it)
      const double* d_pose0 = (const double*)d_stage;
      const double* d_t0 = d_pose0 + 7 * max_add;
      const double* d_last = d_t0 + max_add;
      const uint32_t* d_aid = (const uint32_t*)(d_last + max_add);
      ad.ids = d_aid;
      if (cls_new != 0) {
        add_cls.assign((size_t)n_add, (uint16_t)cls_new);
        ad.cls = to_dev(p, add_cls.data(), (size_t)n_add);
      }
      ad.t0 = d_t0;
      ad.p0 = d_pose0;
      p->mb_add.sec = d_aid + max_add;
      p->mb_add.nsec = d_aid + 2 * max_add;
      p->mb_add.last = d_last;
    }
    // a registered /tf message (te_pool_mailbox_prefetch) starts its way to the device now: this tick's own small uploads are already
    // in the copy engine's queue (the device has ONE host-to-device engine and serves its queue in order -- 71 MB ahead of them held
    // the whole tick back by 1.2 ms), and the message then travels under the kernels of this tick
    prefetch_start(p);
    const bool unfused_env = std::getenv("TE_MB_UNFUSED") != nullptr;   // debugging / test switch: the rebuild-then-step form
    const bool fused = !unfused_env && n_old > 0;
    if (!fused) {
      // reference form: stable rebuild (survivors gathered, new ids merged in and initialised), then the step in place
      if (n_old > 0 || n_add > 0) {
        int alive = 0;
        try {
          alive = compact_and_merge(p, ad, ad.ids, n_add, d_erased);
        } catch (...) {
          p->mb_add = te::MailAdd{nullptr, nullptr, nullptr};
          throw;
        }
        n_dev_erased = n_old - alive;
      }
      p->mb_add = te::MailAdd{nullptr, nullptr, nullptr};
      mark(2);
      // 3. the step: update where the mailbox is readable (the flag is sticky: a silent target re-applies its last pose),
      //    predict elsewhere (:59,:64).  The mailbox arrays are the kernel's measurement block and action array.
      if (p->n > 0) {
        te::StepArgs a = base_args(p);
        const te::MailArrays& mb = p->mb[p->mb_cur].a;
        a.dt = dt;
        a.meas = mb.pose;
        a.meas_stride = 7;
        a.meas_tma = 1;
        a.action = mb.act;
        a.default_action = TE_ACT_PREDICT;
        launch_step(p, a, a.n_tiles);
        te::copy_meas_masked_kernel<<<cdiv(p->n, 256), 256, 0, p->stream>>>(p->buf[p->cur].cold.meas, mb.pose, mb.act, (int)p->n);
        CK(cudaGetLastError());
      }
    } else {
      // fused form (same results bit for bit): the step kernel reads every tile in place and writes the survivors' columns
      // straight to their slots in the merged order (StepArgs::dst_*), so the state crosses HBM once per tick; the promoted
      // mailboxes are initialised in their slots afterwards and get their first update from a sparse follow-up launch
      Buf& ob = p->buf[p->cur];
      const te::MailArrays omb = p->mb[p->mb_cur].a;
      size_t tmp = p->cub_bytes;
      CK(cub::DeviceScan::ExclusiveSum(p->cub_tmp, tmp, p->alive, p->pos, n_old, p->stream));
      int last_pos = 0, last_alive = 0;
      CK(cudaMemcpyAsync(&last_pos, p->pos + n_old - 1, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
      CK(cudaMemcpyAsync(&last_alive, p->alive + n_old - 1, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
      CK(cudaStreamSynchronize(p->stream));
      const int n_alive = last_pos + last_alive;
      n_dev_erased = n_old - n_alive;
      te::StepArgs a = base_args(p);
      a.dt = dt;
      a.meas = omb.pose;
      a.meas_stride = 7;
      a.meas_tma = 1;
      a.action = omb.act;
      a.default_action = TE_ACT_PREDICT;
      te::copy_meas_masked_kernel<<<cdiv(n_old, 256), 256, 0, p->stream>>>(ob.cold.meas, omb.pose, omb.act, n_old);   // measured_pose_
      CK(cudaGetLastError());
      if (n_dev_erased == 0 && n_add == 0) {
        launch_step(p, a, a.n_tiles);   // nothing moves: the ordinary in-place step
        p->mb_add = te::MailAdd{nullptr, nullptr, nullptr};
        mark(2);
      } else {
        const int n_new = n_alive + n_add;
        if (n_dev_erased > 0) {
          te::collect_erased_kernel<<<cdiv(n_old, 256), 256, 0, p->stream>>>(p->alive, p->pos, ob.cold.ids, n_old, d_erased);
          CK(cudaGetLastError());
        }
        ensure_other_capacity(p, (size_t)n_new);
        ensure_mail_other(p, (size_t)n_new);
        Buf& nb = p->buf[1 - p->cur];
        const te::MailArrays nmb = p->mb[1 - p->mb_cur].a;
        int* new_dst = nullptr;
        if (n_add > 0) {
          new_dst = p->arena.get_n<int>((size_t)n_add);
          te::merge_new_dst_kernel<<<cdiv(n_add, 256), 256, 0, p->stream>>>(n_add, ad.ids, ob.cold.ids, n_old, p->pos, n_alive, new_dst);
          te::merge_old_dst_kernel<<<cdiv(n_old, 256), 256, 0, p->stream>>>(n_old, p->alive, p->pos, ob.cold.ids, ad.ids, n_add);
          CK(cudaGetLastError());
        }
        te::compact_cold_kernel<<<cdiv(n_old, 256), 256, 0, p->stream>>>(n_old, p->alive, p->pos, ob.cold, nb.cold);
        te::mb_compact_kernel<<<cdiv(n_old, 256), 256, 0, p->stream>>>(n_old, p->alive, p->pos, omb, nmb);
        CK(cudaGetLastError());
        if (n_alive > 0) {
          a.dst_tiles = nb.tiles;
          a.dst_alive = p->alive;
          a.dst_pos = p->pos;
          launch_step(p, a, a.n_tiles);
        }
        if (n_add > 0) {
          CK(cudaMemsetAsync(p->d_counters, 0, 2 * sizeof(int), p->stream));
          init_promoted(p, n_add, new_dst, nb, ad, nmb);
        }
        p->mb_add = te::MailAdd{nullptr, nullptr, nullptr};
        p->cur = 1 - p->cur;
        p->mb_cur = 1 - p->mb_cur;
        p->n = n_new;
        p->h_ids_valid = false;
        mark(2);
        if (n_add > 0) {   // first update of the new targets with the pose that created them: only their tiles, only their lanes
          te::StepArgs b = base_args(p);
          b.tile_list = p->tile_list;
          b.d_nwork = p->d_counters;
          b.dt = dt;
          b.meas = nmb.pose;
          b.meas_stride = 7;
          b.meas_tma = 1;
          b.action = p->action;
          b.default_action = TE_ACT_NONE;
          b.clear_action = 1;
          b.tile_flag = p->tile_flag;
          launch_step(p, b, std::min(n_add, b.n_tiles));
        }
        fetch_last_id(p);
      }
    }
    mark(3);
    // 4. erased ids of this tick, ascending: targets the device expired + target-less mailboxes the host expired
    std::vector<uint32_t> dev_erased((size_t)n_dev_erased);
    if (n_dev_erased > 0)
      CK(cudaMemcpyAsync(dev_erased.data(), d_erased, (size_t)n_dev_erased * sizeof(uint32_t), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    const long long n_er = n_dev_erased + (long long)host_erased.size();
    if (erased_out && cap > 0 && n_er > 0) {
      std::vector<uint32_t> all((size_t)n_er);
      std::merge(dev_erased.begin(), dev_erased.end(), host_erased.begin(), host_erased.end(), all.begin());
      std::memcpy(erased_out, all.data(), (size_t)std::min(cap, n_er) * sizeof(uint32_t));
    }
    mark(4);
    if (dbg) std::fprintf(stderr, "[te mailbox tick] host mailboxes %.3f ms, flags + merge (fused: + step) %.3f ms, step (fused: first update of the new targets) %.3f ms, erase list %.3f ms (n %lld, +%d, -%lld)\n",
                          tw[1] - tw[0], tw[2] - tw[1], tw[3] - tw[2], tw[4] - tw[3], p->n, n_add, n_er);
    return n_er;
  });
}

long long te_pool_mailbox_count(te_pool* p) {
  return guarded_ll(p, [&]() -> long long {
    fold_pending(p);
    long long n = (long long)p->orphans.size();
    if (!p->mb_on || p->n == 0) return n;
    int* counter = p->arena.get_n<int>(1);
    CK(cudaMemsetAsync(counter, 0, sizeof(int), p->stream));
    te::mb_count_kernel<<<cdiv(p->n, 256), 256, 0, p->stream>>>(p->mb[p->mb_cur].a.act, (int)p->n, counter);
    CK(cudaGetLastError());
    int c = 0;
    CK(cudaMemcpyAsync(&c, counter, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    return n + c;
  });
}

long long te_pool_mailbox_bound(te_pool* p) { return p ? p->n + (long long)p->orphans.size() + (long long)p->pending.size() : -1; }

const double* te_pool_mailbox_dev_pose(te_pool* p) { return (p && p->mb_on) ? p->mb[p->mb_cur].a.pose : nullptr; }
const uint8_t* te_pool_mailbox_dev_action(te_pool* p) { return (p && p->mb_on) ? p->mb[p->mb_cur].a.act : nullptr; }

}  // extern "C"
