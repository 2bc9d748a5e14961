// te_pool.cu -- host side of the thin extern "C" CUDA layer declared in include/te_pool.h: pool lifecycle, model classes,
// add / erase, read-back, expiry.
//
// One te_pool = the targets of one model type on one device, stored as tiles of 32 targets
// ([tile][field][lane], te_device.cuh Layout) in ascending-id slot order -- the iteration order of
// the reference's std::map<unsigned, TargetInterface::Ptr> (include/target_estimation/
// target_manager.hpp:36).  Add / erase rebuild the pool by a stable gather into the second buffer
// (stream compaction; ids stay sorted); the append fast path (all new ids larger than every
// existing id) writes in place.  There is no CPU fallback: every entry point needs a CUDA device.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <cmath>

#include "te_pool_internal.cuh"

namespace tehost {

std::string& last_error() {
  static thread_local std::string g_err;
  return g_err;
}

size_t tile_doubles(const te_pool* p) { return (size_t)p->NF * te::TILE; }

void free_buf(Buf& b) {
  cudaFree(b.tiles);
  cudaFree(b.cold.ids);
  cudaFree(b.cold.cls);
  cudaFree(b.cold.last_meas);
  cudaFree(b.cold.meas);
  b = Buf();
}

void alloc_buf(te_pool* p, Buf& b, size_t slots) {
  slots = (slots + te::TILE - 1) / te::TILE * te::TILE;
  if (slots == 0) slots = te::TILE;
  CK(cudaMalloc(&b.tiles, slots / te::TILE * tile_doubles(p) * sizeof(double)));
  CK(cudaMalloc(&b.cold.ids, slots * sizeof(uint32_t)));
  CK(cudaMalloc(&b.cold.cls, slots * sizeof(uint16_t)));
  CK(cudaMalloc(&b.cold.last_meas, slots * sizeof(double)));
  CK(cudaMalloc(&b.cold.meas, slots * 7 * sizeof(double)));
  b.cap = slots;
  // pad lanes of the last tile are streamed by the step kernel: keep them finite
  CK(cudaMemsetAsync(b.tiles, 0, slots / te::TILE * tile_doubles(p) * sizeof(double), p->stream));
  CK(cudaMemsetAsync(b.cold.meas, 0, slots * 7 * sizeof(double), p->stream));
  CK(cudaMemsetAsync(b.cold.last_meas, 0, slots * sizeof(double), p->stream));
}

// make sure the per-slot work arrays cover `slots`
void ensure_work(te_pool* p, size_t slots) {
  slots = (slots + te::TILE - 1) / te::TILE * te::TILE;
  if (slots <= p->wcap) return;
  size_t cap = std::max(slots, p->wcap + p->wcap / 2);
  cap = (cap + te::TILE - 1) / te::TILE * te::TILE;
  CK(cudaStreamSynchronize(p->stream));
  cudaFree(p->action); cudaFree(p->dt_slot); cudaFree(p->tile_flag); cudaFree(p->tile_list);
  cudaFree(p->alive); cudaFree(p->pos); cudaFree(p->srcmap);
  CK(cudaMalloc(&p->action, cap));
  CK(cudaMalloc(&p->dt_slot, cap * sizeof(double)));
  CK(cudaMalloc(&p->tile_flag, cap / te::TILE + 4));
  CK(cudaMalloc(&p->tile_list, cap / te::TILE * sizeof(int)));
  CK(cudaMalloc(&p->alive, cap * sizeof(int)));
  CK(cudaMalloc(&p->pos, cap * sizeof(int)));
  CK(cudaMalloc(&p->srcmap, cap * sizeof(int)));
  CK(cudaMemsetAsync(p->action, 0, cap, p->stream));
  CK(cudaMemsetAsync(p->tile_flag, 0, cap / te::TILE + 4, p->stream));
  p->wcap = cap;
  size_t need = 0;
  CK(cub::DeviceScan::ExclusiveSum(nullptr, need, p->alive, p->pos, (int)cap, p->stream));
  if (need > p->cub_bytes) {
    cudaFree(p->cub_tmp);
    CK(cudaMalloc(&p->cub_tmp, need));
    p->cub_bytes = need;
  }
}

// current buffer must hold `slots` (append path / reserve): grow by copy
void ensure_cur_capacity(te_pool* p, size_t slots) {
  Buf& b = p->buf[p->cur];
  if (slots <= b.cap) return;
  size_t cap = std::max(slots, b.cap + b.cap / 2);
  Buf nb;
  alloc_buf(p, nb, cap);
  if (p->n > 0) {
    size_t tiles = (size_t)cdiv(p->n, te::TILE);
    CK(cudaMemcpyAsync(nb.tiles, b.tiles, tiles * tile_doubles(p) * sizeof(double), cudaMemcpyDeviceToDevice, p->stream));
    CK(cudaMemcpyAsync(nb.cold.ids, b.cold.ids, p->n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, p->stream));
    CK(cudaMemcpyAsync(nb.cold.cls, b.cold.cls, p->n * sizeof(uint16_t), cudaMemcpyDeviceToDevice, p->stream));
    CK(cudaMemcpyAsync(nb.cold.last_meas, b.cold.last_meas, p->n * sizeof(double), cudaMemcpyDeviceToDevice, p->stream));
    CK(cudaMemcpyAsync(nb.cold.meas, b.cold.meas, p->n * 7 * sizeof(double), cudaMemcpyDeviceToDevice, p->stream));
  }
  CK(cudaStreamSynchronize(p->stream));
  free_buf(b);
  b = nb;
  ensure_work(p, b.cap);
}

void ensure_other_capacity(te_pool* p, size_t slots) {
  Buf& b = p->buf[1 - p->cur];
  if (slots <= b.cap && b.tiles) return;
  CK(cudaStreamSynchronize(p->stream));
  free_buf(b);
  // grow geometrically: a pool that gains a few targets per tick must not re-allocate gigabytes on every tick
  alloc_buf(p, b, std::max(slots + slots / 4, p->buf[p->cur].cap));
  // the work arrays hold the live alive[] / pos[] of the running compaction: callers size them up-front
  if (p->wcap < slots) throw std::logic_error("work arrays not sized before compaction");
}

// ---- mailboxes -------------------------------------------------------------------------------
char* pinned_stage(te_pool* p, size_t bytes) {
  if (bytes > p->h_stage_cap) {
    CK(cudaStreamSynchronize(p->stream));
    if (p->h_stage) cudaFreeHost(p->h_stage);
    p->h_stage = nullptr;
    p->h_stage_cap = 0;
    const size_t cap = bytes + bytes / 2 + 4096;
    CK(cudaHostAlloc((void**)&p->h_stage, cap, cudaHostAllocDefault));
    p->h_stage_cap = cap;
  }
  return p->h_stage;
}
void free_mail(MailBuf& m) {
  cudaFree(m.a.sec); cudaFree(m.a.nsec); cudaFree(m.a.act); cudaFree(m.a.pose);
  m = MailBuf();
}
void alloc_mail(MailBuf& m, size_t slots) {
  slots = (slots + te::TILE - 1) / te::TILE * te::TILE;
  if (slots == 0) slots = te::TILE;
  CK(cudaMalloc(&m.a.sec, slots * sizeof(uint32_t)));
  CK(cudaMalloc(&m.a.nsec, slots * sizeof(uint32_t)));
  CK(cudaMalloc(&m.a.act, slots));
  CK(cudaMalloc(&m.a.pose, slots * 7 * sizeof(double)));   // cudaMalloc is 256-byte aligned: TMA-loadable measurement block
  m.cap = slots;
}
// the current generation holds `slots` mailboxes (grow by copy, like ensure_cur_capacity)
void ensure_mail_cur(te_pool* p, size_t slots) {
  MailBuf& m = p->mb[p->mb_cur];
  if (slots <= m.cap && m.a.sec) return;
  MailBuf nm;
  alloc_mail(nm, std::max({slots, m.cap + m.cap / 2, p->buf[p->cur].cap}));   // sized like the slot buffers: no per-tick regrowth
  if (p->n > 0 && m.a.sec) {
    CK(cudaMemcpyAsync(nm.a.sec, m.a.sec, p->n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, p->stream));
    CK(cudaMemcpyAsync(nm.a.nsec, m.a.nsec, p->n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, p->stream));
    CK(cudaMemcpyAsync(nm.a.act, m.a.act, p->n, cudaMemcpyDeviceToDevice, p->stream));
    CK(cudaMemcpyAsync(nm.a.pose, m.a.pose, p->n * 7 * sizeof(double), cudaMemcpyDeviceToDevice, p->stream));
  }
  CK(cudaStreamSynchronize(p->stream));
  free_mail(m);
  m = nm;
}
void ensure_mail_other(te_pool* p, size_t slots) {
  MailBuf& m = p->mb[1 - p->mb_cur];
  if (slots <= m.cap && m.a.sec) return;
  CK(cudaStreamSynchronize(p->stream));
  free_mail(m);
  alloc_mail(m, std::max({slots + slots / 8, p->mb[p->mb_cur].cap, p->buf[p->cur].cap, p->buf[1 - p->cur].cap}));
}
// first use: every existing target gets an empty mailbox
void enable_mail(te_pool* p) {
  if (p->mb_on) return;
  ensure_mail_cur(p, std::max<size_t>((size_t)p->n, te::TILE));
  if (p->n > 0) {
    te::mb_clear_kernel<<<cdiv(p->n, 256), 256, 0, p->stream>>>(p->mb[p->mb_cur].a, 0, (int)p->n);
    CK(cudaGetLastError());
  }
  p->mb_on = true;
}

void sync_host_ids(te_pool* p) {
  if (p->h_ids_valid) return;
  p->h_ids.resize((size_t)p->n);
  if (p->n) {
    CK(cudaMemcpyAsync(p->h_ids.data(), p->buf[p->cur].cold.ids, p->n * sizeof(uint32_t), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
  }
  p->h_ids_valid = true;
  if (p->n) { p->h_last_id = p->h_ids.back(); p->h_last_valid = true; }
}

void upload_classes(te_pool* p) {
  const int nc = (int)p->hQ.size();
  if (nc > p->cls_cap) {
    CK(cudaStreamSynchronize(p->stream));
    cudaFree(p->dQ); cudaFree(p->dR); cudaFree(p->dP0); cudaFree(p->dT);
    int cap = std::max(nc, std::max(4, p->cls_cap * 2));
    CK(cudaMalloc(&p->dQ, (size_t)cap * p->N * p->N * sizeof(double)));
    CK(cudaMalloc(&p->dR, (size_t)cap * p->M * p->M * sizeof(double)));
    CK(cudaMalloc(&p->dP0, (size_t)cap * p->N * p->N * sizeof(double)));
    CK(cudaMalloc(&p->dT, (size_t)cap * p->M * p->M * sizeof(double)));
    p->cls_cap = cap;
    for (int c = 0; c < nc; ++c) {
      CK(cudaMemcpyAsync(p->dQ + (size_t)c * p->N * p->N, p->hQ[c].data(), p->N * p->N * sizeof(double), cudaMemcpyHostToDevice, p->stream));
      CK(cudaMemcpyAsync(p->dR + (size_t)c * p->M * p->M, p->hR[c].data(), p->M * p->M * sizeof(double), cudaMemcpyHostToDevice, p->stream));
      CK(cudaMemcpyAsync(p->dP0 + (size_t)c * p->N * p->N, p->hP0[c].data(), p->N * p->N * sizeof(double), cudaMemcpyHostToDevice, p->stream));
      CK(cudaMemcpyAsync(p->dT + (size_t)c * p->M * p->M, p->hT[c].data(), p->M * p->M * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    }
  } else {
    const int c = nc - 1;
    CK(cudaMemcpyAsync(p->dQ + (size_t)c * p->N * p->N, p->hQ[c].data(), p->N * p->N * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    CK(cudaMemcpyAsync(p->dR + (size_t)c * p->M * p->M, p->hR[c].data(), p->M * p->M * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    CK(cudaMemcpyAsync(p->dP0 + (size_t)c * p->N * p->N, p->hP0[c].data(), p->N * p->N * sizeof(double), cudaMemcpyHostToDevice, p->stream));
    CK(cudaMemcpyAsync(p->dT + (size_t)c * p->M * p->M, p->hT[c].data(), p->M * p->M * sizeof(double), cudaMemcpyHostToDevice, p->stream));
  }
  CK(cudaStreamSynchronize(p->stream));
}


// ---- rebuild (stable gather of survivors + init of new targets) ----------------------------
template <int TYPE>
void rebuild_t(te_pool* p, int n_new, const te::AddData& ad) {
  Buf& ob = p->buf[p->cur];
  Buf& nb = p->buf[1 - p->cur];
  const dim3 grid(cdiv(n_new, 128), (te::Layout<TYPE>::NF + te::REBUILD_FPT - 1) / te::REBUILD_FPT);
  te::rebuild_kernel<TYPE><<<grid, 128, 0, p->stream>>>(n_new, p->srcmap, ob.tiles, ob.cold, nb.tiles, nb.cold, ad, p->dP0);
  CK(cudaGetLastError());
}
void rebuild(te_pool* p, int n_new, const te::AddData& ad) {
  switch (p->model) {
    case te::UNIFORM_VELOCITY: rebuild_t<te::UNIFORM_VELOCITY>(p, n_new, ad); break;
    case te::UNIFORM_ACCELERATION: rebuild_t<te::UNIFORM_ACCELERATION>(p, n_new, ad); break;
    case te::ANGULAR_VELOCITIES: rebuild_t<te::ANGULAR_VELOCITIES>(p, n_new, ad); break;
    default: rebuild_t<te::ANGULAR_RATES>(p, n_new, ad); break;
  }
}
template <int TYPE>
void init_append_t(te_pool* p, int base, const te::AddData& ad, long long n) {
  Buf& b = p->buf[p->cur];
  te::init_append_kernel<TYPE><<<cdiv(n, 128), 128, 0, p->stream>>>(b.tiles, b.cold, base, ad, n, p->dP0);
  CK(cudaGetLastError());
}
void init_append(te_pool* p, int base, const te::AddData& ad, long long n) {
  switch (p->model) {
    case te::UNIFORM_VELOCITY: init_append_t<te::UNIFORM_VELOCITY>(p, base, ad, n); break;
    case te::UNIFORM_ACCELERATION: init_append_t<te::UNIFORM_ACCELERATION>(p, base, ad, n); break;
    case te::ANGULAR_VELOCITIES: init_append_t<te::ANGULAR_VELOCITIES>(p, base, ad, n); break;
    default: init_append_t<te::ANGULAR_RATES>(p, base, ad, n); break;
  }
}

template <int TYPE>
void init_promoted_t(te_pool* p, int n_add, const int* new_dst, const Buf& nb, const te::AddData& ad, const te::MailArrays& mb) {
  te::init_promoted_kernel<TYPE><<<cdiv(n_add, 128), 128, 0, p->stream>>>(n_add, new_dst, nb.tiles, nb.cold, ad, p->mb_add, mb, p->dP0, p->action,
                                                                          p->tile_flag, p->tile_list, p->d_counters);
  CK(cudaGetLastError());
}
void init_promoted(te_pool* p, int n_add, const int* new_dst, const Buf& nb, const te::AddData& ad, const te::MailArrays& mb) {
  switch (p->model) {
    case te::UNIFORM_VELOCITY: init_promoted_t<te::UNIFORM_VELOCITY>(p, n_add, new_dst, nb, ad, mb); break;
    case te::UNIFORM_ACCELERATION: init_promoted_t<te::UNIFORM_ACCELERATION>(p, n_add, new_dst, nb, ad, mb); break;
    case te::ANGULAR_VELOCITIES: init_promoted_t<te::ANGULAR_VELOCITIES>(p, n_add, new_dst, nb, ad, mb); break;
    default: init_promoted_t<te::ANGULAR_RATES>(p, n_add, new_dst, nb, ad, mb); break;
  }
}

// after a compaction: the largest surviving id (4 bytes; the callers synchronise the stream before they return)
void fetch_last_id(te_pool* p) {
  p->h_last_valid = false;
  if (p->n > 0) {
    CK(cudaMemcpyAsync(&p->h_last_id, p->buf[p->cur].cold.ids + p->n - 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    p->h_last_valid = true;
  }
}

// alive[] (n_old entries) is set on the device; compacts survivors, merges `n_add` sorted new ids.
// Returns the number of survivors.
int compact_and_merge(te_pool* p, const te::AddData& ad, const uint32_t* d_add_ids, int n_add, uint32_t* d_erased /*or null*/) {
  const int n_old = (int)p->n;
  int total_alive = 0;
  if (n_old > 0) {
    size_t tmp = p->cub_bytes;
    CK(cub::DeviceScan::ExclusiveSum(p->cub_tmp, tmp, p->alive, p->pos, n_old, p->stream));
    int last_pos = 0, last_alive = 0;
    CK(cudaMemcpyAsync(&last_pos, p->pos + n_old - 1, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaMemcpyAsync(&last_alive, p->alive + n_old - 1, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    total_alive = last_pos + last_alive;
  }
  const int n_new = total_alive + n_add;
  if (d_erased && n_old > total_alive) {
    te::collect_erased_kernel<<<cdiv(n_old, 256), 256, 0, p->stream>>>(p->alive, p->pos, p->buf[p->cur].cold.ids, n_old, d_erased);
    CK(cudaGetLastError());
  }
  if (n_new == n_old && n_add == 0) return total_alive;   // nothing erased, nothing added
  ensure_other_capacity(p, (size_t)n_new);
  if (n_old > 0) {
    te::map_existing_kernel<<<cdiv(n_old, 256), 256, 0, p->stream>>>(n_old, p->alive, p->pos, p->buf[p->cur].cold.ids, d_add_ids, n_add, p->srcmap);
    CK(cudaGetLastError());
  }
  if (n_add > 0) {
    te::map_new_kernel<<<cdiv(n_add, 256), 256, 0, p->stream>>>(n_add, d_add_ids, p->buf[p->cur].cold.ids, n_old, p->pos, total_alive, p->srcmap);
    CK(cudaGetLastError());
  }
  if (n_new > 0) rebuild(p, n_new, ad);
  if (p->mb_on) {   // the mailboxes follow their slots; promoted host mailboxes are filled in (after rebuild: it zeroes last_meas of new slots)
    ensure_mail_other(p, (size_t)n_new);
    if (n_new > 0) {
      te::mb_move_kernel<<<cdiv(n_new, 256), 256, 0, p->stream>>>(n_new, p->srcmap, p->mb[p->mb_cur].a, p->mb[1 - p->mb_cur].a, p->mb_add, ad.p0,
                                                                  p->buf[1 - p->cur].cold.last_meas);
      CK(cudaGetLastError());
    }
    p->mb_cur = 1 - p->mb_cur;
  }
  p->cur = 1 - p->cur;
  p->n = n_new;
  p->h_ids_valid = false;
  fetch_last_id(p);
  return total_alive;
}

int* lookup_slots(te_pool* p, const uint32_t* d_ids, long long n) {
  int* slots = p->arena.get_n<int>((size_t)n);
  te::lookup_slots_kernel<<<cdiv(n, 256), 256, 0, p->stream>>>(p->buf[p->cur].cold.ids, (int)p->n, d_ids, n, slots);
  CK(cudaGetLastError());
  return slots;
}

// queued records of unknown ids -> their (host) mailboxes, in arrival order
void fold_pending(te_pool* p) {
  for (const PendingRec& r : p->pending) apply_record(p->orphans[r.id], r);
  p->pending.clear();
}

// A target erased by hand keeps its mailbox in the reference (TargetManager::erase does not know the adapter's map,
// src/target_manager.cpp:227-241): the mailboxes of the listed slots move to the host's target-less map before the compaction.
void demote_mailboxes(te_pool* p, const uint32_t* ids, const int* d_slots, long long n) {
  uint32_t* d_sec = p->arena.get_n<uint32_t>((size_t)n);
  uint32_t* d_nsec = p->arena.get_n<uint32_t>((size_t)n);
  uint8_t* d_act = p->arena.get_n<uint8_t>((size_t)n);
  double* d_last = p->arena.get_n<double>((size_t)n);
  double* d_pose = p->arena.get_n<double>((size_t)n * 7);
  te::mb_gather_kernel<<<cdiv(n, 256), 256, 0, p->stream>>>((int)n, d_slots, p->mb[p->mb_cur].a, p->buf[p->cur].cold.last_meas, d_sec, d_nsec, d_act,
                                                            d_last, d_pose);
  CK(cudaGetLastError());
  std::vector<uint32_t> sec((size_t)n), nsec((size_t)n);
  std::vector<uint8_t> act((size_t)n);
  std::vector<double> last((size_t)n), pose((size_t)n * 7);
  CK(cudaMemcpyAsync(sec.data(), d_sec, (size_t)n * 4, cudaMemcpyDeviceToHost, p->stream));
  CK(cudaMemcpyAsync(nsec.data(), d_nsec, (size_t)n * 4, cudaMemcpyDeviceToHost, p->stream));
  CK(cudaMemcpyAsync(act.data(), d_act, (size_t)n, cudaMemcpyDeviceToHost, p->stream));
  CK(cudaMemcpyAsync(last.data(), d_last, (size_t)n * 8, cudaMemcpyDeviceToHost, p->stream));
  CK(cudaMemcpyAsync(pose.data(), d_pose, (size_t)n * 56, cudaMemcpyDeviceToHost, p->stream));
  CK(cudaStreamSynchronize(p->stream));
  for (long long k = 0; k < n; ++k) {
    if (act[(size_t)k] == 0xFF || act[(size_t)k] == (uint8_t)TE_ACT_NONE) continue;   // unknown id / target without a mailbox
    HostMail& m = p->orphans[ids[k]];
    m.sec = sec[(size_t)k];
    m.nsec = nsec[(size_t)k];
    m.last = last[(size_t)k];
    m.fresh = act[(size_t)k] == (uint8_t)TE_ACT_UPDATE;
    std::memcpy(m.pose, &pose[(size_t)k * 7], sizeof(m.pose));
  }
}
// ... and a target created by hand for an id that already has a (target-less) mailbox is fed by it from the next tick on
void attach_mailboxes(te_pool* p, const uint32_t* ids, long long n) {
  fold_pending(p);
  std::vector<uint32_t> a_ids, sec, nsec;
  std::vector<uint8_t> act;
  std::vector<double> last, pose;
  for (long long k = 0; k < n; ++k) {
    auto it = p->orphans.find(ids[k]);
    if (it == p->orphans.end()) continue;
    const HostMail& m = it->second;
    a_ids.push_back(ids[k]);
    sec.push_back(m.sec);
    nsec.push_back(m.nsec);
    act.push_back((uint8_t)(m.fresh ? TE_ACT_UPDATE : TE_ACT_PREDICT));
    last.push_back(m.last);
    pose.insert(pose.end(), m.pose, m.pose + 7);
    p->orphans.erase(it);
  }
  const long long na = (long long)a_ids.size();
  if (na == 0) return;
  uint32_t* d_ids = to_dev(p, a_ids.data(), (size_t)na);
  int* slots = lookup_slots(p, d_ids, na);
  te::mb_scatter_kernel<<<cdiv(na, 256), 256, 0, p->stream>>>((int)na, slots, to_dev(p, sec.data(), (size_t)na), to_dev(p, nsec.data(), (size_t)na),
                                                              to_dev(p, act.data(), (size_t)na), to_dev(p, last.data(), (size_t)na),
                                                              to_dev(p, pose.data(), (size_t)na * 7), p->mb[p->mb_cur].a,
                                                              p->buf[p->cur].cold.last_meas);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(p->stream));   // the host vectors above go out of scope
}

void launch_gather_estimates(te_pool* p, const int* slots, long long n, const double* d_t1, double* pose, double* twist, double* acc,
                             double* pose6, uint8_t* found, int rec13) {
  Buf& b = p->buf[p->cur];
  const int g = cdiv(n, 128);
  switch (p->model) {
    case te::UNIFORM_VELOCITY: te::gather_estimates_kernel<te::UNIFORM_VELOCITY><<<g, 128, 0, p->stream>>>(b.tiles, slots, n, d_t1, pose, twist, acc, pose6, found, rec13); break;
    case te::UNIFORM_ACCELERATION: te::gather_estimates_kernel<te::UNIFORM_ACCELERATION><<<g, 128, 0, p->stream>>>(b.tiles, slots, n, d_t1, pose, twist, acc, pose6, found, rec13); break;
    case te::ANGULAR_VELOCITIES: te::gather_estimates_kernel<te::ANGULAR_VELOCITIES><<<g, 128, 0, p->stream>>>(b.tiles, slots, n, d_t1, pose, twist, acc, pose6, found, rec13); break;
    default: te::gather_estimates_kernel<te::ANGULAR_RATES><<<g, 128, 0, p->stream>>>(b.tiles, slots, n, d_t1, pose, twist, acc, pose6, found, rec13); break;
  }
  CK(cudaGetLastError());
}

}  // namespace tehost

using namespace tehost;
#define g_err (tehost::last_error())

extern "C" {

const char* te_last_error(void) { return g_err.c_str(); }

int te_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int te_host_register(void* ptr, size_t bytes) {
  if (!ptr || !bytes) return 0;
  cudaError_t e = cudaHostRegister(ptr, bytes, cudaHostRegisterDefault);
  if (e != cudaSuccess) { cudaGetLastError(); g_err = std::string("cudaHostRegister: ") + cudaGetErrorString(e); return -1; }
  return 0;
}
int te_host_unregister(void* ptr) {
  if (!ptr) return 0;
  cudaError_t e = cudaHostUnregister(ptr);
  if (e != cudaSuccess) { cudaGetLastError(); g_err = std::string("cudaHostUnregister: ") + cudaGetErrorString(e); return -1; }
  return 0;
}

int te_model_dims(int model, int* n, int* m) {
  if (model < 0 || model > 3) return -1;
  if (n) *n = te::model_n(model);
  if (m) *m = te::model_m(model);
  return 0;
}

size_t te_model_bytes_per_step(int model) {
  // SURVEY.md 8(d): read x, P, measurement (+prev rpy), write x, P (+prev rpy), + 32 B of t / n_meas
  switch (model) {
    case TE_UNIFORM_VELOCITY: return 728;
    case TE_UNIFORM_ACCELERATION: return 1496;
    case TE_ANGULAR_VELOCITIES: return 2632;
    case TE_ANGULAR_RATES: return 5608;
    default: return 0;
  }
}

te_pool* te_pool_create(int model, int device, void* cuda_stream) {
  te_pool* p = nullptr;
  try {
    if (model < 0 || model > 3) throw std::invalid_argument("unknown model type");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
      cudaGetLastError();
      throw std::runtime_error("no CUDA device available: the target pool has no CPU fallback");
    }
    if (device < 0 || device >= ndev) throw std::invalid_argument("bad device index");
    DeviceGuard g(device);
    p = new te_pool();
    p->model = model;
    p->device = device;
    p->N = te::model_n(model);
    p->M = te::model_m(model);
    p->NF = te::model_nf(model);
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) throw std::runtime_error("te_pool needs an sm_100a (Blackwell) device");
    p->n_sm = prop.multiProcessorCount;
    if (cuda_stream) {
      p->stream = (cudaStream_t)cuda_stream;
    } else {
      CK(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
      p->own_stream = true;
    }
    CK(cudaMalloc(&p->d_counters, 4 * sizeof(int)));
    CK(cudaMemsetAsync(p->d_counters, 0, 4 * sizeof(int), p->stream));
    if (const char* cap = std::getenv("TE_GRID_CAP")) p->grid_cap = std::max(0, std::atoi(cap));   // test hook, see te_pool_set_grid_cap
    return p;
  } catch (const std::exception& e) {
    g_err = e.what();
    delete p;
    return nullptr;
  }
}

void te_pool_destroy(te_pool* p) {
  if (!p) return;
  int prev = 0;
  cudaGetDevice(&prev);
  cudaSetDevice(p->device);
  if (p->live.active && p->live.h_ring) {   // a resident live launch waits for the host: tell it to stop
    __atomic_store_n(p->live.h_ring + 258, 1, __ATOMIC_RELEASE);
    p->live.active = false;
  }
  cudaStreamSynchronize(p->stream);
  if (p->h2d_stream) cudaStreamSynchronize(p->h2d_stream);
  if (p->d2h_stream) cudaStreamSynchronize(p->d2h_stream);
  free_buf(p->buf[0]);
  free_buf(p->buf[1]);
  free_mail(p->mb[0]);
  free_mail(p->mb[1]);
  if (p->h_stage) cudaFreeHost(p->h_stage);
  cudaFree(p->action); cudaFree(p->dt_slot); cudaFree(p->tile_flag); cudaFree(p->tile_list);
  cudaFree(p->alive); cudaFree(p->pos); cudaFree(p->srcmap); cudaFree(p->d_counters); cudaFree(p->cub_tmp);
  cudaFree(p->dQ); cudaFree(p->dR); cudaFree(p->dP0); cudaFree(p->dT);
  p->arena.destroy();
  cudaFree(p->live.d_gate);
  if (p->live.h_ring) cudaFreeHost(p->live.h_ring);
  cudaFree(p->prefetch.dev);
  if (p->prefetch.done) cudaEventDestroy(p->prefetch.done);
  for (te_pool::TickSet& ts : p->tick_set) {
    for (cudaEvent_t e : ts.ev) cudaEventDestroy(e);
    if (ts.step_done) cudaEventDestroy(ts.step_done);
    if (ts.d2h_done) cudaEventDestroy(ts.d2h_done);
    cudaFree(ts.meas);
    cudaFree(ts.act);
    cudaFree(ts.pos);
  }
  if (p->h2d_stream) cudaStreamDestroy(p->h2d_stream);
  if (p->d2h_stream) cudaStreamDestroy(p->d2h_stream);
  if (p->own_stream) cudaStreamDestroy(p->stream);
  cudaSetDevice(prev);
  delete p;
}

int te_pool_set_stream(te_pool* p, void* cuda_stream) {
  return guarded(p, [&] {
    CK(cudaStreamSynchronize(p->stream));
    if (p->own_stream) cudaStreamDestroy(p->stream);
    p->own_stream = false;
    if (cuda_stream) {
      p->stream = (cudaStream_t)cuda_stream;
    } else {
      CK(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
      p->own_stream = true;
    }
    return 0;
  });
}

int te_pool_sync(te_pool* p) {
  return guarded(p, [&] {
    CK(cudaStreamSynchronize(p->stream));
    return 0;
  });
}

int te_pool_set_variant(te_pool* p, int variant) {
  if (!p) return -1;
  p->variant = variant;
  return 0;
}

int te_pool_set_grid_cap(te_pool* p, int max_ctas) {
  if (!p || max_ctas < 0) return -1;
  p->grid_cap = max_ctas;
  return 0;
}

int te_pool_reserve(te_pool* p, size_t n_targets) {
  return guarded(p, [&] {
    if (!p->buf[p->cur].tiles) {
      alloc_buf(p, p->buf[p->cur], n_targets);
      ensure_work(p, p->buf[p->cur].cap);
    } else {
      ensure_cur_capacity(p, n_targets);
    }
    ensure_work(p, std::max(n_targets, p->buf[p->cur].cap));   // (a flipped buffer can be larger than the work arrays)
    // the second generation too (every compaction -- erase, merge-add, expiry -- gathers into it): no tick pays for a
    // multi-gigabyte allocation later
    ensure_other_capacity(p, n_targets);
    if (p->mb_on) {
      ensure_mail_cur(p, n_targets);
      ensure_mail_other(p, n_targets);
    }
    return 0;
  });
}

long long te_pool_size(te_pool* p) { return p ? p->n : -1; }

size_t te_pool_device_bytes(te_pool* p) {
  if (!p) return 0;
  size_t b = 0;
  for (int i = 0; i < 2; ++i)
    if (p->buf[i].tiles) b += p->buf[i].cap / te::TILE * tile_doubles(p) * 8 + p->buf[i].cap * (4 + 2 + 8 + 56);
  b += p->wcap * (1 + 8 + 4 + 4 + 4) + p->wcap / te::TILE * 5 + p->cub_bytes;
  return b;
}

int te_pool_register_class(te_pool* p, const double* Q, const double* R, const double* P0) {
  return guarded(p, [&] {
    if (!Q || !R || !P0) throw std::invalid_argument("null model matrix");
    const size_t nn = (size_t)p->N * p->N, mm = (size_t)p->M * p->M;
    for (size_t c = 0; c < p->hQ.size(); ++c)
      if (!std::memcmp(p->hQ[c].data(), Q, nn * 8) && !std::memcmp(p->hR[c].data(), R, mm * 8) && !std::memcmp(p->hP0[c].data(), P0, nn * 8))
        return (int)c;
    if (p->hQ.size() >= 65535) throw std::runtime_error("too many model classes (max 65535)");
    p->hQ.emplace_back(Q, Q + nn);
    p->hR.emplace_back(R, R + mm);
    p->hP0.emplace_back(P0, P0 + nn);
    auto sym = [](const double* A, int n) {
      for (int i = 0; i < n; ++i)
        for (int j = 0; j < i; ++j)
          if (std::memcmp(&A[i * n + j], &A[j * n + i], 8) != 0) return false;
      return true;
    };
    if (!sym(Q, p->N) || !sym(R, p->M) || !sym(P0, p->N)) p->all_sym = false;
    auto decoupled = [](const double* A, int n, int axes) {   // entry (i, j) belongs to axes i % axes and j % axes
      for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j)
          if (i % axes != j % axes && A[i * n + j] != 0.0) return false;
      return true;
    };
    const bool kin = p->model == te::UNIFORM_VELOCITY || p->model == te::UNIFORM_ACCELERATION;
    if (!kin || !decoupled(Q, p->N, 3) || !decoupled(P0, p->N, 3) || !decoupled(R, p->M, p->M)) p->all_axis = false;
    {
      // T = L^-1, R = L L^T (plain FP64 Cholesky, then forward substitution against the identity); zeros if R has no factor
      const int m = p->M;
      std::vector<double> L((size_t)m * m, 0.0), T((size_t)m * m, 0.0);
      bool ok = true;
      for (int j = 0; j < m && ok; ++j) {
        double d = R[j * m + j];
        for (int k = 0; k < j; ++k) d -= L[j * m + k] * L[j * m + k];
        if (!(d > 0.0) || !std::isfinite(d)) { ok = false; break; }
        L[j * m + j] = std::sqrt(d);
        for (int i = j + 1; i < m; ++i) {
          double s2 = R[i * m + j];
          for (int k = 0; k < j; ++k) s2 -= L[i * m + k] * L[j * m + k];
          L[i * m + j] = s2 / L[j * m + j];
        }
      }
      if (ok) {
        for (int c = 0; c < m; ++c)
          for (int i = c; i < m; ++i) {
            double s2 = (i == c) ? 1.0 : 0.0;
            for (int k = c; k < i; ++k) s2 -= L[i * m + k] * T[k * m + c];
            T[i * m + c] = s2 / L[i * m + i];
          }
      } else {
        std::fill(T.begin(), T.end(), 0.0);
        p->whiten_ok = false;
      }
      p->hT.push_back(T);
    }
    upload_classes(p);
    return (int)p->hQ.size() - 1;
  });
}

int te_pool_class_count(te_pool* p) { return p ? (int)p->hQ.size() : -1; }

int te_pool_get_class(te_pool* p, int cls, double* Q, double* R, double* P0) {
  if (!p || cls < 0 || cls >= (int)p->hQ.size()) return -1;
  if (Q) std::memcpy(Q, p->hQ[cls].data(), p->hQ[cls].size() * 8);
  if (R) std::memcpy(R, p->hR[cls].data(), p->hR[cls].size() * 8);
  if (P0) std::memcpy(P0, p->hP0[cls].data(), p->hP0[cls].size() * 8);
  return 0;
}

long long te_pool_add_batch(te_pool* p, long long n, const uint32_t* ids, const uint16_t* cls, const double* t0, const double* p0,
                            const double* v0, const double* a0, const double* p0_scale) {
  return guarded_ll(p, [&]() -> long long {
    if (n <= 0) return 0;
    if (!ids || !p0) throw std::invalid_argument("ids and p0 are required");
    if (p->hQ.empty()) throw std::runtime_error("no model class registered");
    // order the batch by id (first occurrence wins), drop ids that already exist
    std::vector<long long> ord((size_t)n);
    std::iota(ord.begin(), ord.end(), 0LL);
    bool sorted = true;
    for (long long k = 1; k < n && sorted; ++k) sorted = ids[k - 1] < ids[k];
    if (!sorted) std::stable_sort(ord.begin(), ord.end(), [&](long long a, long long b) { return ids[a] < ids[b]; });
    std::vector<long long> keep;
    keep.reserve((size_t)n);
    if (p->n == 0) { p->h_ids.clear(); p->h_ids_valid = true; }
    if (p->n > 0 && !p->h_ids_valid && !p->h_last_valid) sync_host_ids(p);
    const bool append_only = p->n == 0 || ids[ord[0]] > (p->h_ids_valid ? p->h_ids.back() : p->h_last_id);
    if (!append_only) sync_host_ids(p);   // membership test and merge need the whole sorted id array
    for (long long k = 0; k < n; ++k) {
      const long long s = ord[k];
      if (!keep.empty() && ids[keep.back()] == ids[s]) continue;
      if (!append_only && std::binary_search(p->h_ids.begin(), p->h_ids.end(), ids[s])) continue;   // "already exists"
      if (cls && cls[s] >= p->hQ.size()) throw std::invalid_argument("unknown model class in add batch");
      keep.push_back(s);
    }
    const long long na = (long long)keep.size();
    if (na == 0) return 0;
    const bool identity = sorted && na == n;
    // gather payload in id order
    std::vector<uint32_t> g_ids;
    std::vector<uint16_t> g_cls;
    std::vector<double> g_t0, g_p0, g_v0, g_a0, g_sc;
    const uint32_t* s_ids = ids;
    const uint16_t* s_cls = cls;
    const double *s_t0 = t0, *s_p0 = p0, *s_v0 = v0, *s_a0 = a0, *s_sc = p0_scale;
    if (!identity) {
      g_ids.resize(na);
      for (long long k = 0; k < na; ++k) g_ids[k] = ids[keep[k]];
      s_ids = g_ids.data();
      auto gather = [&](const double* src, int w, std::vector<double>& dst) -> const double* {
        if (!src) return nullptr;
        dst.resize((size_t)na * w);
        for (long long k = 0; k < na; ++k) std::memcpy(&dst[(size_t)k * w], src + (size_t)keep[k] * w, w * 8);
        return dst.data();
      };
      s_t0 = gather(t0, 1, g_t0);
      s_p0 = gather(p0, 7, g_p0);
      s_v0 = gather(v0, 6, g_v0);
      s_a0 = gather(a0, 6, g_a0);
      s_sc = gather(p0_scale, 1, g_sc);
      if (cls) {
        g_cls.resize(na);
        for (long long k = 0; k < na; ++k) g_cls[k] = cls[keep[k]];
        s_cls = g_cls.data();
      }
    }
    te::AddData ad{};
    ad.ids = to_dev(p, s_ids, na);
    ad.cls = to_dev(p, s_cls, na);
    ad.t0 = to_dev(p, s_t0, na);
    ad.p0 = to_dev(p, s_p0, na * 7);
    ad.v0 = to_dev(p, s_v0, na * 6);
    ad.a0 = to_dev(p, s_a0, na * 6);
    ad.scale = to_dev(p, s_sc, na);
    if (append_only) {
      if (!p->buf[p->cur].tiles) {
        alloc_buf(p, p->buf[p->cur], (size_t)na);
        ensure_work(p, p->buf[p->cur].cap);
      } else {
        ensure_cur_capacity(p, (size_t)(p->n + na));
      }
      init_append(p, (int)p->n, ad, na);
      if (p->mb_on) {
        ensure_mail_cur(p, (size_t)(p->n + na));
        te::mb_clear_kernel<<<cdiv(na, 256), 256, 0, p->stream>>>(p->mb[p->mb_cur].a, (int)p->n, (int)na);
        CK(cudaGetLastError());
      }
      p->n += na;
      if (p->h_ids_valid) p->h_ids.insert(p->h_ids.end(), s_ids, s_ids + na);
      p->h_last_id = s_ids[na - 1];
      p->h_last_valid = true;
    } else {
      ensure_work(p, (size_t)(p->n + na));
      te::fill_i32_kernel<<<cdiv(p->n, 256), 256, 0, p->stream>>>(p->alive, (int)p->n, 1);
      CK(cudaGetLastError());
      compact_and_merge(p, ad, ad.ids, (int)na, nullptr);
      std::vector<uint32_t> merged(p->h_ids.size() + (size_t)na);
      std::merge(p->h_ids.begin(), p->h_ids.end(), s_ids, s_ids + na, merged.begin());
      p->h_ids.swap(merged);
      p->h_ids_valid = true;
    }
    if (p->mb_on && (!p->orphans.empty() || !p->pending.empty())) attach_mailboxes(p, s_ids, na);
    CK(cudaStreamSynchronize(p->stream));   // host payload vectors go out of scope
    return na;
  });
}

long long te_pool_erase_batch(te_pool* p, long long n, const uint32_t* ids) {
  return guarded_ll(p, [&]() -> long long {
    if (n <= 0 || p->n == 0) return 0;
    if (!ids) throw std::invalid_argument("null ids");
    ensure_work(p, (size_t)p->n);
    uint32_t* d_ids = to_dev(p, ids, n);
    int* slots = lookup_slots(p, d_ids, n);
    if (p->mb_on) demote_mailboxes(p, ids, slots, n);
    te::fill_i32_kernel<<<cdiv(p->n, 256), 256, 0, p->stream>>>(p->alive, (int)p->n, 1);
    te::clear_listed_kernel<<<cdiv(n, 256), 256, 0, p->stream>>>(p->alive, slots, n);
    CK(cudaGetLastError());
    const long long n_old = p->n;
    te::AddData ad{};
    const int alive = compact_and_merge(p, ad, nullptr, 0, nullptr);
    return n_old - alive;
  });
}

long long te_pool_ids(te_pool* p, uint32_t* out, long long cap) {
  return guarded_ll(p, [&]() -> long long {
    sync_host_ids(p);
    if (out) std::memcpy(out, p->h_ids.data(), (size_t)std::min<long long>(cap, p->n) * sizeof(uint32_t));
    return p->n;
  });
}

int te_pool_contains(te_pool* p, uint32_t id) {
  return guarded(p, [&] {
    sync_host_ids(p);
    return std::binary_search(p->h_ids.begin(), p->h_ids.end(), id) ? 1 : 0;
  });
}

int te_pool_class_of(te_pool* p, uint32_t id) {
  return guarded(p, [&] {
    sync_host_ids(p);
    auto it = std::lower_bound(p->h_ids.begin(), p->h_ids.end(), id);
    if (it == p->h_ids.end() || *it != id) throw std::invalid_argument("unknown target id");
    uint16_t c = 0;
    CK(cudaMemcpyAsync(&c, p->buf[p->cur].cold.cls + (it - p->h_ids.begin()), sizeof(uint16_t), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    return (int)c;
  });
}
int te_pool_read_state(te_pool* p, long long n, const uint32_t* ids, double* x, double* P, double* t, long long* n_meas, double* prev_rpy,
                       double* measured_pose) {
  return guarded(p, [&] {
    if (n <= 0) return 0;
    if (!ids && n != p->n) throw std::invalid_argument("ids == NULL requires n == pool size");
    const int N = p->N;
    int* slots = nullptr;
    if (ids) slots = lookup_slots(p, to_dev(p, ids, n), n);
    double* dx = x ? p->arena.get_n<double>((size_t)n * N) : nullptr;
    double* dP = P ? p->arena.get_n<double>((size_t)n * N * N) : nullptr;
    double* dt_ = t ? p->arena.get_n<double>((size_t)n) : nullptr;
    long long* dn = n_meas ? p->arena.get_n<long long>((size_t)n) : nullptr;
    double* dprev = prev_rpy ? p->arena.get_n<double>((size_t)n * 3) : nullptr;
    double* dmp = measured_pose ? p->arena.get_n<double>((size_t)n * 7) : nullptr;
    if (dx) CK(cudaMemsetAsync(dx, 0, (size_t)n * N * 8, p->stream));
    if (dP) CK(cudaMemsetAsync(dP, 0, (size_t)n * N * N * 8, p->stream));
    if (dt_) CK(cudaMemsetAsync(dt_, 0, (size_t)n * 8, p->stream));
    if (dn) CK(cudaMemsetAsync(dn, 0, (size_t)n * 8, p->stream));
    if (dprev) CK(cudaMemsetAsync(dprev, 0, (size_t)n * 24, p->stream));
    if (dmp) CK(cudaMemsetAsync(dmp, 0, (size_t)n * 56, p->stream));
    Buf& b = p->buf[p->cur];
    const int g = cdiv(n, 128);
    switch (p->model) {
      case te::UNIFORM_VELOCITY: te::gather_state_kernel<te::UNIFORM_VELOCITY><<<g, 128, 0, p->stream>>>(b.tiles, b.cold, slots, n, dx, dP, dt_, dn, dprev, dmp, p->lower_stale ? 1 : 0); break;
      case te::UNIFORM_ACCELERATION: te::gather_state_kernel<te::UNIFORM_ACCELERATION><<<g, 128, 0, p->stream>>>(b.tiles, b.cold, slots, n, dx, dP, dt_, dn, dprev, dmp, p->lower_stale ? 1 : 0); break;
      case te::ANGULAR_VELOCITIES: te::gather_state_kernel<te::ANGULAR_VELOCITIES><<<g, 128, 0, p->stream>>>(b.tiles, b.cold, slots, n, dx, dP, dt_, dn, dprev, dmp, p->lower_stale ? 1 : 0); break;
      default: te::gather_state_kernel<te::ANGULAR_RATES><<<g, 128, 0, p->stream>>>(b.tiles, b.cold, slots, n, dx, dP, dt_, dn, dprev, dmp, p->lower_stale ? 1 : 0); break;
    }
    CK(cudaGetLastError());
    if (x) CK(cudaMemcpyAsync(x, dx, (size_t)n * N * 8, cudaMemcpyDeviceToHost, p->stream));
    if (P) CK(cudaMemcpyAsync(P, dP, (size_t)n * N * N * 8, cudaMemcpyDeviceToHost, p->stream));
    if (t) CK(cudaMemcpyAsync(t, dt_, (size_t)n * 8, cudaMemcpyDeviceToHost, p->stream));
    if (n_meas) CK(cudaMemcpyAsync(n_meas, dn, (size_t)n * 8, cudaMemcpyDeviceToHost, p->stream));
    if (prev_rpy) CK(cudaMemcpyAsync(prev_rpy, dprev, (size_t)n * 24, cudaMemcpyDeviceToHost, p->stream));
    if (measured_pose) CK(cudaMemcpyAsync(measured_pose, dmp, (size_t)n * 56, cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    return 0;
  });
}

int te_pool_read_estimates(te_pool* p, long long n, const uint32_t* ids, const double* t1, double* pose7, double* twist6, double* acc6,
                           double* pose6_internal, uint8_t* found) {
  return guarded(p, [&] {
    if (n <= 0) return 0;
    if (!ids && n != p->n) throw std::invalid_argument("ids == NULL requires n == pool size");
    int* slots = nullptr;
    if (ids) slots = lookup_slots(p, to_dev(p, ids, n), n);
    const double* d_t1 = to_dev(p, t1, n);
    double* dpose = pose7 ? p->arena.get_n<double>((size_t)n * 7) : nullptr;
    double* dtw = twist6 ? p->arena.get_n<double>((size_t)n * 6) : nullptr;
    double* dac = acc6 ? p->arena.get_n<double>((size_t)n * 6) : nullptr;
    double* dp6 = pose6_internal ? p->arena.get_n<double>((size_t)n * 6) : nullptr;
    uint8_t* dfound = found ? p->arena.get_n<uint8_t>((size_t)n) : nullptr;
    if (dpose) CK(cudaMemsetAsync(dpose, 0, (size_t)n * 56, p->stream));
    if (dtw) CK(cudaMemsetAsync(dtw, 0, (size_t)n * 48, p->stream));
    if (dac) CK(cudaMemsetAsync(dac, 0, (size_t)n * 48, p->stream));
    if (dp6) CK(cudaMemsetAsync(dp6, 0, (size_t)n * 48, p->stream));
    launch_gather_estimates(p, slots, n, d_t1, dpose, dtw, dac, dp6, dfound, 0);
    if (pose7) CK(cudaMemcpyAsync(pose7, dpose, (size_t)n * 56, cudaMemcpyDeviceToHost, p->stream));
    if (twist6) CK(cudaMemcpyAsync(twist6, dtw, (size_t)n * 48, cudaMemcpyDeviceToHost, p->stream));
    if (acc6) CK(cudaMemcpyAsync(acc6, dac, (size_t)n * 48, cudaMemcpyDeviceToHost, p->stream));
    if (pose6_internal) CK(cudaMemcpyAsync(pose6_internal, dp6, (size_t)n * 48, cudaMemcpyDeviceToHost, p->stream));
    if (found) CK(cudaMemcpyAsync(found, dfound, (size_t)n, cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    return 0;
  });
}

int te_pool_estimates_dev(te_pool* p, double* dev_out) {
  return guarded(p, [&] {
    if (p->n == 0) return 0;
    if (!dev_out) throw std::invalid_argument("null output");
    launch_gather_estimates(p, nullptr, p->n, nullptr, dev_out, nullptr, nullptr, nullptr, nullptr, 1);
    return 0;
  });
}

const uint32_t* te_pool_dev_ids(te_pool* p) { return p ? p->buf[p->cur].cold.ids : nullptr; }

int te_pool_set_stamps(te_pool* p, long long n, const uint32_t* ids, const uint32_t* sec, const uint32_t* nsec) {
  return guarded(p, [&] {
    if (n <= 0 || p->n == 0) return 0;
    if (!ids || !sec || !nsec) throw std::invalid_argument("null stamp arrays");
    uint32_t* d_ids = to_dev(p, ids, n);
    uint32_t* d_sec = to_dev(p, sec, n);
    uint32_t* d_nsec = to_dev(p, nsec, n);
    Buf& b = p->buf[p->cur];
    te::set_stamps_kernel<<<cdiv(n, 256), 256, 0, p->stream>>>(b.cold.ids, (int)p->n, n, d_ids, d_sec, d_nsec, b.cold.last_meas);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(p->stream));
    return 0;
  });
}

int te_pool_stamp_dense(te_pool* p, const uint8_t* dev_action, int default_action, uint32_t sec, uint32_t nsec) {
  return guarded(p, [&] {
    if (p->n == 0) return 0;
    volatile double ns = 1e-9 * (double)nsec;   // toSec (utils.hpp:59-62), never contracted
    const double stamp = (double)sec + ns;
    te::stamp_dense_kernel<<<cdiv(p->n, 256), 256, 0, p->stream>>>(dev_action, default_action, (int)p->n, stamp, p->buf[p->cur].cold.last_meas);
    CK(cudaGetLastError());
    return 0;
  });
}

long long te_pool_expire(te_pool* p, uint32_t now_sec, uint32_t now_nsec, double timeout, uint32_t* erased_out, long long cap) {
  return guarded_ll(p, [&]() -> long long {
    if (p->n == 0) return 0;
    ensure_work(p, (size_t)p->n);
    const long long n_old = p->n;
    // toSec on the host in the same non-contracted arithmetic (utils.hpp:59-62)
    volatile double ns = 1e-9 * (double)now_nsec;
    const double now = (double)now_sec + ns;
    te::expire_flags_kernel<<<cdiv(n_old, 256), 256, 0, p->stream>>>(p->buf[p->cur].cold.last_meas, (int)n_old, now, timeout, p->alive);
    CK(cudaGetLastError());
    uint32_t* d_erased = p->arena.get_n<uint32_t>((size_t)n_old);
    te::AddData ad{};
    const int alive = compact_and_merge(p, ad, nullptr, 0, d_erased);
    const long long n_er = n_old - alive;
    if (n_er > 0 && erased_out && cap > 0)
      CK(cudaMemcpyAsync(erased_out, d_erased, (size_t)std::min(cap, n_er) * sizeof(uint32_t), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    return n_er;
  });
}
}  // extern "C"
