// te_assoc.cu -- te_pool_associate, te_pool_gated_candidates, te_assign_greedy and te_pool_update_at of include/te_pool.h: one
// frame of unlabelled position detections gated against a pool through a grid index, assigned greedily on the device, and the
// assigned targets updated at the frame's time (kernels in te_assoc.cuh).  Only the detections go to the device and only the q
// rows of the answer come back.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "te_assoc.cuh"
#include "te_pool_internal.cuh"
#include "te_query_args.h"

using namespace tehost;

namespace {

// what the last association call of a pool saw (te_pool_assoc_stats)
struct AssocStats {
  long long levels = 0, every = 0, candidates = 0, rounds = 0;
};
void note_stats(te_pool* p, const AssocStats& s) {
  p->assoc_stats[0] = s.levels;
  p->assoc_stats[1] = s.every;
  p->assoc_stats[2] = s.candidates;
  p->assoc_stats[3] = s.rounds;
}

// device candidate rows of q detections (position det[j * stride + 0 .. 2]) over the pool: slot_out / d2_out [q][K], count [q]
struct Cand {
  unsigned* slot;
  double* d2;
  long long* count;
};

template <int TYPE>
void launch_box(te_pool* p, int n, const double* pose7, const double* chol, double t1, double sg, uint8_t* kind, te::AssocGrid* g) {
  te::assoc_box_kernel<TYPE><<<cdiv(n, 256), 256, 0, p->stream>>>(n, p->buf[p->cur].tiles, pose7, chol, t1, sg, kind, g);
}

Cand candidates(te_pool* p, double t1, long long q, const double* d_det, int stride, double gate, int K, AssocStats& st) {
  const int n = (int)p->n;
  Cand c;
  c.slot = p->arena.get_n<unsigned>((size_t)q * K);
  c.d2 = p->arena.get_n<double>((size_t)q * K);
  c.count = p->arena.get_n<long long>((size_t)q);
  // positions and factors at t1: the gating query's kernels, so d^2 is gatedTargets' bit for bit
  double* pose7 = p->arena.get_n<double>((size_t)n * 7);
  double* chol = p->arena.get_n<double>((size_t)n * 6);
  double* b_t1 = p->arena.get_n<double>((size_t)n);
  te::fill_dt_kernel<<<cdiv(n, 256), 256, 0, p->stream>>>(b_t1, n, t1);
  launch_gather_estimates(p, nullptr, n, b_t1, pose7, nullptr, nullptr, nullptr, nullptr, 0);
  launch_gate_prep(p, n, &t1, chol);
  // the grid
  const double sg = std::sqrt(gate);
  uint8_t* kind = p->arena.get_n<uint8_t>((size_t)n);
  auto* g = p->arena.get_n<te::AssocGrid>(1);
  te::AssocGrid g0{};
  for (int a = 0; a < 3; ++a) g0.lo_min[a] = ~0ull;
  g0.w_min = ~0ull;
  CK(cudaMemcpyAsync(g, &g0, sizeof(g0), cudaMemcpyHostToDevice, p->stream));
  switch (p->model) {
    case te::UNIFORM_VELOCITY: launch_box<te::UNIFORM_VELOCITY>(p, n, pose7, chol, t1, sg, kind, g); break;
    case te::UNIFORM_ACCELERATION: launch_box<te::UNIFORM_ACCELERATION>(p, n, pose7, chol, t1, sg, kind, g); break;
    case te::ANGULAR_VELOCITIES: launch_box<te::ANGULAR_VELOCITIES>(p, n, pose7, chol, t1, sg, kind, g); break;
    default: launch_box<te::ANGULAR_RATES>(p, n, pose7, chol, t1, sg, kind, g); break;
  }
  te::assoc_grid_kernel<<<1, 1, 0, p->stream>>>(g);
  const long long n_keys = (long long)te::ASSOC_CELLS_PER_SLOT * n;
  if (n_keys >= (1LL << 31)) throw std::invalid_argument("association: 8 x pool size must be below 2^31");
  auto* keys_a = p->arena.get_n<unsigned long long>((size_t)n_keys);
  auto* keys_b = p->arena.get_n<unsigned long long>((size_t)n_keys);
  auto* vals_a = p->arena.get_n<unsigned>((size_t)n_keys);
  auto* vals_b = p->arena.get_n<unsigned>((size_t)n_keys);
  auto* every = p->arena.get_n<unsigned>((size_t)n);
  te::assoc_cell_kernel<<<cdiv(n, 256), 256, 0, p->stream>>>(n, pose7, chol, sg, kind, g, keys_a, vals_a, every);
  CK(cudaGetLastError());
  size_t tmp_bytes = 0;
  CK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys_a, keys_b, vals_a, vals_b, (int)n_keys, 0, 64, p->stream));
  void* tmp = p->arena.get(tmp_bytes);
  CK(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, keys_a, keys_b, vals_a, vals_b, (int)n_keys, 0, 64, p->stream));
  te::assoc_lookup_kernel<<<cdiv(q * 32, 256), 256, 0, p->stream>>>((int)q, d_det, stride, gate, K, pose7, chol, g, keys_b, vals_b, n_keys,
                                                                   every, c.slot, c.d2, c.count);
  CK(cudaGetLastError());
  te::AssocGrid hg;
  CK(cudaMemcpyAsync(&hg, g, sizeof(hg), cudaMemcpyDeviceToHost, p->stream));
  CK(cudaStreamSynchronize(p->stream));
  st.levels = hg.levels > 0 ? __builtin_popcount(hg.level_mask) : 0;
  st.every = hg.n_every;
  return c;
}

// greedy matching of q detections with K rows each (target key tgt[j][r], d^2 d2[j][r]; d^2 < 0 = no edge; a detection's rows in
// (d^2, key) order) on the pool's device: det_match[j] = the assigned row of j or -1.  Returns the number of rounds.
int* match(te_pool* p, long long q, int K, const unsigned* tgt, const double* d2, AssocStats& st) {
  const long long E = q * K;
  if (E >= (1LL << 31)) throw std::invalid_argument("association: q x K must be below 2^31");
  auto* dkey_a = p->arena.get_n<unsigned long long>((size_t)E);
  auto* dkey_b = p->arena.get_n<unsigned long long>((size_t)E);
  auto* idx_a = p->arena.get_n<unsigned>((size_t)E);
  auto* idx_b = p->arena.get_n<unsigned>((size_t)E);
  int* head = p->arena.get_n<int>((size_t)E);
  int* tix = p->arena.get_n<int>((size_t)E);
  int* row_tgt = p->arena.get_n<int>((size_t)E);
  int* seg_begin = p->arena.get_n<int>((size_t)E);
  int* seg_end = p->arena.get_n<int>((size_t)E);
  int* tgt_ptr = p->arena.get_n<int>((size_t)E);
  int* tgt_best = p->arena.get_n<int>((size_t)E);
  int* tgt_match = p->arena.get_n<int>((size_t)E);
  int* det_ptr = p->arena.get_n<int>((size_t)q);
  int* det_best = p->arena.get_n<int>((size_t)q);
  int* det_match = p->arena.get_n<int>((size_t)q);
  auto* matched = p->arena.get_n<unsigned long long>(1);
  size_t b1 = 0, b2 = 0, b3 = 0;
  CK(cub::DeviceRadixSort::SortPairs(nullptr, b1, dkey_a, dkey_b, idx_a, idx_b, (int)E, 0, 64, p->stream));
  CK(cub::DeviceScan::InclusiveSum(nullptr, b3, head, tix, (int)E, p->stream));
  b2 = std::max(b1, b3);
  void* tmp = p->arena.get(b2);
  // 1. edges sorted by (d^2, j), then stably by target: (target, d^2, j); a dense index per target
  te::assoc_edge_init_kernel<<<cdiv(E, 256), 256, 0, p->stream>>>(E, d2, dkey_a, idx_a);
  CK(cub::DeviceRadixSort::SortPairs(tmp, b1, dkey_a, dkey_b, idx_a, idx_b, (int)E, 0, 64, p->stream));
  te::assoc_edge_tkey_kernel<<<cdiv(E, 256), 256, 0, p->stream>>>(E, idx_b, d2, tgt, dkey_a);
  CK(cub::DeviceRadixSort::SortPairs(tmp, b1, dkey_a, dkey_b, idx_b, idx_a, (int)E, 0, 33, p->stream));
  te::assoc_edge_head_kernel<<<cdiv(E, 256), 256, 0, p->stream>>>(E, dkey_b, head);
  CK(cub::DeviceScan::InclusiveSum(tmp, b3, head, tix, (int)E, p->stream));
  te::assoc_edge_seg_kernel<<<cdiv(E, 256), 256, 0, p->stream>>>(E, K, dkey_b, tix, idx_a, seg_begin, seg_end, tgt_ptr, tgt_match, row_tgt);
  CK(cudaMemsetAsync(det_ptr, 0, (size_t)q * sizeof(int), p->stream));
  CK(cudaMemsetAsync(det_match, 0xff, (size_t)q * sizeof(int), p->stream));
  CK(cudaMemsetAsync(matched, 0, sizeof(unsigned long long), p->stream));
  CK(cudaGetLastError());
  // 2. rounds of mutual best edges until one matches nothing
  unsigned long long total = 0;
  int rounds = 0;
  for (;;) {
    ++rounds;
    te::assoc_propose_kernel<<<cdiv(std::max(q, E), 256), 256, 0, p->stream>>>((int)q, K, E, tix + E - 1, row_tgt, idx_a, seg_end, det_match,
                                                                               tgt_match, det_ptr, det_best, tgt_ptr, tgt_best);
    te::assoc_match_kernel<<<cdiv(q, 256), 256, 0, p->stream>>>((int)q, det_ptr, det_best, tgt_best, det_match, tgt_match, matched);
    CK(cudaGetLastError());
    unsigned long long now = 0;
    CK(cudaMemcpyAsync(&now, matched, sizeof(now), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    if (now == total) break;
    total = now;
  }
  st.rounds = rounds;
  return det_match;
}

// the q x K rows and counts to the host; slots become ids
void rows_to_host(te_pool* p, long long q, int K, const Cand& c, uint32_t* ids_out, double* d2_out, long long* count_out) {
  auto* d_ids = p->arena.get_n<uint32_t>((size_t)q * K);
  const uint32_t* cold_ids = p->buf[p->cur].cold.ids;
  te::assoc_slot_ids_kernel<<<cdiv(q * K, 256), 256, 0, p->stream>>>(q * K, c.slot, cold_ids, d_ids);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(ids_out, d_ids, (size_t)q * K * sizeof(uint32_t), cudaMemcpyDeviceToHost, p->stream));
  CK(cudaMemcpyAsync(d2_out, c.d2, (size_t)q * K * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
  if (count_out) CK(cudaMemcpyAsync(count_out, c.count, (size_t)q * sizeof(long long), cudaMemcpyDeviceToHost, p->stream));
  CK(cudaStreamSynchronize(p->stream));
}

// the update of te_pool_update_at over device arrays (act NULL = every op): dt of every op from its slot's time, refused as a whole
// when one is not >= 0, then te_pool_step_ids' scatter and step
long long update_at(te_pool* p, long long n, const uint32_t* d_ids, double t1, const double* d_meas, const uint8_t* d_act) {
  if (n <= 0 || p->n == 0) return 0;
  double* d_dt = p->arena.get_n<double>((size_t)n);
  int* bad = p->arena.get_n<int>(1);
  CK(cudaMemsetAsync(bad, 0, sizeof(int), p->stream));
  const Buf& b = p->buf[p->cur];
  const int g = cdiv(n, 256);
  switch (p->model) {
    case te::UNIFORM_VELOCITY: te::assoc_dt_kernel<te::UNIFORM_VELOCITY><<<g, 256, 0, p->stream>>>(b.tiles, b.cold.ids, (int)p->n, n, d_ids, d_act, t1, d_dt, bad); break;
    case te::UNIFORM_ACCELERATION: te::assoc_dt_kernel<te::UNIFORM_ACCELERATION><<<g, 256, 0, p->stream>>>(b.tiles, b.cold.ids, (int)p->n, n, d_ids, d_act, t1, d_dt, bad); break;
    case te::ANGULAR_VELOCITIES: te::assoc_dt_kernel<te::ANGULAR_VELOCITIES><<<g, 256, 0, p->stream>>>(b.tiles, b.cold.ids, (int)p->n, n, d_ids, d_act, t1, d_dt, bad); break;
    default: te::assoc_dt_kernel<te::ANGULAR_RATES><<<g, 256, 0, p->stream>>>(b.tiles, b.cold.ids, (int)p->n, n, d_ids, d_act, t1, d_dt, bad); break;
  }
  CK(cudaGetLastError());
  int h_bad = 0;
  CK(cudaMemcpyAsync(&h_bad, bad, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
  CK(cudaStreamSynchronize(p->stream));
  if (h_bad) throw std::invalid_argument("a target's time is later than t1 or NaN: nothing applied");
  return step_ops(p, n, d_ids, d_dt, 0.0, d_meas, d_act);
}

}  // namespace

extern "C" long long te_pool_gated_candidates(te_pool* p, double t1, long long q, const double* z, double gate, int K, uint32_t* ids_out,
                                              double* d2_out, long long* count_out) {
  return guarded_ll(p, [&]() -> long long {
    te::check_assoc_args(te::CANDIDATE_ARGS, t1, q, z, gate, K, ids_out, d2_out);
    if (q == 0) return 0;
    AssocStats st;
    long long total = 0;
    if (p->n == 0) {
      std::fill(ids_out, ids_out + q * K, 0xFFFFFFFFu);
      std::fill(d2_out, d2_out + q * K, -1.0);
      if (count_out) std::fill(count_out, count_out + q, 0LL);
    } else {
      const double* d_z = to_dev(p, z, (size_t)q * 3);
      std::vector<long long> cnt((size_t)q);
      const Cand c = candidates(p, t1, q, d_z, 3, gate, K, st);
      rows_to_host(p, q, K, c, ids_out, d2_out, cnt.data());
      for (long long j = 0; j < q; ++j) total += cnt[(size_t)j];
      if (count_out) std::copy(cnt.begin(), cnt.end(), count_out);
    }
    st.candidates = total;
    note_stats(p, st);
    return total;
  });
}

extern "C" long long te_assign_greedy(te_pool* p, long long q, int K, const uint32_t* ids, const double* d2, uint32_t* id_out, double* d2_out) {
  return guarded_ll(p, [&]() -> long long {
    te::check_assign_rows(q, K, ids, d2, id_out, d2_out);
    if (q == 0) return 0;
    AssocStats st;
    const uint32_t* d_ids = to_dev(p, ids, (size_t)q * K);
    const double* d_d2 = to_dev(p, d2, (size_t)q * K);
    int* det_match = match(p, q, K, d_ids, d_d2, st);
    auto* o_ids = p->arena.get_n<uint32_t>((size_t)q);
    auto* o_d2 = p->arena.get_n<double>((size_t)q);
    te::assoc_out_kernel<<<cdiv(q, 256), 256, 0, p->stream>>>((int)q, K, det_match, d_ids, d_d2, nullptr, o_ids, o_d2, nullptr);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(id_out, o_ids, (size_t)q * sizeof(uint32_t), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaMemcpyAsync(d2_out, o_d2, (size_t)q * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    long long assigned = 0;
    for (long long j = 0; j < q; ++j) assigned += d2_out[j] >= 0.0;
    note_stats(p, st);
    return assigned;
  });
}

extern "C" long long te_pool_update_at(te_pool* p, long long n, const uint32_t* ids, double t1, const double* meas) {
  return guarded_ll(p, [&]() -> long long {
    if (n < 0) throw std::invalid_argument("n must be >= 0");
    if (!std::isfinite(t1)) throw std::invalid_argument("t1 must be finite");
    if (n > 0 && (!ids || !meas)) throw std::invalid_argument("ids and meas are required");
    if (n == 0 || p->n == 0) return 0;
    return update_at(p, n, to_dev(p, ids, (size_t)n), t1, to_dev(p, meas, (size_t)n * 7), nullptr);
  });
}

extern "C" long long te_pool_associate(te_pool* p, double t1, long long q, const double* det, double gate, int K, int apply, uint32_t* id_out,
                                       double* d2_out, long long* count_out) {
  return guarded_ll(p, [&]() -> long long {
    te::check_assoc_args(te::ASSOC_ARGS, t1, q, det, gate, K, id_out, d2_out);
    if (q == 0) return 0;
    AssocStats st;
    if (p->n == 0) {
      std::fill(id_out, id_out + q, 0xFFFFFFFFu);
      std::fill(d2_out, d2_out + q, -1.0);
      if (count_out) std::fill(count_out, count_out + q, 0LL);
      note_stats(p, st);
      return 0;
    }
    const double* d_det = to_dev(p, det, (size_t)q * 7);
    const Cand c = candidates(p, t1, q, d_det, 7, gate, K, st);
    int* det_match = match(p, q, K, c.slot, c.d2, st);
    auto* o_ids = p->arena.get_n<uint32_t>((size_t)q);
    auto* o_d2 = p->arena.get_n<double>((size_t)q);
    auto* o_act = p->arena.get_n<uint8_t>((size_t)q);
    te::assoc_out_kernel<<<cdiv(q, 256), 256, 0, p->stream>>>((int)q, K, det_match, c.slot, c.d2, p->buf[p->cur].cold.ids, o_ids, o_d2, o_act);
    CK(cudaGetLastError());
    // (the rows come back before the update: the update does not change them, and a refused update leaves nothing applied)
    CK(cudaMemcpyAsync(id_out, o_ids, (size_t)q * sizeof(uint32_t), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaMemcpyAsync(d2_out, o_d2, (size_t)q * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    std::vector<long long> cnt((size_t)q);
    CK(cudaMemcpyAsync(cnt.data(), c.count, (size_t)q * sizeof(long long), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    long long assigned = 0, total = 0;
    for (long long j = 0; j < q; ++j) {
      assigned += d2_out[j] >= 0.0;
      total += cnt[(size_t)j];
    }
    if (count_out) std::copy(cnt.begin(), cnt.end(), count_out);
    st.candidates = total;
    if (apply && assigned > 0) {
      const long long applied = update_at(p, q, o_ids, t1, d_det, o_act);
      if (applied != assigned) throw std::logic_error("te_pool_associate: " + std::to_string(applied) + " of " + std::to_string(assigned) + " updates applied");
    }
    note_stats(p, st);
    return assigned;
  });
}

extern "C" int te_pool_assoc_stats(te_pool* p, long long* out) {
  return guarded(p, [&] {
    if (!out) throw std::invalid_argument("null output");
    std::copy(p->assoc_stats, p->assoc_stats + 4, out);
    return 0;
  });
}
