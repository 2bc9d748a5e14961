// te_sweep.cu -- te_pool_earliest_intersections, te_pool_nearest_targets and te_pool_gated_targets of include/te_pool.h: the k
// earliest sphere intercepts, the k nearest targets inside a sphere and the k targets of smallest Mahalanobis distance inside a gate,
// over every target of a pool, selected on the device (kernels in te_sweep.cuh).  All three produce one key per (query, slot) and
// share the selection below.  Only q x k rows and q counts cross PCIe.
#include <cub/device/device_segmented_sort.cuh>

#include "te_query_args.h"
#include "te_pool_internal.cuh"
#include "te_sweep.cuh"

using namespace tehost;

namespace {
// keys of one chunk: at most this many (query, target) pairs, 256 MB
constexpr long long SWEEP_PAIRS = 1LL << 25;

// delta of every slot for one sphere into keys (as doubles): the kernel and arguments of te_isolver_query_dense, so every bit is
// te_isolver_query's
template <int TYPE>
void launch_deltas(te_pool* p, int n, const double* t1, const double* origin, const double* radius, unsigned long long* keys) {
  te::isolver_kernel<TYPE><<<cdiv(n, 128), 128, 0, p->stream>>>(p->buf[p->cur].tiles, nullptr, nullptr, n, t1, origin, radius, nullptr, nullptr,
                                                                 te::IsolverState{}, reinterpret_cast<double*>(keys), nullptr, nullptr);
}

// the answer of q queries over no candidate: zero counts and sentinel rows
long long no_rows(long long q, long long k, uint32_t* ids_out, double* val_out, long long* count_out) {
  std::fill(count_out, count_out + q, 0LL);
  if (k > 0) {
    std::fill(ids_out, ids_out + q * k, 0xFFFFFFFFu);
    std::fill(val_out, val_out + q * k, -1.0);
  }
  return 0;
}

// The selection both queries share, over a pool of n > 0 targets.  Queries run in chunks of C sized from the pool;
// produce(j0, nq, keys, counts) enqueues on the pool's stream the keys of queries j0 .. j0 + nq - 1 (keys + c * n: one key per slot,
// SWEEP_MISS for no candidate; a candidate's key is the bits of a non-negative value, -0.0 allowed) and adds the candidates of query
// j0 + c to counts[c].  Per query: radix select of the k-th smallest (rank(key), slot), collect, two stable segmented sorts, rows of
// (id, value) ordered by (value, id) and sentinel rows after them, copied to the host with the counts.  Returns the total count.
template <class Produce>
long long select_rows(te_pool* p, long long q, long long k, uint32_t* ids_out, double* val_out, long long* count_out, Produce&& produce) {
  const long long n = p->n;
  const int C = (int)std::max(1LL, std::min({q, (long long)te::SWEEP_MAX_CHUNK, SWEEP_PAIRS / n}));
  const unsigned cap = (unsigned)k + te::SWEEP_SLACK;
  auto* keys = p->arena.get_n<unsigned long long>((size_t)C * n);
  auto* counts = p->arena.get_n<unsigned long long>(C);
  auto* sel = p->arena.get_n<te::SweepSel>(C);
  auto* hist = p->arena.get_n<unsigned>((size_t)C * te::SWEEP_BINS);
  auto* count = p->arena.get_n<unsigned>(C);
  int* seg = p->arena.get_n<int>(2 * (size_t)C + 1);   // begin offsets | end offsets | overflow flag
  int* overflow = seg + 2 * C;
  unsigned long long *rank_a = nullptr, *rank_b = nullptr;
  unsigned *slot_a = nullptr, *slot_b = nullptr;
  uint32_t* d_ids = nullptr;
  double* d_val = nullptr;
  void* sort_tmp = nullptr;
  size_t sort_bytes = 0;
  const int items = C * (int)cap;
  if (k > 0) {
    rank_a = p->arena.get_n<unsigned long long>(items);
    rank_b = p->arena.get_n<unsigned long long>(items);
    slot_a = p->arena.get_n<unsigned>(items);
    slot_b = p->arena.get_n<unsigned>(items);
    d_ids = p->arena.get_n<uint32_t>((size_t)C * k);
    d_val = p->arena.get_n<double>((size_t)C * k);
    size_t by_slot = 0, by_rank = 0;
    CK(cub::DeviceSegmentedSort::StableSortPairs(nullptr, by_slot, slot_a, slot_b, rank_a, rank_b, items, C, seg, seg + C, p->stream));
    CK(cub::DeviceSegmentedSort::StableSortPairs(nullptr, by_rank, rank_a, rank_b, slot_a, slot_b, items, C, seg, seg + C, p->stream));
    sort_bytes = std::max(by_slot, by_rank);
    sort_tmp = p->arena.get(sort_bytes);
  }
  CK(cudaMemsetAsync(hist, 0, (size_t)C * te::SWEEP_BINS * sizeof(unsigned), p->stream));
  CK(cudaMemsetAsync(overflow, 0, sizeof(int), p->stream));
  const int bx = std::max(1, std::min(cdiv(n, 256 * 4), (p->n_sm * 8 + C - 1) / C));
  for (long long j0 = 0; j0 < q; j0 += C) {
    const int nq = (int)std::min<long long>(C, q - j0);
    CK(cudaMemsetAsync(counts, 0, (size_t)nq * sizeof(unsigned long long), p->stream));
    produce(j0, nq, keys, counts);
    CK(cudaGetLastError());
    if (k > 0) {
      te::sweep_init_kernel<<<1, te::SWEEP_MAX_CHUNK, 0, p->stream>>>(nq, (unsigned)k, counts, sel, count);
      for (int pass = 0; pass < te::SWEEP_PASSES; ++pass) {
        te::sweep_hist_kernel<<<dim3(bx, nq), 256, 0, p->stream>>>(keys, (int)n, sel, te::sweep_shift(pass), hist);
        te::sweep_select_kernel<<<nq, 1024, 0, p->stream>>>(hist, sel, te::sweep_shift(pass));
      }
      te::sweep_collect_kernel<<<dim3(bx, nq), 256, 0, p->stream>>>(keys, (int)n, sel, cap, count, rank_a, slot_a);
      te::sweep_segments_kernel<<<1, te::SWEEP_MAX_CHUNK, 0, p->stream>>>(nq, cap, count, seg, seg + C, overflow);
      CK(cudaGetLastError());
      // (slot, then stable by rank: ties of the value come out in ascending slot = ascending id)
      CK(cub::DeviceSegmentedSort::StableSortPairs(sort_tmp, sort_bytes, slot_a, slot_b, rank_a, rank_b, nq * (int)cap, nq, seg, seg + C, p->stream));
      CK(cub::DeviceSegmentedSort::StableSortPairs(sort_tmp, sort_bytes, rank_b, rank_a, slot_b, slot_a, nq * (int)cap, nq, seg, seg + C, p->stream));
      te::sweep_output_kernel<<<dim3(cdiv(k, 256), nq), 256, 0, p->stream>>>((int)k, sel, slot_a, cap, keys, (int)n, p->buf[p->cur].cold.ids,
                                                                              d_ids, d_val);
      CK(cudaGetLastError());
      CK(cudaMemcpyAsync(ids_out + j0 * k, d_ids, (size_t)nq * k * sizeof(uint32_t), cudaMemcpyDeviceToHost, p->stream));
      CK(cudaMemcpyAsync(val_out + j0 * k, d_val, (size_t)nq * k * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    }
    CK(cudaMemcpyAsync(count_out + j0, counts, (size_t)nq * sizeof(long long), cudaMemcpyDeviceToHost, p->stream));
  }
  int h_overflow = 0;
  CK(cudaMemcpyAsync(&h_overflow, overflow, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
  CK(cudaStreamSynchronize(p->stream));
  if (h_overflow) throw std::logic_error("te_sweep: candidate overflow (selection invariant broken)");
  long long total = 0;
  for (long long j = 0; j < q; ++j) total += count_out[j];
  return total;
}

unsigned long long bits_of(double v) {
  unsigned long long b;
  std::memcpy(&b, &v, 8);
  return b;
}

}  // namespace

namespace tehost {
// gate_prep_kernel of the pool's model over every slot: t1 NULL = no predict
template <int TYPE>
void launch_gate_prep_t(te_pool* p, int n, const double* t1, double* chol) {
  const Buf& b = p->buf[p->cur];
  te::gate_prep_kernel<TYPE><<<cdiv(n, 256), 256, 0, p->stream>>>(n, b.tiles, b.cold.cls, p->dQ, p->dR, t1 ? 1 : 0, t1 ? *t1 : 0.0, chol);
}
void launch_gate_prep(te_pool* p, int n, const double* t1, double* chol) {
  switch (p->model) {
    case te::UNIFORM_VELOCITY: launch_gate_prep_t<te::UNIFORM_VELOCITY>(p, n, t1, chol); break;
    case te::UNIFORM_ACCELERATION: launch_gate_prep_t<te::UNIFORM_ACCELERATION>(p, n, t1, chol); break;
    case te::ANGULAR_VELOCITIES: launch_gate_prep_t<te::ANGULAR_VELOCITIES>(p, n, t1, chol); break;
    default: launch_gate_prep_t<te::ANGULAR_RATES>(p, n, t1, chol); break;
  }
}
}  // namespace tehost

extern "C" long long te_pool_earliest_intersections(te_pool* p, long long q, const double* t1, const double* origin, const double* radius,
                                                    long long k, uint32_t* ids_out, double* delta_out, long long* hits_out) {
  return guarded_ll(p, [&]() -> long long {
    if (q < 0) throw std::invalid_argument("q must be >= 0");
    if (k < 0 || k > 65536) throw std::invalid_argument("k must be in [0, 65536]");
    if (q == 0) return 0;
    if (!t1 || !origin || !radius || !hits_out) throw std::invalid_argument("t1, origin, radius and hits_out are required");
    if (k > 0 && (!ids_out || !delta_out)) throw std::invalid_argument("ids_out and delta_out are required when k > 0");
    const long long n = p->n;
    // uniform-velocity and angular-velocity targets carry no acceleration: the t^4 coefficient is 0 and no target intercepts
    if (n == 0 || p->model == te::UNIFORM_VELOCITY || p->model == te::ANGULAR_VELOCITIES) return no_rows(q, k, ids_out, delta_out, hits_out);
    std::vector<double> sph((size_t)q * 5);   // t1, origin, radius of sphere j as one record
    for (long long j = 0; j < q; ++j) {
      sph[5 * j] = t1[j];
      std::memcpy(&sph[5 * j + 1], origin + 3 * j, 24);
      sph[5 * j + 4] = radius[j];
    }
    const double* d_sph = to_dev(p, sph.data(), sph.size());
    double* b_t1 = p->arena.get_n<double>((size_t)n * 5);   // one sphere broadcast to every slot: isolver_kernel's inputs
    double* b_origin = b_t1 + n;
    double* b_radius = b_t1 + 4 * n;
    return select_rows(p, q, k, ids_out, delta_out, hits_out, [&](long long j0, int nq, unsigned long long* keys, unsigned long long* hits) {
      for (int c = 0; c < nq; ++c) {
        unsigned long long* kc = keys + (size_t)c * n;
        te::sweep_broadcast_kernel<<<cdiv(n, 256), 256, 0, p->stream>>>((int)n, d_sph + 5 * (j0 + c), b_t1, b_origin, b_radius);
        if (p->model == te::UNIFORM_ACCELERATION) launch_deltas<te::UNIFORM_ACCELERATION>(p, (int)n, b_t1, b_origin, b_radius, kc);
        else launch_deltas<te::ANGULAR_RATES>(p, (int)n, b_t1, b_origin, b_radius, kc);
        te::sweep_key_kernel<<<cdiv(n, 256), 256, 0, p->stream>>>((int)n, kc, hits + c);
      }
    });
  });
}

extern "C" long long te_pool_nearest_targets(te_pool* p, long long q, const double* t1, const double* point, const double* radius, long long k,
                                             uint32_t* ids_out, double* dist_out, long long* count_out) {
  return guarded_ll(p, [&]() -> long long {
    te::check_query_args(te::NEAREST_ARGS, q, point, radius, k, ids_out, dist_out, count_out);
    if (q == 0) return 0;
    const long long n = p->n;
    if (n == 0) return no_rows(q, k, ids_out, dist_out, count_out);
    // The positions come from gather_estimates_kernel in its dense form -- the kernel te_pool_read_estimates runs -- so they are
    // getEstimatedPose(t1) bit for bit (a second copy of derive_outputs would be contracted differently, see sweep_broadcast_kernel).
    // Consecutive queries at the same t1 (every query when t1 is NULL) share one gather.
    double* pose7 = p->arena.get_n<double>((size_t)n * 7);
    double* b_t1 = t1 ? p->arena.get_n<double>((size_t)n) : nullptr;   // t1 of the query broadcast to every slot
    bool gathered = false;
    unsigned long long gathered_t1 = 0;
    return select_rows(p, q, k, ids_out, dist_out, count_out, [&](long long j0, int nq, unsigned long long* keys, unsigned long long* inside) {
      for (int c = 0; c < nq; ++c) {
        const long long j = j0 + c;
        if (!gathered || (t1 && bits_of(t1[j]) != gathered_t1)) {
          if (t1) te::fill_dt_kernel<<<cdiv(n, 256), 256, 0, p->stream>>>(b_t1, (int)n, t1[j]);
          launch_gather_estimates(p, nullptr, n, b_t1, pose7, nullptr, nullptr, nullptr, nullptr, 0);
          gathered = true;
          gathered_t1 = t1 ? bits_of(t1[j]) : 0;
        }
        te::near_key_kernel<<<cdiv(n, 256), 256, 0, p->stream>>>((int)n, pose7, point[3 * j], point[3 * j + 1], point[3 * j + 2], radius[j],
                                                                 keys + (size_t)c * n, inside + c);
      }
    });
  });
}

extern "C" long long te_pool_gated_targets(te_pool* p, long long q, const double* t1, const double* z, const double* gate, long long k,
                                           uint32_t* ids_out, double* d2_out, long long* count_out) {
  return guarded_ll(p, [&]() -> long long {
    te::check_query_args(te::GATE_ARGS, q, z, gate, k, ids_out, d2_out, count_out);
    if (q == 0) return 0;
    const long long n = p->n;
    if (n == 0) return no_rows(q, k, ids_out, d2_out, count_out);
    // positions as te_pool_nearest_targets gathers them; consecutive queries at the same t1 (every query when t1 is NULL) share one
    // gather and one factor of S per slot
    double* pose7 = p->arena.get_n<double>((size_t)n * 7);
    double* chol = p->arena.get_n<double>((size_t)n * 6);
    double* b_t1 = t1 ? p->arena.get_n<double>((size_t)n) : nullptr;
    bool prepared = false;
    unsigned long long prepared_t1 = 0;
    return select_rows(p, q, k, ids_out, d2_out, count_out, [&](long long j0, int nq, unsigned long long* keys, unsigned long long* inside) {
      for (int c = 0; c < nq; ++c) {
        const long long j = j0 + c;
        if (!prepared || (t1 && bits_of(t1[j]) != prepared_t1)) {
          if (t1) te::fill_dt_kernel<<<cdiv(n, 256), 256, 0, p->stream>>>(b_t1, (int)n, t1[j]);
          launch_gather_estimates(p, nullptr, n, b_t1, pose7, nullptr, nullptr, nullptr, nullptr, 0);
          launch_gate_prep(p, (int)n, t1 ? t1 + j : nullptr, chol);
          prepared = true;
          prepared_t1 = t1 ? bits_of(t1[j]) : 0;
        }
        te::gate_key_kernel<<<cdiv(n, 256), 256, 0, p->stream>>>((int)n, pose7, chol, z[3 * j], z[3 * j + 1], z[3 * j + 2], gate[j],
                                                                 keys + (size_t)c * n, inside + c);
      }
    });
  });
}
