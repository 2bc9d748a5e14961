// te_query_args.h -- the argument rules of the k-nearest and the gating query and of the association, shared by the pool entry points
// (te_pool_nearest_targets / te_pool_gated_targets, te_sweep.cu; te_pool_associate / te_pool_gated_candidates / te_assign_greedy,
// te_assoc.cu) and the managers (TargetManager::nearestTargets / gatedTargets / associate, host/target_manager.cpp).  The manager
// checks them itself because a manager without targets never reaches a pool; one copy keeps both layers' errors and messages the
// same.  Host code only.
#pragma once
#include <cmath>
#include <stdexcept>
#include <string>

namespace te {

// the names a query's messages use for its point array, its bound and its value output
struct QueryNames {
  const char* point;
  const char* bound;
  const char* val_out;
};
constexpr QueryNames NEAREST_ARGS{"point", "radius", "dist_out"};
constexpr QueryNames GATE_ARGS{"z", "gate", "d2_out"};
// association: the detection array and the two outputs of te_pool_associate / te_pool_gated_candidates
constexpr QueryNames ASSOC_ARGS{"det", "id_out", "d2_out"};
constexpr QueryNames CANDIDATE_ARGS{"z", "ids_out", "d2_out"};

// throws std::invalid_argument; t1 may always be NULL, the other arrays only when q == 0 (ids_out / val_out also when k == 0);
// every bound must be >= 0 and not NaN
inline void check_query_args(const QueryNames& names, long long q, const double* point, const double* bound, long long k,
                             const void* ids_out, const double* val_out, const long long* count_out) {
  if (q < 0) throw std::invalid_argument("q must be >= 0");
  if (k < 0 || k > 65536) throw std::invalid_argument("k must be in [0, 65536]");
  if (q == 0) return;
  if (!point || !bound || !count_out)
    throw std::invalid_argument(std::string(names.point) + ", " + names.bound + " and count_out are required");
  if (k > 0 && (!ids_out || !val_out)) throw std::invalid_argument(std::string("ids_out and ") + names.val_out + " are required when k > 0");
  for (long long j = 0; j < q; ++j)
    if (!(bound[j] >= 0.0))
      throw std::invalid_argument(std::string(names.bound) + " must be >= 0 and not NaN (query " + std::to_string(j) + ")");
}

constexpr int ASSOC_MAX_K = 32;

// association of one frame (names: ASSOC_ARGS / CANDIDATE_ARGS): t1 finite; gate >= 0 and finite (+inf has no spatial bound:
// gatedTargets serves it); 1 <= K <= 32; q >= 0; the detections and both outputs required when q > 0 (count_out may be NULL)
inline void check_assoc_args(const QueryNames& names, double t1, long long q, const double* det, double gate, long long K,
                             const void* id_out, const double* d2_out) {
  if (!std::isfinite(t1)) throw std::invalid_argument("t1 must be finite");
  if (!(gate >= 0.0) || std::isinf(gate)) throw std::invalid_argument("gate must be >= 0 and finite");
  if (K < 1 || K > ASSOC_MAX_K) throw std::invalid_argument("K must be in [1, 32]");
  if (q < 0) throw std::invalid_argument("q must be >= 0");
  if (q > 0 && (!det || !id_out || !d2_out))
    throw std::invalid_argument(std::string(names.point) + ", " + names.bound + " and " + names.val_out + " are required");
}

// te_assign_greedy's rows: detection j's rows ids[j][.] / d2[j][.] hold its candidates by (d^2, id), each d^2 >= 0, then rows of
// d^2 -1 (what te_pool_gated_candidates and gatedTargets return)
inline void check_assign_rows(long long q, long long K, const unsigned* ids, const double* d2, const void* id_out, const double* d2_out) {
  if (K < 1 || K > ASSOC_MAX_K) throw std::invalid_argument("K must be in [1, 32]");
  if (q < 0) throw std::invalid_argument("q must be >= 0");
  if (q == 0) return;
  if (!ids || !d2 || !id_out || !d2_out) throw std::invalid_argument("ids, d2, id_out and d2_out are required");
  for (long long j = 0; j < q; ++j) {
    const unsigned* r_id = ids + j * K;
    const double* r_d2 = d2 + j * K;
    bool open = true;
    for (long long r = 0; r < K; ++r) {
      if (!(r_d2[r] >= 0.0)) {
        if (r_d2[r] != -1.0) throw std::invalid_argument("d2 rows hold d^2 >= 0, then -1 (detection " + std::to_string(j) + ")");
        open = false;
        continue;
      }
      if (!open) throw std::invalid_argument("d2 rows hold d^2 >= 0, then -1 (detection " + std::to_string(j) + ")");
      if (r > 0 && (r_d2[r] < r_d2[r - 1] || (r_d2[r] == r_d2[r - 1] && r_id[r] <= r_id[r - 1])))
        throw std::invalid_argument("rows must be ordered by (d2, id) (detection " + std::to_string(j) + ")");
    }
  }
}

}  // namespace te
