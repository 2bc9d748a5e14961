// te_query_args.h -- the argument rules of the k-nearest and the gating query, shared by the pool entry points
// (te_pool_nearest_targets / te_pool_gated_targets, te_sweep.cu) and the managers (TargetManager::nearestTargets / gatedTargets,
// host/target_manager.cpp).  The manager checks them itself because a manager without targets never reaches a pool; one copy keeps
// both layers' errors and messages the same.  Host code only.
#pragma once
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

}  // namespace te
