// te_nearest_args.h -- the argument rules of the k-nearest query, shared by the pool entry point (te_pool_nearest_targets,
// te_sweep.cu) and the manager (TargetManager::nearestTargets, host/target_manager.cpp).  The manager checks them itself because a
// manager without targets never reaches a pool; one copy keeps both layers' errors and messages the same.  Host code only.
#pragma once
#include <stdexcept>
#include <string>

namespace te {

// throws std::invalid_argument; t1 may always be NULL, the other arrays only when q == 0 (ids_out / dist_out also when k == 0)
inline void check_nearest_args(long long q, const double* point, const double* radius, long long k, const void* ids_out,
                               const double* dist_out, const long long* count_out) {
  if (q < 0) throw std::invalid_argument("q must be >= 0");
  if (k < 0 || k > 65536) throw std::invalid_argument("k must be in [0, 65536]");
  if (q == 0) return;
  if (!point || !radius || !count_out) throw std::invalid_argument("point, radius and count_out are required");
  if (k > 0 && (!ids_out || !dist_out)) throw std::invalid_argument("ids_out and dist_out are required when k > 0");
  for (long long j = 0; j < q; ++j)
    if (!(radius[j] >= 0.0)) throw std::invalid_argument("radius must be >= 0 and not NaN (query " + std::to_string(j) + ")");
}

}  // namespace te
