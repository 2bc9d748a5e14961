// rows.hpp -- the gather and scatter of the host's batched calls: a batch split by model type (TargetManager::rowsByType) or by owner
// (ShardedTargetManager::routeOnHost) is a list of row indices into the caller's arrays, and every field of W elements a row moves
// through these two.
#pragma once
#include <cstring>
#include <vector>

namespace target_estimation_b200 {

// rows[i] of src (W elements each) into buf[i]; returns buf's data, or NULL for a NULL source
template <int W, class T>
const T* gatherRows(const T* src, const std::vector<long long>& rows, std::vector<T>& buf) {
  if (!src) return nullptr;
  buf.resize(rows.size() * W);
  for (size_t i = 0; i < rows.size(); ++i) std::memcpy(&buf[i * W], src + (size_t)rows[i] * W, W * sizeof(T));
  return buf.data();
}

// src[i] (W elements each) into row rows[i] of dst; nothing for a NULL destination
template <int W, class T>
void scatterRows(T* dst, const std::vector<long long>& rows, const T* src) {
  if (!dst) return;
  for (size_t i = 0; i < rows.size(); ++i) std::memcpy(dst + (size_t)rows[i] * W, src + i * W, W * sizeof(T));
}

}  // namespace target_estimation_b200
