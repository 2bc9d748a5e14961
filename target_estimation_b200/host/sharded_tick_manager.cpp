// sharded_tick_manager.cpp -- ShardedTickTargetManager: the node loop of RosTargetManager (src/target_manager_ros.cpp:26-92) over
// every GPU of the box, /tf messages routed to the owners on the devices (te_group_route_records).  See the class comment in
// include/target_estimation_b200/target_manager.hpp.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <stdexcept>

#include "target_estimation_b200/target_manager.hpp"

namespace target_estimation_b200 {

namespace {
// grow-only output whose storage is page-locked while it lasts: the shards' read-backs into it run at PCIe speed
template <class T> void reservePinned(std::vector<T>& v, void*& pinned, size_t n) {
  if (v.capacity() >= n) return;
  if (pinned) te_host_unregister(pinned);
  pinned = nullptr;
  v.clear();
  v.reserve(n + n / 4);
  if (v.capacity() * sizeof(T) >= (1u << 20) && te_host_register(v.data(), v.capacity() * sizeof(T)) == 0) pinned = v.data();
}
}  // namespace

ShardedTickTargetManager::ShardedTickTargetManager(const std::string& yaml_file, int n_shards, const int* devices)
    : ShardedTargetManager(yaml_file, n_shards, devices, [&yaml_file](int d) { return new TickTargetManager(yaml_file, d); }),
      force_host_route_(std::getenv("TE_SHARD_HOST_ROUTE") != nullptr) {
  host_stage_.resize((size_t)n_shards);
}

ShardedTickTargetManager::~ShardedTickTargetManager() {
  for (void* p : pub_pinned_)
    if (p) te_host_unregister(p);
}

void ShardedTickTargetManager::setExpirationTime(double t) {
  if (!(t >= 0.0)) throw std::invalid_argument("expiration time must be >= 0 (assert of src/target_manager_ros.cpp:101)");
  for (int r = 0; r < shards(); ++r) tickShard(r).setExpirationTime(t);
}

double ShardedTickTargetManager::time() const {   // every shard ticks every time: one clock
  return static_cast<const TickTargetManager&>(*shard_[0]).time();
}

size_t ShardedTickTargetManager::mailboxCount() {
  std::vector<size_t> n((size_t)shards(), 0);
  forEachShard([&](int r) { n[(size_t)r] = tickShard(r).mailboxCount(); });
  size_t total = 0;
  for (size_t k : n) total += k;
  return total;
}

void ShardedTickTargetManager::measurementCallBack(long long n, const char* const* frames, const uint32_t* sec, const uint32_t* nsec,
                                                   const double* poses) {
  // parsed over the whole message: the first unparsable frame ends the message for every shard, as it ends the reference's loop
  std::vector<unsigned> ids;
  std::vector<uint32_t> s, ns;
  std::vector<double> p;
  parseFrames(token_name_, n, frames, sec, nsec, poses, ids, s, ns, p);
  measurementCallBackIds((long long)ids.size(), ids.data(), s.data(), ns.data(), p.data());
}

void ShardedTickTargetManager::measurementCallBackIds(long long n, const unsigned* ids, const uint32_t* sec, const uint32_t* nsec,
                                                      const double* poses) {
  if (n <= 0) return;
  const int G = shards();
  // every shard flushes its queued by-hand calls and says whether all its mailboxes live on the device
  std::vector<te_pool*> pools((size_t)G, nullptr);
  forEachShard([&](int r) { pools[(size_t)r] = tickShard(r).devicePool(); });
  const bool on_device = !force_host_route_ && std::all_of(pools.begin(), pools.end(), [](te_pool* p) { return p != nullptr; });
  if (on_device) {
    te_group* g = group();
    if (te_group_route_records(g, pools.data(), n, ids, sec, nsec, poses, nullptr) < 0) throw std::runtime_error(te_last_error());
    forEachShard([&](int r) {
      long long m = 0;
      const uint32_t *d_ids = nullptr, *d_sec = nullptr, *d_nsec = nullptr;
      const double* d_poses = nullptr;
      if (te_group_routed(g, r, &m, &d_ids, &d_sec, &d_nsec, &d_poses) < 0) throw std::runtime_error(te_last_error());
      tickShard(r).ingestDev(m, d_ids, d_sec, d_nsec, d_poses);
    });
    return;
  }
  // host route: the router threads partition the message by owner, then every shard splits its records per id as one manager does
  const FastMod owner_of((unsigned)G);
  const std::vector<size_t> total = routeOnHost(
      n, ids,
      [&](int r, size_t m) {
        HostStage& st = host_stage_[(size_t)r];
        st.ids.resize(m);
        st.sec.resize(m);
        st.nsec.resize(m);
        st.poses.resize(m * 7);
      },
      [&](int, long long lo, long long hi, size_t* at) {
        for (long long k = lo; k < hi; ++k) {
          const unsigned r = owner_of(ids[k]);
          HostStage& st = host_stage_[r];
          const size_t j = at[r]++;
          st.ids[j] = ids[k];
          st.sec[j] = sec[k];
          st.nsec[j] = nsec[k];
          std::memcpy(&st.poses[7 * j], poses + 7 * (size_t)k, 56);
        }
      });
  forEachShard([&](int r) {
    const HostStage& st = host_stage_[(size_t)r];
    if (total[(size_t)r] > 0)
      tickShard(r).measurementCallBackIds((long long)total[(size_t)r], st.ids.data(), st.sec.data(), st.nsec.data(), st.poses.data());
  });
}

void ShardedTickTargetManager::tick(const double& dt, uint32_t now_sec, uint32_t now_nsec, std::vector<unsigned>* erased) {
  if (!(dt >= 0.0)) throw std::invalid_argument("dt must be >= 0");
  const int G = shards();
  std::vector<std::vector<unsigned>> gone((size_t)G);
  std::vector<long long> n_pub((size_t)G, 0);
  const bool pub = publish;
  forEachShard([&](int r) {
    TickTargetManager& s = tickShard(r);
    s.advance(dt, now_sec, now_nsec, &gone[(size_t)r]);
    if (pub) n_pub[(size_t)r] = s.publishCount();
  });
  if (erased) {   // every shard's list is ascending and the shards' ids are disjoint: merge pairwise
    erased->clear();
    for (const auto& part : gone) {
      const size_t mid = erased->size();
      erased->insert(erased->end(), part.begin(), part.end());
      std::inplace_merge(erased->begin(), erased->begin() + (long)mid, erased->end());
    }
  }
  if (!pub) {
    pub_ids_.clear();
    pub_poses_.clear();
    return;
  }
  std::vector<long long> off((size_t)G + 1, 0);
  for (int r = 0; r < G; ++r) off[(size_t)r + 1] = off[(size_t)r] + n_pub[(size_t)r];
  const size_t n = (size_t)off[(size_t)G];
  reservePinned(pub_ids_, pub_pinned_[0], n);
  reservePinned(pub_poses_, pub_pinned_[1], n * 7);
  pub_ids_.resize(n);
  pub_poses_.resize(n * 7);
  // shard-major: every shard's worker reads its ids and poses straight into its slice
  forEachShard([&](int r) {
    const long long o = off[(size_t)r];
    tickShard(r).publishInto(pub_ids_.data() + o, pub_poses_.data() + 7 * o, n_pub[(size_t)r]);
  });
}

}  // namespace target_estimation_b200
