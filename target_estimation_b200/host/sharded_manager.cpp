// sharded_manager.cpp -- ShardedTargetManager: one TargetManager per GPU of the box behind the reference's TargetManager API
// (/root/reference/include/target_estimation/target_manager.hpp:66-203), owner(id) = id mod G, no collective on the hot path;
// the optional exchange of estimates goes over NCCL (te_group_*, csrc/te_group.cu).  See the class comment in
// include/target_estimation_b200/target_manager.hpp.
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <stdexcept>
#include <thread>

#include "../csrc/te_query_args.h"
#include "rows.hpp"
#include "target_estimation_b200/target_manager.hpp"

namespace target_estimation_b200 {

// one worker thread per shard: a batched call runs on all shards at once (every shard's host-to-device copies, launches and
// read-backs are issued by its own thread against its own device)
class ShardWorkers {
 public:
  explicit ShardWorkers(int n) : n_(n), err_((size_t)n) {
    for (int r = 0; r < n; ++r) th_.emplace_back([this, r] { loop(r); });
  }
  ~ShardWorkers() {
    {
      std::lock_guard<std::mutex> lg(m_);
      stop_ = true;
      ++gen_;
    }
    cv_.notify_all();
    for (auto& t : th_) t.join();
  }
  int size() const { return n_; }
  void run(const std::function<void(int)>& f) {
    {
      std::lock_guard<std::mutex> lg(m_);
      job_ = &f;
      left_ = n_;
      ++gen_;
    }
    cv_.notify_all();
    std::unique_lock<std::mutex> lk(m_);
    done_.wait(lk, [this] { return left_ == 0; });
    job_ = nullptr;
    for (auto& e : err_)
      if (e) {
        std::exception_ptr x = e;
        for (auto& c : err_) c = nullptr;
        std::rethrow_exception(x);
      }
  }

 private:
  void loop(int r) {
    unsigned long seen = 0;
    for (;;) {
      const std::function<void(int)>* job = nullptr;
      {
        std::unique_lock<std::mutex> lk(m_);
        cv_.wait(lk, [&] { return gen_ != seen; });
        seen = gen_;
        if (stop_) return;
        job = job_;
      }
      try {
        (*job)(r);
      } catch (...) {
        err_[(size_t)r] = std::current_exception();
      }
      {
        std::lock_guard<std::mutex> lg(m_);
        if (--left_ == 0) done_.notify_all();
      }
    }
  }
  int n_;
  std::vector<std::thread> th_;
  std::vector<std::exception_ptr> err_;
  std::mutex m_;
  std::condition_variable cv_, done_;
  const std::function<void(int)>* job_ = nullptr;
  unsigned long gen_ = 0;
  int left_ = 0;
  bool stop_ = false;
};

namespace {
// page-locked staging of one shard (the shard's batched calls copy from it at PCIe speed)
void stageReserve(double*& meas, unsigned char*& action, size_t& cap, size_t n) {
  if (n <= cap) return;
  const size_t want = n + n / 4 + 1024;
  if (meas) { te_host_unregister(meas); std::free(meas); }
  if (action) { te_host_unregister(action); std::free(action); }
  meas = (double*)std::malloc(want * 7 * sizeof(double));
  action = (unsigned char*)std::malloc(want);
  if (!meas || !action) throw std::bad_alloc();
  te_host_register(meas, want * 7 * sizeof(double));   // (a failed registration leaves pageable memory: slower, still correct)
  te_host_register(action, want);
  cap = want;
}
}  // namespace

ShardedTargetManager::ShardedTargetManager(const std::string& file, int n_shards, const int* devices)
    : ShardedTargetManager(file, n_shards, devices, [&file](int d) { return new TargetManager(file, d); }) {}

ShardedTargetManager::ShardedTargetManager(const std::string& file, int n_shards, const int* devices,
                                           const std::function<TargetManager*(int)>& make_shard)
    : TargetManager(file, devices ? devices[0] : 0) {
  if (n_shards <= 0) throw std::invalid_argument("a sharded manager needs at least one shard");
  const int n_dev = te_device_count();
  if (n_dev <= 0) throw std::runtime_error("no CUDA device available");
  for (int r = 0; r < n_shards; ++r) {
    const int d = devices ? devices[r] : r;
    if (d < 0 || d >= n_dev) throw std::invalid_argument("no such CUDA device: " + std::to_string(d));
    devices_.push_back(d);
    shard_.emplace_back(make_shard(d));
    shard_.back()->quiet = true;
  }
  stage_.resize((size_t)n_shards);
  workers_.reset(new ShardWorkers(n_shards));
  const unsigned hw = std::thread::hardware_concurrency();
  const int n_route = (int)std::max<unsigned>((unsigned)n_shards, std::min<unsigned>(hw ? hw : 1u, 16u));
  routers_.reset(new ShardWorkers(n_route));
  quiet = true;
}

ShardedTargetManager::~ShardedTargetManager() {
  workers_.reset();
  routers_.reset();
  if (group_) te_group_destroy(group_);
  for (Stage& s : stage_) {
    if (s.meas) { te_host_unregister(s.meas); std::free(s.meas); }
    if (s.action) { te_host_unregister(s.action); std::free(s.action); }
  }
}

void ShardedTargetManager::forEachShard(const std::function<void(int)>& f) {
  if (shard_.size() == 1) { f(0); return; }
  workers_->run(f);
}

// ---- per-id calls: the owner's ------------------------------------------------------------------------------------------
void ShardedTargetManager::init(const unsigned int& id, const double& dt0, const double& t0, const Vector7d& p0, const Vector6d& v0, const Vector6d& a0) {
  shard_[(size_t)owner(id)]->init(id, dt0, t0, p0, v0, a0);
}
void ShardedTargetManager::init(const target_t& type, const unsigned int& id, const double& dt0, const double& t0, const MatrixXd& Q, const MatrixXd& R,
                                const MatrixXd& P0, const Vector7d& p0, const Vector6d& v0, const Vector6d& a0) {
  shard_[(size_t)owner(id)]->init(type, id, dt0, t0, Q, R, P0, p0, v0, a0);
}
bool ShardedTargetManager::update(const unsigned int& id, const double& dt, const Vector7d& meas) { return shard_[(size_t)owner(id)]->update(id, dt, meas); }
bool ShardedTargetManager::update(const unsigned int& id, const double& dt) { return shard_[(size_t)owner(id)]->update(id, dt); }
void ShardedTargetManager::update(const double& dt) {
  for (auto& s : shard_) s->update(dt);   // asynchronous launches: the devices predict concurrently
}
bool ShardedTargetManager::erase(const unsigned int& id) { return shard_[(size_t)owner(id)]->erase(id); }
TargetInterface::Ptr ShardedTargetManager::getTarget(const unsigned int& id) { return shard_[(size_t)owner(id)]->getTarget(id); }
bool ShardedTargetManager::getTargetPose(const unsigned int& id, Vector7d& pose) { return shard_[(size_t)owner(id)]->getTargetPose(id, pose); }
bool ShardedTargetManager::getTargetTwist(const unsigned int& id, Vector6d& twist) { return shard_[(size_t)owner(id)]->getTargetTwist(id, twist); }
bool ShardedTargetManager::getTargetAcceleration(const unsigned int& id, Vector6d& acc) { return shard_[(size_t)owner(id)]->getTargetAcceleration(id, acc); }
long long ShardedTargetManager::getNumberMeasurements(const unsigned int& id) { return shard_[(size_t)owner(id)]->getNumberMeasurements(id); }
void ShardedTargetManager::log() {
  for (auto& s : shard_) s->log();
}
void ShardedTargetManager::flush() {
  for (auto& s : shard_) s->flush();
}
void ShardedTargetManager::watch(long long n, const unsigned* ids, size_t max_samples) {
  std::vector<std::vector<unsigned>> per(shard_.size());
  for (long long k = 0; k < n; ++k) per[(size_t)owner(ids[k])].push_back(ids[k]);
  for (size_t r = 0; r < shard_.size(); ++r) shard_[r]->watch((long long)per[r].size(), per[r].data(), max_samples);
}

std::vector<unsigned int> ShardedTargetManager::getAvailableTargets() {
  std::vector<unsigned int> all;
  for (auto& s : shard_) {   // every shard's list is ascending: merge pairwise
    std::vector<unsigned int> part = s->getAvailableTargets();
    const size_t mid = all.size();
    all.insert(all.end(), part.begin(), part.end());
    std::inplace_merge(all.begin(), all.begin() + (long)mid, all.end());
  }
  return all;
}

// ---- batched calls: routed by owner, all shards at once -------------------------------------------------------------------------
long long ShardedTargetManager::initBatch(target_t type, const MatrixXd& Q, const MatrixXd& R, const MatrixXd& P0, long long n, const unsigned* ids,
                                          double dt0, const double* t0, const double* p0, const double* v0, const double* a0, const double* p0_scale) {
  if (n <= 0) return 0;
  const std::vector<std::vector<long long>> rows = rowsByOwner(n, ids);
  std::atomic<long long> added{0};
  forEachShard([&](int r) {
    const std::vector<long long>& mine = rows[(size_t)r];
    if (mine.empty()) return;
    std::vector<unsigned> s_ids;
    std::vector<double> s_t0, s_p0, s_v0, s_a0, s_sc;
    added += shard_[(size_t)r]->initBatch(type, Q, R, P0, (long long)mine.size(), gatherRows<1>(ids, mine, s_ids), dt0, gatherRows<1>(t0, mine, s_t0),
                                          gatherRows<7>(p0, mine, s_p0), gatherRows<6>(v0, mine, s_v0), gatherRows<6>(a0, mine, s_a0),
                                          gatherRows<1>(p0_scale, mine, s_sc));
  });
  return added.load();
}

long long ShardedTargetManager::updateBatch(long long n, const unsigned* ids, double dt, const double* meas, const unsigned char* action) {
  if (n <= 0) return 0;
  const unsigned G = (unsigned)shard_.size();
  const FastMod owner_of(G);
  if (G == 1) return shard_[0]->updateBatch(n, ids, dt, meas, action);
  requireMeasurements(n, meas, action);   // before any shard steps
  const std::vector<size_t> total = routeOnHost(
      n, ids,
      [&](int r, size_t m) {   // (each worker sizes its own shard's staging: page-locking is the slow part and runs in parallel)
        Stage& st = stage_[(size_t)r];
        st.ids.resize(m);
        stageReserve(st.meas, st.action, st.cap, m);
      },
      [&](int, long long lo, long long hi, size_t* at) {
        for (long long k = lo; k < hi; ++k) {
          const unsigned r = owner_of(ids[k]);
          Stage& st = stage_[r];
          const size_t j = at[r]++;
          st.ids[j] = ids[k];
          if (meas) std::memcpy(st.meas + 7 * j, meas + 7 * (size_t)k, 56);
          st.action[j] = action ? action[k] : (unsigned char)TE_ACT_UPDATE;
        }
      });
  std::atomic<long long> applied{0};
  forEachShard([&](int r) {
    Stage& st = stage_[(size_t)r];
    if (total[(size_t)r] == 0) return;
    applied += shard_[(size_t)r]->updateBatch((long long)total[(size_t)r], st.ids.data(), dt, meas ? st.meas : nullptr, st.action);
  });
  return applied.load();
}

// Routing = a parallel stable partition of the batch by owner, every access sequential.  Routing thread t (there are as many as
// the host offers, at most 16, at least G) takes the t-th contiguous chunk of the records: (1) it counts the owners in its chunk; the
// prefix sums give chunk t a place in every shard's staging behind the chunks before it; (2) it streams its chunk once more and
// appends every record to its owner's staging (G write streams per worker).  Inside a shard the records keep the caller's order
// (chunks are ordered, and so is each chunk), so the records of one id stay in sequence.  (A pass per shard over the whole batch,
// each picking its own records out, gathered 56-byte records at a stride of G records: 300 ms for 33 M records on 8 shards.)
std::vector<size_t> ShardedTargetManager::routeOnHost(long long n, const unsigned* ids, const std::function<void(int, size_t)>& reserve,
                                                      const std::function<void(int, long long, long long, size_t*)>& scatter) {
  const unsigned G = (unsigned)shard_.size();
  const FastMod owner_of(G);
  const unsigned T = (unsigned)routers_->size();   // routing threads (>= G)
  std::vector<size_t> count((size_t)T * G, 0);     // [chunk t][owner r]
  auto chunk_lo = [&](unsigned t) { return (long long)((__int128)n * t / T); };
  const std::function<void(int)> count_pass = [&](int t) {
    std::vector<size_t> c(G, 0);   // (local: neighbouring rows of `count` share cache lines)
    for (long long k = chunk_lo((unsigned)t), e = chunk_lo((unsigned)t + 1); k < e; ++k) ++c[owner_of(ids[k])];
    std::copy(c.begin(), c.end(), count.begin() + (long)t * G);
  };
  routers_->run(count_pass);
  std::vector<size_t> offset((size_t)T * G, 0), total(G, 0);
  for (unsigned r = 0; r < G; ++r)
    for (unsigned t = 0; t < T; ++t) {
      offset[(size_t)t * G + r] = total[r];
      total[r] += count[(size_t)t * G + r];
    }
  forEachShard([&](int r) { reserve(r, total[(size_t)r]); });
  const std::function<void(int)> scatter_pass = [&](int t) {
    std::vector<size_t> at(offset.begin() + (long)t * G, offset.begin() + (long)(t + 1) * G);
    scatter(t, chunk_lo((unsigned)t), chunk_lo((unsigned)t + 1), at.data());
  };
  routers_->run(scatter_pass);
  return total;
}

std::vector<std::vector<long long>> ShardedTargetManager::rowsByOwner(long long n, const unsigned* ids) {
  const FastMod owner_of((unsigned)shard_.size());
  std::vector<std::vector<long long>> rows(shard_.size());
  routeOnHost(
      n, ids, [&](int r, size_t m) { rows[(size_t)r].resize(m); },
      [&](int, long long lo, long long hi, size_t* at) {
        for (long long k = lo; k < hi; ++k) {
          const unsigned r = owner_of(ids[k]);
          rows[r][at[r]++] = k;
        }
      });
  return rows;
}

long long ShardedTargetManager::eraseBatch(long long n, const unsigned* ids) {
  if (n <= 0) return 0;
  const std::vector<std::vector<long long>> rows = rowsByOwner(n, ids);
  std::atomic<long long> erased{0};
  forEachShard([&](int r) {
    const std::vector<long long>& mine = rows[(size_t)r];
    std::vector<unsigned> s_ids;
    if (!mine.empty()) erased += shard_[(size_t)r]->eraseBatch((long long)mine.size(), gatherRows<1>(ids, mine, s_ids));
  });
  return erased.load();
}

void ShardedTargetManager::getEstimatesBatch(long long n, const unsigned* ids, const double* t1, double* pose7, double* twist6, double* acc6,
                                             unsigned char* found) {
  if (n <= 0) return;
  if (shard_.size() == 1) return shard_[0]->getEstimatesBatch(n, ids, t1, pose7, twist6, acc6, found);
  const std::vector<std::vector<long long>> rows = rowsByOwner(n, ids);
  forEachShard([&](int r) {
    const std::vector<long long>& mine = rows[(size_t)r];
    const size_t m = mine.size();
    if (m == 0) return;
    std::vector<unsigned> s_ids;
    std::vector<double> s_t1, po(pose7 ? m * 7 : 0), tw(twist6 ? m * 6 : 0), ac(acc6 ? m * 6 : 0);
    std::vector<unsigned char> fo(m, 0);
    shard_[(size_t)r]->getEstimatesBatch((long long)m, gatherRows<1>(ids, mine, s_ids), gatherRows<1>(t1, mine, s_t1), pose7 ? po.data() : nullptr,
                                         twist6 ? tw.data() : nullptr, acc6 ? ac.data() : nullptr, fo.data());
    // rows of different shards are disjoint: no two threads write the same output row
    scatterRows<7>(pose7, mine, po.data());
    scatterRows<6>(twist6, mine, tw.data());
    scatterRows<6>(acc6, mine, ac.data());
    scatterRows<1>(found, mine, fo.data());
  });
}

long long ShardedTargetManager::nearestTargets(long long q, const double* t1, const double* point, const double* radius, long long k,
                                               unsigned* ids_out, double* dist_out, long long* count_out) {
  te::check_query_args(te::NEAREST_ARGS, q, point, radius, k, ids_out, dist_out, count_out);
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  if (q == 0) return 0;
  flush();
  std::vector<TargetManager*> shards;
  for (auto& s : shard_) shards.push_back(s.get());
  return nearest_rows_.run(
      shards, [this](const std::function<void(int)>& f) { forEachShard(f); }, q, k,
      [&](te_pool* p, unsigned* ids, double* dist, long long* count) {
        return te_pool_nearest_targets(p, q, t1, point, radius, k, ids, dist, count);
      },
      ids_out, dist_out, count_out);
}

long long ShardedTargetManager::gatedTargets(long long q, const double* t1, const double* z, const double* gate, long long k,
                                             unsigned* ids_out, double* d2_out, long long* count_out) {
  te::check_query_args(te::GATE_ARGS, q, z, gate, k, ids_out, d2_out, count_out);
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  if (q == 0) return 0;
  flush();
  std::vector<TargetManager*> shards;
  for (auto& s : shard_) shards.push_back(s.get());
  return gated_rows_.run(
      shards, [this](const std::function<void(int)>& f) { forEachShard(f); }, q, k,
      [&](te_pool* p, unsigned* ids, double* d2, long long* count) { return te_pool_gated_targets(p, q, t1, z, gate, k, ids, d2, count); },
      ids_out, d2_out, count_out);
}

long long ShardedTargetManager::associate(double t1, long long q, const double* det, double gate, int K, int apply, unsigned* id_out,
                                          double* d2_out, long long* count_out) {
  te::check_assoc_args(te::ASSOC_ARGS, t1, q, det, gate, K, id_out, d2_out);
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  if (q == 0) return 0;
  flush();
  std::vector<TargetManager*> shards;
  for (auto& s : shard_) shards.push_back(s.get());
  return associateOver(
      shards, [this](const std::function<void(int)>& f) { forEachShard(f); }, t1, q, det, gate, K, apply, id_out, d2_out, count_out,
      [&](long long n, const unsigned* ids, const double* rec) {
        const std::vector<std::vector<long long>> rows = rowsByOwner(n, ids);
        forEachShard([&](int r) {
          const std::vector<long long>& mine = rows[(size_t)r];
          if (mine.empty()) return;
          std::vector<unsigned> s_ids;
          std::vector<double> s_rec;
          shard_[(size_t)r]->updateAt(t1, (long long)mine.size(), gatherRows<1>(ids, mine, s_ids), gatherRows<7>(rec, mine, s_rec));
        });
      });
}

// ---- dense ticks: shard-major records, every shard's slice on its own device at once ---------------------------------------------
std::vector<unsigned int> ShardedTargetManager::denseIds() {
  std::vector<unsigned int> all;
  for (auto& s : shard_) {
    std::vector<unsigned int> part = s->getAvailableTargets();
    all.insert(all.end(), part.begin(), part.end());
  }
  return all;
}

long long ShardedTargetManager::updateDense(double dt, const double* meas, int meas_stride, const unsigned char* action, double* est_pos_out) {
  std::vector<long long> off(shard_.size() + 1, 0);
  for (size_t r = 0; r < shard_.size(); ++r) off[r + 1] = off[r] + (long long)shard_[r]->size();
  forEachShard([&](int r) {
    const long long o = off[(size_t)r];
    if (off[(size_t)r + 1] == o) return;
    shard_[(size_t)r]->updateDense(dt, meas ? meas + o * meas_stride : nullptr, meas_stride, action ? action + o : nullptr, est_pos_out ? est_pos_out + 3 * o : nullptr);
  });
  return off.back();
}

long long ShardedTargetManager::updateDenseAsync(double dt, const double* meas, int meas_stride, const unsigned char* action, double* est_pos_out) {
  // enqueueing costs microseconds per shard: one thread issues all of them, the devices then run concurrently
  long long o = 0;
  for (auto& s : shard_) {
    const long long n = (long long)s->size();
    if (n > 0) s->updateDenseAsync(dt, meas ? meas + o * meas_stride : nullptr, meas_stride, action ? action + o : nullptr, est_pos_out ? est_pos_out + 3 * o : nullptr);
    o += n;
  }
  return o;
}

void ShardedTargetManager::updateDenseWait(int lag) {
  for (auto& s : shard_) s->updateDenseWait(lag);
}

// ---- the optional exchange of estimates ----------------------------------------------------------------------------------------
te_group* ShardedTargetManager::group() {
  if (!group_) {
    group_ = te_group_create((int)devices_.size(), devices_.data());
    if (!group_) throw std::runtime_error(te_last_error());
  }
  return group_;
}

bool ShardedTargetManager::gatherUsesNccl() { return te_group_uses_nccl(group()) == 1; }

long long ShardedTargetManager::gatherEstimates(std::vector<unsigned>* ids, std::vector<double>* records13, int publisher) {
  if (publisher < 0 || publisher >= (int)shard_.size()) throw std::invalid_argument("no such shard");
  gatherUsesNccl();   // (creates the group)
  flush();
  if (ids) ids->clear();
  if (records13) records13->clear();
  long long total = 0;
  gather_ms_ = 0.0;
  std::vector<te_pool*> pools(shard_.size());
  for (int type = 0; type < 4; ++type) {
    bool any = false;
    for (size_t r = 0; r < shard_.size(); ++r) {
      pools[r] = (shard_[r]->heldTypes() >> type) & 1u ? shard_[r]->poolOf(type, false) : nullptr;
      any = any || pools[r];
    }
    if (!any) continue;
    const long long n = te_group_allgather_estimates(group_, pools.data(), nullptr);
    if (n < 0) throw std::runtime_error(te_last_error());
    if (ids || records13) {
      const size_t o = (size_t)total;
      if (ids) ids->resize(o + (size_t)n);
      if (records13) records13->resize((o + (size_t)n) * 13);
      if (te_group_fetch(group_, publisher, records13 ? records13->data() + o * 13 : nullptr, ids ? ids->data() + o : nullptr, n) < 0)
        throw std::runtime_error(te_last_error());
    } else if (te_group_sync(group_) < 0) {
      throw std::runtime_error(te_last_error());
    }
    gather_ms_ += te_group_last_gather_ms(group_);
    total += n;
  }
  return total;
}

}  // namespace target_estimation_b200
