// tick_manager.cpp -- RosTargetManager's tick / mailbox / expiry semantics without ROS
// (/root/reference/include/target_estimation/target_manager_ros.hpp:74-134, src/target_manager_ros.cpp:6-107),
// driving the device pool with one batch per tick instead of one call per id.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <stdexcept>

#include "target_estimation_b200/target_manager.hpp"

namespace target_estimation_b200 {

double toSec(uint32_t sec, uint32_t nsec) {   // utils.hpp:59-62: (double)sec + 1e-9*(double)nsec, two roundings
  volatile double ns = 1e-9 * (double)nsec;
  return (double)sec + ns;
}

void Measurement::update(const StampedPose& tr) {   // target_manager_ros.hpp:96-115
  const double current_time_stamp = toSec(tr.sec, tr.nsec);
  const double prev_time_stamp = toSec(tr_.sec, tr_.nsec);
  if (current_time_stamp > prev_time_stamp) {   // new measurement
    new_meas_ = true;
    last_meas_time_ = current_time_stamp;
    acc_sec_ = tr.sec;
    acc_nsec_ = tr.nsec;
    stamp_dirty_ = true;
  } else {
    new_meas_ = false;
  }
  tr_ = tr;
}

TickTargetManager::TickTargetManager(target_t type, const MatrixXd& Q, const MatrixXd& R, const MatrixXd& P, int device)
    : TargetManager(device), type_(type), Q_(Q), P_(P), R_(R), token_name_("target"), t_(0.0), expiration_time_(1000.0) {}   // :6-24

// (a manager built from a model file also carries it as its default model, like TargetManager(file): by-hand init(id, ...) works)
TickTargetManager::TickTargetManager(const std::string& yaml_file, int device)
    : TargetManager(yaml_file, device), type_(UNIFORM_VELOCITY), token_name_("target"), t_(0.0), expiration_time_(1000.0) {
  if (!loadYamlFile(yaml_file, Q_, R_, P_, type_)) throw std::runtime_error("Can not load the Cov Matrices!");   // :19-23
}

TickTargetManager::~TickTargetManager() {
  if (pub_pinned_) te_host_unregister(pub_pinned_);
}

void TickTargetManager::setExpirationTime(double t) {
  if (!(t >= 0.0)) throw std::invalid_argument("expiration time must be >= 0 (assert of src/target_manager_ros.cpp:101)");
  expiration_time_ = t;
}

// The mailboxes live on the device, beside the slots of the pool of type_ (te_pool_mailbox_*, include/te_pool.h).  Only ids
// the manager knows under ANOTHER model type (created by hand through TargetManager::init) cannot be fed from that pool:
// they keep a host Measurement in measurements_ and go through the by-id loop of tickForeign().
te_pool* TickTargetManager::tickPool() {
  te_pool* pool = poolOf((int)type_, true);
  if (cls_ < 0) cls_ = registerClass((int)type_, Q_, R_, P_);
  return pool;
}

void TickFrontEnd::parseFrames(const std::string& token, long long n, const char* const* frames, const uint32_t* sec, const uint32_t* nsec,
                               const double* poses, std::vector<unsigned>& ids, std::vector<uint32_t>& s, std::vector<uint32_t>& ns,
                               std::vector<double>& p) {   // :26-39
  // frame names -> ids; the loop ends at the first frame that carries the token but does not parse (e.g. the node's own
  // "<token>_filt_<id>" output frames, SURVEY.md H10); frames without the token are skipped
  ids.clear(); s.clear(); ns.clear(); p.clear();
  ids.reserve((size_t)n); s.reserve((size_t)n); ns.reserve((size_t)n); p.reserve((size_t)n * 7);
  for (long long i = 0; i < n; ++i) {
    const std::string name(frames[i]);
    if (name.find(token) != std::string::npos) {
      unsigned id;
      if (!getId(name, id)) break;
      ids.push_back(id);
      s.push_back(sec[i]);
      ns.push_back(nsec[i]);
      p.insert(p.end(), poses + 7 * i, poses + 7 * i + 7);
    }
  }
}

void TickTargetManager::measurementCallBack(long long n, const char* const* frames, const uint32_t* sec, const uint32_t* nsec,
                                            const double* poses) {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  std::vector<unsigned> ids;
  std::vector<uint32_t> s, ns;
  std::vector<double> p;
  parseFrames(token_name_, n, frames, sec, nsec, poses, ids, s, ns, p);
  measurementCallBackIds((long long)ids.size(), ids.data(), s.data(), ns.data(), p.data());
}

// an id the manager knows under another model type, or a host mailbox, may be named: the records must be split per id
bool TickTargetManager::foreignPossible(te_pool* pool) { return !measurements_.empty() || targets_.size() != (size_t)te_pool_size(pool); }

te_pool* TickTargetManager::devicePool() {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  flushLocked();
  te_pool* pool = tickPool();
  return foreignPossible(pool) ? nullptr : pool;
}

void TickTargetManager::ingestDev(long long n, const uint32_t* dev_ids, const uint32_t* dev_sec, const uint32_t* dev_nsec, const double* dev_poses) {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  if (n <= 0) return;
  if (te_pool_mailbox_ingest_dev(tickPool(), n, dev_ids, dev_sec, dev_nsec, dev_poses) < 0) throw std::runtime_error(te_last_error());
}

void TickTargetManager::measurementCallBackIds(long long n, const unsigned* ids, const uint32_t* sec, const uint32_t* nsec,
                                               const double* poses) {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  if (n <= 0) return;
  flushLocked();
  te_pool* pool = tickPool();
  if (!foreignPossible(pool)) {   // the whole message in one call: lookup, stable sort by slot, per-slot Measurement::update on the device
    if (te_pool_mailbox_ingest(pool, n, ids, sec, nsec, poses) < 0) throw std::runtime_error(te_last_error());
    return;
  }
  std::vector<unsigned> d_ids;
  std::vector<uint32_t> d_sec, d_nsec;
  std::vector<double> d_pose;
  for (long long i = 0; i < n; ++i) {
    auto it = targets_.find(ids[i]);
    const bool foreign = (it != targets_.end() && it->second != (uint8_t)type_) || measurements_.count(ids[i]);
    if (foreign) {
      StampedPose tr;
      tr.sec = sec[i];
      tr.nsec = nsec[i];
      std::memcpy(tr.pose.data(), poses + 7 * i, 7 * sizeof(double));
      measurements_[ids[i]].update(tr);
    } else {
      d_ids.push_back(ids[i]);
      d_sec.push_back(sec[i]);
      d_nsec.push_back(nsec[i]);
      d_pose.insert(d_pose.end(), poses + 7 * i, poses + 7 * i + 7);
    }
  }
  if (!d_ids.empty() && te_pool_mailbox_ingest(pool, (long long)d_ids.size(), d_ids.data(), d_sec.data(), d_nsec.data(), d_pose.data()) < 0)
    throw std::runtime_error(te_last_error());
}

// by-id tick for the host mailboxes of measurements_ (ids living in a pool of another model type): the reference's loop
// (:46-76) turned into one add, one sparse step launch and one expiry call
void TickTargetManager::tickForeign(const double& dt, uint32_t now_sec, uint32_t now_nsec, std::vector<unsigned>& gone_out) {
  const size_t nm = measurements_.size();
  std::vector<unsigned> new_ids, step_ids;
  std::vector<double> new_p0, step_meas;
  std::vector<uint8_t> step_act;
  step_ids.reserve(nm); step_meas.reserve(nm * 7); step_act.reserve(nm);
  const double now = toSec(now_sec, now_nsec);
  std::vector<unsigned> expired;
  for (auto& kv : measurements_) {
    const unsigned id = kv.first;
    StampedPose tr;
    const bool known = targets_.count(id) != 0;
    const double last = kv.second.getTime();
    if (kv.second.read(tr)) {
      if (!known) {   // target does not exist: create it from the measurement (:54-58), then update with the same one
        new_ids.push_back(id);
        new_p0.insert(new_p0.end(), tr.pose.begin(), tr.pose.end());
      }
      step_ids.push_back(id);
      step_act.push_back((uint8_t)TE_ACT_UPDATE);
      step_meas.insert(step_meas.end(), tr.pose.begin(), tr.pose.end());
    } else if (known) {
      step_ids.push_back(id);
      step_act.push_back((uint8_t)TE_ACT_PREDICT);
      step_meas.insert(step_meas.end(), 7, 0.0);
    } else if (!quiet) {
      std::printf("Target(%u) does not exist!\n", id);   // TargetManager::update(id,dt) on an unknown id (:209)
    }
    if (last > 0.0 && (now - last) >= expiration_time_) expired.push_back(id);   // :67
  }
  if (!new_ids.empty()) {   // init on first sight: p0 = the measurement, t0 = t_, v0 = a0 = 0 (:57)
    std::vector<double> t0(new_ids.size(), t_);
    const bool q = quiet;
    quiet = true;
    initBatch(type_, Q_, R_, P_, (long long)new_ids.size(), new_ids.data(), dt, t0.data(), new_p0.data());
    quiet = q;
  }
  if (!step_ids.empty()) updateBatch((long long)step_ids.size(), step_ids.data(), dt, step_meas.data(), step_act.data());
  for (unsigned id : expired) {   // :69-71: the mailbox and the target go
    if (!quiet) std::printf("Timeout for target %u\n", id);
    measurements_.erase(id);
    const bool q = quiet;
    quiet = true;
    erase(id);
    quiet = q;
    gone_out.push_back(id);
  }
  flushLocked();
}

void TickTargetManager::tick(const double& dt, uint32_t now_sec, uint32_t now_nsec, std::vector<unsigned>* erased) {   // :41-92
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  advance(dt, now_sec, now_nsec, erased);
  // 3. the filtered poses the node broadcasts (:76-87)
  if (!publish) {
    pub_ids_.clear();
    pub_poses_.clear();
    return;
  }
  const long long n = publishCount();
  // The output vectors keep their storage across ticks (no re-zeroing) and that storage is page-locked while it lasts, so the
  // read-back of 56 B per target runs at PCIe speed instead of through the driver's pageable staging
  if (pub_poses_.capacity() < (size_t)n * 7) {
    if (pub_pinned_) te_host_unregister(pub_pinned_);
    pub_pinned_ = nullptr;
    pub_poses_.clear();
    pub_poses_.reserve((size_t)(n + n / 4) * 7);
    if (pub_poses_.capacity() * sizeof(double) >= (1u << 20) && te_host_register(pub_poses_.data(), pub_poses_.capacity() * sizeof(double)) == 0)
      pub_pinned_ = pub_poses_.data();
  }
  pub_ids_.resize((size_t)n);
  pub_poses_.resize((size_t)n * 7);
  publishInto(pub_ids_.data(), pub_poses_.data(), n);
}

void TickTargetManager::advance(const double& dt, uint32_t now_sec, uint32_t now_nsec, std::vector<unsigned>* erased) {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  if (!(dt >= 0.0)) throw std::invalid_argument("dt must be >= 0");
  flushLocked();
  te_pool* pool = tickPool();
  // 1. the device tick: first-sight init, sticky update / predict, expiry -- one rebuild + one step launch (:46-76)
  const long long cap = std::max<long long>(te_pool_mailbox_bound(pool), 1);
  if ((long long)gone_buf_.size() < cap) {   // reused across ticks: sizing them per tick would zero 8 bytes per target per tick
    gone_buf_.resize((size_t)(cap + cap / 4));
    born_buf_.resize((size_t)(cap + cap / 4));
  }
  long long n_born = 0;
  const long long n_gone = te_pool_mailbox_tick(pool, dt, t_, cls_, now_sec, now_nsec, expiration_time_, gone_buf_.data(), cap, born_buf_.data(), cap,
                                                &n_born);
  if (n_gone < 0) throw std::runtime_error(te_last_error());
  std::vector<uint32_t> gone(gone_buf_.begin(), gone_buf_.begin() + std::min(n_gone, cap));
  std::vector<uint32_t> born(born_buf_.begin(), born_buf_.begin() + std::min(n_born, cap));
  targets_.insertSorted(born.data(), born.size(), (uint8_t)type_);   // both lists are ascending: one linear pass each
  targets_.eraseSorted(gone.data(), gone.size());                    // (a target-less mailbox that expired has no entry here)
  if (!quiet)
    for (uint32_t id : gone) std::printf("Timeout for target %u\n", id);
  // 2. host mailboxes of ids living under another model type, if any
  if (!measurements_.empty()) {
    std::vector<unsigned> gone2;
    tickForeign(dt, now_sec, now_nsec, gone2);
    if (!gone2.empty()) {
      std::vector<uint32_t> all(gone.size() + gone2.size());
      std::merge(gone.begin(), gone.end(), gone2.begin(), gone2.end(), all.begin());
      gone.swap(all);
    }
  }
  if (erased) erased->assign(gone.begin(), gone.end());
  t_ = t_ + dt;   // :89
}

long long TickTargetManager::publishCount() {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  return (long long)targets_.size();
}

void TickTargetManager::publishInto(unsigned* ids, double* poses, long long n) {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  if (n != (long long)targets_.size()) throw std::logic_error("publishInto: the output does not fit the targets");
  if (n == 0) return;
  te_pool* pool = tickPool();
  if (measurements_.empty() && targets_.size() == (size_t)te_pool_size(pool)) {
    // every target lives in the tick's pool: ids and poses of all slots in slot order = ascending ids, no per-id lookups
    if (te_pool_ids(pool, ids, n) < 0 || te_pool_read_estimates(pool, n, nullptr, nullptr, poses, nullptr, nullptr, nullptr, nullptr) < 0)
      throw std::runtime_error(te_last_error());
  } else {
    const std::vector<unsigned> all = getAvailableTargets();
    std::copy(all.begin(), all.end(), ids);
    getEstimatesBatch(n, ids, nullptr, poses, nullptr, nullptr, nullptr);
  }
}

size_t TickTargetManager::mailboxCount() {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  te_pool* pool = poolOf((int)type_, false);
  const long long n = pool ? te_pool_mailbox_count(pool) : 0;
  if (n < 0) throw std::runtime_error(te_last_error());
  return (size_t)n + measurements_.size();
}

}  // namespace target_estimation_b200
