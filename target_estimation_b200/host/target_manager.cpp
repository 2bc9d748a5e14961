// target_manager.cpp -- host surface (TargetManager / TargetInterface / IntersectionSolver) over the
// device pools of include/te_pool.h.  Mirrors /root/reference/src/target_manager.cpp:18-295,
// src/target_interface.cpp:80-152 and src/intersection_solver.cpp:19-124 call for call; the arithmetic
// itself runs in the CUDA layer (no computation of filter state happens on the host).
#include "target_estimation_b200/target_manager.hpp"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>
#include <fstream>
#include <iostream>
#include <numeric>
#include <sstream>
#include <stdexcept>
#include <unordered_set>

#include "../csrc/te_query_args.h"
#include "rows.hpp"

namespace target_estimation_b200 {

namespace {

struct PoolError : std::runtime_error {
  using std::runtime_error::runtime_error;
};
inline void ck(long long rc) {
  if (rc < 0) throw PoolError(te_last_error());
}
// the model type of a TargetManager::heldTypes() mask: the one type, -1 = no target, -2 = several types
inline int onlyType(unsigned held) { return held == 0 ? -1 : (held & (held - 1)) ? -2 : __builtin_ctz(held); }

// --- minimal reader for the reference's model files (models/*.yaml: `key: scalar` and
// `key: [v, v, ...]` lines; yaml-cpp is not available in this image) -------------------------
bool yamlLite(const std::string& file, std::map<std::string, std::string>& scalars, std::map<std::string, std::vector<double>>& lists) {
  std::ifstream in(file);
  if (!in) return false;
  std::stringstream ss;
  ss << in.rdbuf();
  std::string text = ss.str();
  size_t pos = 0;
  while (pos < text.size()) {
    size_t eol = text.find('\n', pos);
    if (eol == std::string::npos) eol = text.size();
    std::string line = text.substr(pos, eol - pos);
    size_t hash = line.find('#');
    if (hash != std::string::npos) line = line.substr(0, hash);
    size_t colon = line.find(':');
    if (colon == std::string::npos) { pos = eol + 1; continue; }
    std::string key = line.substr(0, colon);
    key.erase(0, key.find_first_not_of(" \t"));
    key.erase(key.find_last_not_of(" \t") + 1);
    std::string val = line.substr(colon + 1);
    size_t lb = val.find('[');
    if (lb != std::string::npos) {
      // flow sequence, possibly spanning lines
      size_t abs_lb = pos + colon + 1 + lb;
      size_t rb = text.find(']', abs_lb);
      if (rb == std::string::npos) return false;
      std::string body = text.substr(abs_lb + 1, rb - abs_lb - 1);
      for (char& ch : body) if (ch == ',' || ch == '\n' || ch == '\r') ch = ' ';
      std::stringstream ls(body);
      std::vector<double> v;
      std::string tok;
      while (ls >> tok) {
        try { v.push_back(std::stod(tok)); } catch (...) { return false; }
      }
      lists[key] = v;
      eol = text.find('\n', rb);
      if (eol == std::string::npos) eol = text.size();
    } else {
      val.erase(0, val.find_first_not_of(" \t\"'"));
      size_t e = val.find_last_not_of(" \t\r\"'");
      val = (e == std::string::npos) ? std::string() : val.substr(0, e + 1);
      scalars[key] = val;
    }
    pos = eol + 1;
  }
  return true;
}

// parseSquareMatrix (src/target_manager.cpp:18-33): size = sqrt(len); Eigen::Map<MatrixXd> is COLUMN-major,
// so M(i,j) = v[i + s*j] (the transpose of the file's visual layout).
bool squareFromList(const std::map<std::string, std::vector<double>>& lists, const std::string& key, MatrixXd& M) {
  auto it = lists.find(key);
  if (it == lists.end()) return false;
  const std::vector<double>& v = it->second;
  const unsigned s = static_cast<unsigned>(std::sqrt((double)v.size()));
  if (s == 0) return false;
  M = MatrixXd((int)s, (int)s);
  for (unsigned i = 0; i < s; ++i)
    for (unsigned j = 0; j < s; ++j) M((int)i, (int)j) = v[i + (size_t)s * j];
  return true;
}

}  // namespace

// ----------------------------------------------------------------------------------------------
// TargetManager
// ----------------------------------------------------------------------------------------------
TargetManager::TargetManager(int device) : device_(device) {}

TargetManager::TargetManager(const std::string& file, int device) : TargetManager(device) {
  if (!loadYamlFile(file, default_Q_, default_R_, default_P_, default_type_))
    throw "TargetManager default constructor failed!";
  default_values_loaded_ = true;
}

TargetManager::~TargetManager() {
  for (te_pool*& p : pools_) {
    if (p) te_pool_destroy(p);
    p = nullptr;
  }
}

bool TargetManager::selectTargetType(const std::string& s, target_t& type) {   // src/target_manager.cpp:52-65
  if (s == "angular_rates") type = ANGULAR_RATES;
  else if (s == "angular_velocities") type = ANGULAR_VELOCITIES;
  else if (s == "uniform_acceleration") type = UNIFORM_ACCELERATION;
  else if (s == "uniform_velocity") type = UNIFORM_VELOCITY;
  else return false;
  return true;
}

bool TargetManager::loadYamlFile(const std::string& file, MatrixXd& Q, MatrixXd& R, MatrixXd& P, target_t& type) {   // :67-104
  std::map<std::string, std::string> scalars;
  std::map<std::string, std::vector<double>> lists;
  bool success = true;
  if (!yamlLite(file, scalars, lists)) {
    std::cerr << "Can not parse file: " << file << std::endl;
    return false;
  }
  if (!squareFromList(lists, "Q", Q)) { std::cerr << "Can not load matrix Q from file: " << file << std::endl; success = false; }
  if (!squareFromList(lists, "R", R)) { std::cerr << "Can not load matrix R from file: " << file << std::endl; success = false; }
  if (!squareFromList(lists, "P", P)) { std::cerr << "Can not load matrix P from file: " << file << std::endl; success = false; }
  auto it = scalars.find("type");
  if (it == scalars.end()) {
    std::cerr << "Can not load type from file: " << file << std::endl;
    success = false;
  } else if (!selectTargetType(it->second, type)) {
    std::cerr << "Can not parse type: " << it->second << std::endl;   // the reference keeps going with an unset type (:40-41)
    success = false;
  }
  return success;
}

te_pool* TargetManager::poolOf(int type, bool create) {
  if (type < 0 || type > 3) return nullptr;
  if (!pools_[type] && create) {
    pools_[type] = te_pool_create(type, device_, nullptr);
    if (!pools_[type]) throw PoolError(te_last_error());
  }
  return pools_[type];
}

// ---- IdRegistry ------------------------------------------------------------------------------------------
IdRegistry::iterator IdRegistry::find(unsigned id) {
  auto it = std::lower_bound(v_.begin(), v_.end(), id, [](const value_type& a, unsigned key) { return a.first < key; });
  return (it != v_.end() && it->first == id) ? it : v_.end();
}
uint8_t& IdRegistry::operator[](unsigned id) {
  if (v_.empty() || v_.back().first < id) {   // ascending arrivals (track ids grow): append
    v_.emplace_back(id, (uint8_t)0);
    return v_.back().second;
  }
  auto it = std::lower_bound(v_.begin(), v_.end(), id, [](const value_type& a, unsigned key) { return a.first < key; });
  if (it == v_.end() || it->first != id) it = v_.insert(it, value_type(id, (uint8_t)0));
  return it->second;
}
size_t IdRegistry::erase(unsigned id) {
  auto it = find(id);
  if (it == v_.end()) return 0;
  v_.erase(it);
  return 1;
}
void IdRegistry::mergeSorted(const std::vector<value_type>& add) {
  if (add.empty()) return;
  if (v_.empty() || v_.back().first < add.front().first) {   // append-only batch
    v_.insert(v_.end(), add.begin(), add.end());
    return;
  }
  std::vector<value_type> out;
  out.reserve(v_.size() + add.size());
  size_t i = 0, j = 0;
  while (i < v_.size() && j < add.size()) {
    if (v_[i].first < add[j].first) out.push_back(v_[i++]);
    else if (add[j].first < v_[i].first) out.push_back(add[j++]);
    else { out.push_back(v_[i++]); ++j; }   // existing entry wins
  }
  out.insert(out.end(), v_.begin() + (long)i, v_.end());
  out.insert(out.end(), add.begin() + (long)j, add.end());
  v_.swap(out);
}
void IdRegistry::insertSorted(const uint32_t* ids, size_t n, uint8_t type) {
  std::vector<value_type> add;
  add.reserve(n);
  for (size_t k = 0; k < n; ++k) add.emplace_back(ids[k], type);
  mergeSorted(add);
}
void IdRegistry::eraseSorted(const uint32_t* ids, size_t n) {
  if (n == 0 || v_.empty()) return;
  size_t w = 0, j = 0;
  auto first = std::lower_bound(v_.begin(), v_.end(), ids[0], [](const value_type& a, unsigned key) { return a.first < key; });
  w = (size_t)(first - v_.begin());
  for (size_t i = w; i < v_.size(); ++i) {
    while (j < n && ids[j] < v_[i].first) ++j;
    if (j < n && ids[j] == v_[i].first) continue;   // dropped
    v_[w++] = v_[i];
  }
  v_.resize(w);
}

int TargetManager::registerClass(int type, const MatrixXd& Q, const MatrixXd& R, const MatrixXd& P0) {
  int n = 0, m = 0;
  te_model_dims(type, &n, &m);
  // asserts of the model constructors (e.g. src/types/uniform_acceleration.cpp:35-37) + the hard-wired
  // measurement sizes of addMeasurement (SURVEY.md Appendix A: m must be 3 / 6)
  if (Q.rows() != n || Q.cols() != n || P0.rows() != n || P0.cols() != n || R.rows() != m || R.cols() != m)
    throw std::invalid_argument("model matrices do not match the target type (n=" + std::to_string(n) + ", m=" + std::to_string(m) + ")");
  te_pool* p = poolOf(type, true);
  int cls = te_pool_register_class(p, Q.data(), R.data(), P0.data());
  ck(cls);
  return cls;
}

bool TargetManager::typeOf(unsigned id, int& type) {
  auto it = targets_.find(id);
  if (it == targets_.end()) return false;
  type = it->second;
  return true;
}

unsigned TargetManager::heldTypes() {
  unsigned held = 0;
  for (int t = 0; t < 4; ++t)
    if (pools_[t] && te_pool_size(pools_[t]) > 0) held |= 1u << t;
  return held;
}

void TargetManager::rowsByType(long long n, const unsigned* ids, std::vector<long long> rows[4]) {
  for (int t = 0; t < 4; ++t) rows[t].clear();
  for (long long k = 0; k < n; ++k) {
    auto it = targets_.find(ids[k]);
    if (it != targets_.end()) rows[it->second].push_back(k);
  }
}

void TargetManager::requireMeasurements(long long n, const double* meas, const unsigned char* action) {
  if (meas) return;
  bool needs = !action;
  for (long long k = 0; k < n && !needs; ++k) needs = action[k] == TE_ACT_UPDATE;
  if (needs) throw std::invalid_argument("update ops without measurements");
}

void TargetManager::init(const unsigned int& id, const double& dt0, const double& t0, const Vector7d& p0, const Vector6d& v0,
                         const Vector6d& a0) {   // :135-142
  if (default_values_loaded_) init(default_type_, id, dt0, t0, default_Q_, default_R_, default_P_, p0, v0, a0);
  else throw "TargetManager::init failed, can not find default values to load!";
}

void TargetManager::init(const target_t& type, const unsigned int& id, const double& dt0, const double& t0, const MatrixXd& Q,
                         const MatrixXd& R, const MatrixXd& P0, const Vector7d& p0, const Vector6d& v0, const Vector6d& a0) {   // :144-179
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  if (targets_.find(id) != targets_.end()) {
    if (!quiet) std::cout << "Target(" << id << ") already exists!" << std::endl;
    return;
  }
  if (!(dt0 >= 0.0) || !(t0 >= 0.0)) throw std::invalid_argument("dt0 and t0 must be >= 0 (asserts of src/target_interface.cpp:20)");
  flushLocked();
  const int cls = registerClass((int)type, Q, R, P0);
  const uint32_t uid = id;
  const uint16_t c16 = (uint16_t)cls;
  ck(te_pool_add_batch(poolOf((int)type, true), 1, &uid, &c16, &t0, p0.data(), v0.data(), a0.data(), nullptr));
  targets_[id] = (uint8_t)type;
  if (!quiet) {
    static const char* msg[4] = {"Using angular rates for the orientation", "Using angular velocities for the orientation",
                                 "Uniformly accelerated motion", "Uniform rectilinear motion"};
    std::cout << msg[(int)type] << std::endl;
  }
}

void TargetManager::init(const std::string& file, const unsigned int& id, const double& dt0, const double& t0, const Vector7d& p0,
                         const Vector6d& v0, const Vector6d& a0) {   // :181-188
  MatrixXd Q, P, R;
  target_t type = UNIFORM_VELOCITY;
  if (!loadYamlFile(file, Q, R, P, type)) throw std::invalid_argument("cannot load model file " + file);
  init(type, id, dt0, t0, Q, R, P, p0, v0, a0);
}

long long TargetManager::initBatch(long long n, const unsigned* ids, double dt0, const double* t0, const double* p0, const double* v0,
                                   const double* a0) {
  if (!default_values_loaded_) throw "TargetManager::init failed, can not find default values to load!";
  return initBatch(default_type_, default_Q_, default_R_, default_P_, n, ids, dt0, t0, p0, v0, a0, nullptr);
}

long long TargetManager::initBatch(target_t type, const MatrixXd& Q, const MatrixXd& R, const MatrixXd& P0, long long n, const unsigned* ids,
                                   double dt0, const double* t0, const double* p0, const double* v0, const double* a0,
                                   const double* p0_scale) {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  if (n <= 0) return 0;
  if (!(dt0 >= 0.0)) throw std::invalid_argument("dt0 must be >= 0");
  flushLocked();
  const int cls = registerClass((int)type, Q, R, P0);
  // ids already known to the manager under ANY type are skipped ("already exists"); first occurrence wins
  std::vector<long long> keep;
  keep.reserve((size_t)n);
  std::vector<std::pair<unsigned, uint8_t>> fresh;   // ascending (id, type) pairs for the registry
  bool ascending = true;
  for (long long k = 1; k < n && ascending; ++k) ascending = ids[k - 1] < ids[k];
  if (ascending) {
    // the usual batch (track ids grow): no id repeats inside it, and one walk along the sorted registry finds the known ones
    fresh.reserve((size_t)n);
    auto it = targets_.begin();
    for (long long k = 0; k < n; ++k) {
      while (it != targets_.end() && it->first < ids[k]) ++it;
      if (it != targets_.end() && it->first == ids[k]) {
        if (!quiet) std::cout << "Target(" << ids[k] << ") already exists!" << std::endl;
        continue;
      }
      fresh.emplace_back(ids[k], (uint8_t)type);
      keep.push_back(k);
    }
  } else {
    std::map<unsigned, uint8_t> seen;
    for (long long k = 0; k < n; ++k) {
      if (targets_.count(ids[k]) || seen.count(ids[k])) {
        if (!quiet) std::cout << "Target(" << ids[k] << ") already exists!" << std::endl;
        continue;
      }
      seen[ids[k]] = (uint8_t)type;
      keep.push_back(k);
    }
    fresh.assign(seen.begin(), seen.end());
  }
  if (keep.empty()) return 0;
  const long long na = (long long)keep.size();
  std::vector<uint32_t> g_ids;
  std::vector<uint16_t> g_cls((size_t)na, (uint16_t)cls);
  std::vector<double> g_t0, g_p0, g_v0, g_a0, g_sc;
  const bool all = na == n;
  const double* s_p0 = all ? p0 : gatherRows<7>(p0, keep, g_p0);
  const double* s_t0 = all ? t0 : gatherRows<1>(t0, keep, g_t0);
  const double* s_v0 = all ? v0 : gatherRows<6>(v0, keep, g_v0);
  const double* s_a0 = all ? a0 : gatherRows<6>(a0, keep, g_a0);
  const double* s_sc = all ? p0_scale : gatherRows<1>(p0_scale, keep, g_sc);
  long long added = te_pool_add_batch(poolOf((int)type, true), na, gatherRows<1>(ids, keep, g_ids), g_cls.data(), s_t0, s_p0, s_v0, s_a0, s_sc);
  ck(added);
  targets_.insert(fresh.begin(), fresh.end());
  return added;
}

void TargetManager::queue(int type, unsigned id, double dt, const double* meas, int action) {
  if (pending_ids_.count(id)) flushLocked();   // an id may appear once per launch: keep call order observable
  Pending& q = pending_[type];
  q.ids.push_back(id);
  q.dt.push_back(dt);
  q.action.push_back((uint8_t)action);
  const size_t o = q.meas.size();
  q.meas.resize(o + 7, 0.0);
  if (meas) std::memcpy(&q.meas[o], meas, 7 * sizeof(double));
  pending_ids_[id] = (uint8_t)type;
}

void TargetManager::flushLocked() {
  if (pending_ids_.empty()) return;
  for (int t = 0; t < 4; ++t) {
    Pending& q = pending_[t];
    if (q.ids.empty()) continue;
    long long rc = te_pool_step_ids(pools_[t], (long long)q.ids.size(), q.ids.data(), q.dt.data(), 0.0, q.meas.data(), q.action.data());
    q.ids.clear(); q.dt.clear(); q.meas.clear(); q.action.clear();
    if (rc < 0) {
      pending_ids_.clear();
      throw PoolError(te_last_error());
    }
  }
  pending_ids_.clear();
}

void TargetManager::flush() {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  flushLocked();
}

bool TargetManager::update(const unsigned int& id, const double& dt, const Vector7d& meas) {   // :190-202
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  int type;
  if (!typeOf(id, type)) {
    if (!quiet) std::cout << "Target(" << id << ") does not exist!" << std::endl;
    return false;
  }
  if (!(dt >= 0.0)) throw std::invalid_argument("dt must be >= 0 (assert of src/target_interface.cpp:150)");
  queue(type, id, dt, meas.data(), TE_ACT_UPDATE);
  return true;
}

bool TargetManager::update(const unsigned int& id, const double& dt) {   // :204-218
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  int type;
  if (!typeOf(id, type)) {
    if (!quiet) std::cout << "Target(" << id << ") does not exist!" << std::endl;
    return false;
  }
  if (!(dt >= 0.0)) throw std::invalid_argument("dt must be >= 0");
  queue(type, id, dt, nullptr, TE_ACT_PREDICT);
  return true;
}

void TargetManager::update(const double& dt) {   // :220-225
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  flushLocked();
  for (int t = 0; t < 4; ++t)
    if (pools_[t]) ck(te_pool_predict_all(pools_[t], dt));
}

long long TargetManager::updateBatch(long long n, const unsigned* ids, double dt, const double* meas, const unsigned char* action) {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  if (n <= 0) return 0;
  requireMeasurements(n, meas, action);
  flushLocked();
  // te_pool_step_ids applies one op per id per launch.  A batch that names an id again stands for the reference's sequential
  // update() calls, which apply every record in order: cut the batch in front of each repeat and launch the pieces one after
  // the other (strictly ascending ids -- the usual batch -- cannot repeat and skip the hash set).
  bool ascending = true;
  for (long long k = 1; k < n && ascending; ++k) ascending = ids[k - 1] < ids[k];
  if (ascending) return updateBatchUnique(n, ids, dt, meas, action);
  {
    // ids in arbitrary order (a /tf message lists its targets as they come): a homogeneous manager hands the batch over as it is --
    // the device finds a repeated id while it looks the ids up, before anything is stepped (te_pool_step_ids returns -2) -- and
    // only then the batch is cut on the host (a hash set of four million ids costs 50 x the tick it guards)
    const int only = onlyType(heldTypes());
    if (only == -1) return 0;
    if (only >= 0) {
      const long long rc = te_pool_step_ids(pools_[only], n, ids, nullptr, dt, meas, action);
      if (rc != -2) {
        ck(rc);
        return rc;
      }
    }
  }
  long long applied = 0, start = 0;
  std::unordered_set<unsigned> seen;
  seen.reserve((size_t)std::min<long long>(n, 1 << 22));
  for (long long k = 0; k < n; ++k) {
    if (!seen.insert(ids[k]).second) {
      applied += updateBatchUnique(k - start, ids + start, dt, meas ? meas + 7 * (size_t)start : nullptr, action ? action + start : nullptr);
      start = k;
      seen.clear();
      seen.insert(ids[k]);
    }
  }
  return applied + updateBatchUnique(n - start, ids + start, dt, meas ? meas + 7 * (size_t)start : nullptr, action ? action + start : nullptr);
}

long long TargetManager::updateBatchUnique(long long n, const unsigned* ids, double dt, const double* meas, const unsigned char* action) {
  if (n <= 0) return 0;
  const int only = onlyType(heldTypes());
  if (only == -1) return 0;
  if (only >= 0) {   // homogeneous manager: the batch goes to the device as it is
    long long rc = te_pool_step_ids(pools_[only], n, ids, nullptr, dt, meas, action);
    ck(rc);
    return rc;
  }
  // mixed manager: split the batch by model type on the host
  std::vector<long long> rows[4];
  rowsByType(n, ids, rows);
  std::vector<uint32_t> s_ids;
  std::vector<double> s_meas;
  std::vector<uint8_t> s_act;
  long long applied = 0;
  for (int t = 0; t < 4; ++t) {
    if (rows[t].empty()) continue;
    long long rc = te_pool_step_ids(pools_[t], (long long)rows[t].size(), gatherRows<1>(ids, rows[t], s_ids), nullptr, dt,
                                    gatherRows<7>(meas, rows[t], s_meas), gatherRows<1>(action, rows[t], s_act));
    ck(rc);
    applied += rc;
  }
  return applied;
}

te_pool* TargetManager::densePool() {
  const int only = onlyType(heldTypes());
  if (only < 0) throw std::invalid_argument("a dense tick needs a manager whose targets share one model type");
  return pools_[only];
}

long long TargetManager::updateDense(double dt, const double* meas, int meas_stride, const unsigned char* action, double* est_pos_out) {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  flushLocked();
  if (targets_.empty()) return 0;
  te_pool* p = densePool();
  ck(te_pool_tick_host(p, dt, meas, meas_stride, action, TE_ACT_UPDATE, est_pos_out));
  return te_pool_size(p);
}

long long TargetManager::updateDenseAsync(double dt, const double* meas, int meas_stride, const unsigned char* action, double* est_pos_out) {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  flushLocked();
  if (targets_.empty()) return 0;
  te_pool* p = densePool();
  ck(te_pool_tick_host_async(p, dt, meas, meas_stride, action, TE_ACT_UPDATE, est_pos_out));
  return te_pool_size(p);
}

void TargetManager::updateDenseWait(int lag) {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  for (int t = 0; t < 4; ++t)
    if (pools_[t]) ck(te_pool_tick_host_wait(pools_[t], lag));
}

std::vector<unsigned int> TargetManager::denseIds() { return getAvailableTargets(); }

size_t TargetManager::size() {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  return targets_.size();
}

bool TargetManager::erase(const unsigned int& id) {   // :227-241
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  auto it = targets_.find(id);
  if (it == targets_.end()) {
    if (!quiet) std::cout << "Target(" << id << ") does not exist!" << std::endl;
    return false;
  }
  flushLocked();
  const uint32_t uid = id;
  ck(te_pool_erase_batch(pools_[it->second], 1, &uid));
  targets_.erase(it);
  return true;
}

long long TargetManager::eraseBatch(long long n, const unsigned* ids) {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  flushLocked();
  std::vector<long long> rows[4];
  rowsByType(n, ids, rows);
  std::vector<uint32_t> per[4], found;
  for (int t = 0; t < 4; ++t) {
    gatherRows<1>(ids, rows[t], per[t]);
    found.insert(found.end(), per[t].begin(), per[t].end());
  }
  std::sort(found.begin(), found.end());
  targets_.eraseSorted(found.data(), found.size());
  long long erased = 0;
  for (int t = 0; t < 4; ++t) {
    if (per[t].empty()) continue;
    long long rc = te_pool_erase_batch(pools_[t], (long long)per[t].size(), per[t].data());
    ck(rc);
    erased += rc;
  }
  return erased;
}

TargetInterface::Ptr TargetManager::getTarget(const unsigned int& id) {   // :243-250
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  if (targets_.count(id) != 0) return std::make_shared<TargetInterface>(this, id);
  return nullptr;
}

void TargetManager::getEstimatesBatch(long long n, const unsigned* ids, const double* t1, double* pose7, double* twist6, double* acc6,
                                      unsigned char* found) {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  if (n <= 0) return;
  flushLocked();
  if (found) std::memset(found, 0, (size_t)n);
  const int only = onlyType(heldTypes());
  if (only == -1) return;
  if (only >= 0) {
    ck(te_pool_read_estimates(pools_[only], n, ids, t1, pose7, twist6, acc6, nullptr, found));
    return;
  }
  std::vector<long long> rows[4];
  rowsByType(n, ids, rows);
  std::vector<uint32_t> s_ids;
  std::vector<double> s_t1, po, tw, ac;
  std::vector<uint8_t> fo;
  for (int t = 0; t < 4; ++t) {
    const size_t m = rows[t].size();
    if (m == 0) continue;
    po.resize(m * 7); tw.resize(m * 6); ac.resize(m * 6); fo.resize(m);
    ck(te_pool_read_estimates(pools_[t], (long long)m, gatherRows<1>(ids, rows[t], s_ids), gatherRows<1>(t1, rows[t], s_t1), po.data(),
                              tw.data(), ac.data(), nullptr, fo.data()));
    scatterRows<7>(pose7, rows[t], po.data());
    scatterRows<6>(twist6, rows[t], tw.data());
    scatterRows<6>(acc6, rows[t], ac.data());
    scatterRows<1>(found, rows[t], fo.data());
  }
}

bool TargetManager::getTargetPose(const unsigned int& id, Vector7d& pose) {   // :252-261
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  int type;
  if (!typeOf(id, type)) return false;
  flushLocked();
  const uint32_t uid = id;
  ck(te_pool_read_estimates(pools_[type], 1, &uid, nullptr, pose.data(), nullptr, nullptr, nullptr, nullptr));
  return true;
}

bool TargetManager::getTargetTwist(const unsigned int& id, Vector6d& twist) {   // :263-272
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  int type;
  if (!typeOf(id, type)) return false;
  flushLocked();
  const uint32_t uid = id;
  ck(te_pool_read_estimates(pools_[type], 1, &uid, nullptr, nullptr, twist.data(), nullptr, nullptr, nullptr));
  return true;
}

bool TargetManager::getTargetAcceleration(const unsigned int& id, Vector6d& acc) {   // :274-283
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  int type;
  if (!typeOf(id, type)) return false;
  flushLocked();
  const uint32_t uid = id;
  ck(te_pool_read_estimates(pools_[type], 1, &uid, nullptr, nullptr, nullptr, acc.data(), nullptr, nullptr));
  return true;
}

long long TargetManager::getNumberMeasurements(const unsigned int& id) {   // :285-295
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  int type;
  if (!typeOf(id, type)) {
    if (!quiet) std::cout << "Target(" << id << ") does not exist!" << std::endl;
    return 0;
  }
  flushLocked();
  const uint32_t uid = id;
  long long nm = 0;
  ck(te_pool_read_state(pools_[type], 1, &uid, nullptr, nullptr, nullptr, &nm, nullptr, nullptr));
  return nm;
}

// ---- sampled logging (the reference's rt_logger publishers + writeTxtFile dumps) ----------------------------
void TargetManager::watch(long long n, const unsigned* ids, size_t max_samples) {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  log_ids_.assign(ids, ids + (n > 0 ? n : 0));
  log_cap_ = max_samples;
  log_t_.clear(); log_rows_.clear(); log_P_.clear(); log_n_.clear();
}

void TargetManager::log() {   // :119-123: every target publishes measurement / pose / twist / acceleration / covariance
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  flushLocked();
  const size_t m = log_ids_.size();
  if (m == 0 || log_t_.size() >= log_cap_) return;
  const size_t base = log_t_.size();
  log_rows_.resize((base + 1) * m * 26, 0.0);
  log_P_.resize((base + 1) * m * 324, 0.0);
  log_n_.resize((base + 1) * m, 0);
  double t_sample = std::nan("");
  // one batched read-back per pool that holds watched ids
  std::vector<long long> rows[4];
  rowsByType((long long)m, log_ids_.data(), rows);
  std::vector<uint32_t> sub;
  for (int type = 0; type < 4; ++type) {
    if (rows[type].empty()) continue;
    gatherRows<1>(log_ids_.data(), rows[type], sub);
    int N = 0, M = 0;
    te_model_dims(type, &N, &M);
    const long long k = (long long)sub.size();
    std::vector<double> t((size_t)k), P((size_t)k * N * N), mp((size_t)k * 7), tw((size_t)k * 6), ac((size_t)k * 6), pi((size_t)k * 6);
    ck(te_pool_read_state(pools_[type], k, sub.data(), nullptr, P.data(), t.data(), nullptr, nullptr, mp.data()));
    ck(te_pool_read_estimates(pools_[type], k, sub.data(), nullptr, nullptr, tw.data(), ac.data(), pi.data(), nullptr));
    for (long long q = 0; q < k; ++q) {
      const size_t j = (size_t)rows[type][(size_t)q];
      double* row = &log_rows_[(base * m + j) * 26];
      row[0] = t[(size_t)q];
      std::memcpy(row + 1, &mp[(size_t)q * 7], 7 * sizeof(double));
      std::memcpy(row + 8, &pi[(size_t)q * 6], 6 * sizeof(double));
      std::memcpy(row + 14, &tw[(size_t)q * 6], 6 * sizeof(double));
      std::memcpy(row + 20, &ac[(size_t)q * 6], 6 * sizeof(double));
      std::memcpy(&log_P_[(base * m + j) * 324], &P[(size_t)q * N * N], sizeof(double) * (size_t)N * N);
      log_n_[base * m + j] = N;
      if (std::isnan(t_sample)) t_sample = t[(size_t)q];
    }
  }
  log_t_.push_back(t_sample);
}

bool TargetManager::logSample(size_t k, size_t j, double* row26, double* P, int* n_state) const {
  const size_t m = log_ids_.size();
  if (k >= log_t_.size() || j >= m) return false;
  const int N = log_n_[k * m + j];
  if (n_state) *n_state = N;
  if (row26) std::memcpy(row26, &log_rows_[(k * m + j) * 26], 26 * sizeof(double));
  if (P && N > 0) std::memcpy(P, &log_P_[(k * m + j) * 324], sizeof(double) * (size_t)N * N);
  return N > 0;
}

bool writeTxtFile(const std::string& filename, const double* values, size_t rows, size_t cols) {   // utils.hpp:78-120
  std::ofstream f(filename.c_str());
  if (!f.is_open()) {
    std::cerr << "Unable to open file : [" << filename << "]" << std::endl;
    return false;
  }
  for (size_t r = 0; r < rows; ++r) {
    if (cols == 1) {   // the VectorXd overload: "value\n"
      f << values[r] << "\n";
    } else {           // the MatrixXd overload: "value " per column, then "\n"
      for (size_t c = 0; c < cols; ++c) f << values[r * cols + c] << " ";
      f << "\n";
    }
  }
  return true;
}

int TargetManager::writeLog(const std::string& folder) const {
  const size_t m = log_ids_.size(), S = log_t_.size();
  int files = 0;
  for (size_t j = 0; j < m; ++j) {
    std::vector<double> time, meas, pose, twist, acc, diag;
    size_t n_diag = 0;
    for (size_t k = 0; k < S; ++k) {
      const int N = log_n_[k * m + j];
      if (N == 0) continue;   // the id did not exist at that sample
      const double* row = &log_rows_[(k * m + j) * 26];
      time.push_back(row[0]);
      meas.insert(meas.end(), row + 1, row + 8);
      pose.insert(pose.end(), row + 8, row + 14);
      twist.insert(twist.end(), row + 14, row + 20);
      acc.insert(acc.end(), row + 20, row + 26);
      n_diag = (size_t)N;
      for (int d = 0; d < N; ++d) diag.push_back(log_P_[(k * m + j) * 324 + (size_t)d * N + d]);
    }
    if (time.empty()) continue;
    const std::string id = std::to_string(log_ids_[j]);
    files += writeTxtFile(folder + "time_" + id, time.data(), time.size(), 1);
    files += writeTxtFile(folder + "meas_pose_" + id, meas.data(), time.size(), 7);
    files += writeTxtFile(folder + "est_pose_" + id, pose.data(), time.size(), 6);
    files += writeTxtFile(folder + "est_twist_" + id, twist.data(), time.size(), 6);
    files += writeTxtFile(folder + "est_acc_" + id, acc.data(), time.size(), 6);
    files += writeTxtFile(folder + "cov_diag_" + id, diag.data(), time.size(), n_diag);
  }
  return files;
}

std::vector<unsigned int> TargetManager::getAvailableTargets() {   // :125-133
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  std::vector<unsigned int> ids;
  ids.reserve(targets_.size());
  for (auto const& kv : targets_) ids.push_back(kv.first);
  return ids;
}

// ----------------------------------------------------------------------------------------------
// TargetInterface proxy / EstimatorView
// ----------------------------------------------------------------------------------------------
namespace {
struct SlotRead {
  te_pool* pool = nullptr;
  int type = -1;
  int n = 0, m = 0;
};
bool locate(TargetManager* mgr, unsigned id, SlotRead& s) {
  if (!mgr->typeOf(id, s.type)) return false;
  mgr->flush();
  s.pool = mgr->poolOf(s.type, false);
  te_model_dims(s.type, &s.n, &s.m);
  return s.pool != nullptr;
}
}  // namespace

VectorXd EstimatorView::getState() const {
  std::lock_guard<std::recursive_mutex> lg(mgr_->lock());
  SlotRead s;
  if (!locate(mgr_, id_, s)) return VectorXd();
  VectorXd x((size_t)s.n, 0.0);
  const uint32_t uid = id_;
  ck(te_pool_read_state(s.pool, 1, &uid, x.data(), nullptr, nullptr, nullptr, nullptr, nullptr));
  return x;
}
MatrixXd EstimatorView::getP() const {
  std::lock_guard<std::recursive_mutex> lg(mgr_->lock());
  SlotRead s;
  if (!locate(mgr_, id_, s)) return MatrixXd();
  MatrixXd P(s.n, s.n);
  const uint32_t uid = id_;
  ck(te_pool_read_state(s.pool, 1, &uid, nullptr, P.d.data(), nullptr, nullptr, nullptr, nullptr));
  return P;
}
namespace {
MatrixXd classMatrix(TargetManager* mgr, unsigned id, int which) {
  std::lock_guard<std::recursive_mutex> lg(mgr->lock());
  SlotRead s;
  if (!locate(mgr, id, s)) return MatrixXd();
  const uint32_t uid = id;
  int cls = te_pool_class_of(s.pool, uid);
  ck(cls);
  MatrixXd Q(s.n, s.n), R(s.m, s.m), P0(s.n, s.n);
  ck(te_pool_get_class(s.pool, cls, Q.d.data(), R.d.data(), P0.d.data()));
  return which == 0 ? Q : (which == 1 ? R : P0);
}
}  // namespace
MatrixXd EstimatorView::getQ() const { return classMatrix(mgr_, id_, 0); }
MatrixXd EstimatorView::getR() const { return classMatrix(mgr_, id_, 1); }
MatrixXd EstimatorView::getP0() const { return classMatrix(mgr_, id_, 2); }

void TargetInterface::addMeasurement(const double& dt, const Vector7d& meas) { mgr_->update(id_, dt, meas); }
void TargetInterface::update(const double& dt) { mgr_->update(id_, dt); }

namespace {
template <int W> std::array<double, W> readEst(TargetManager* mgr, unsigned id, const double* t1, int which) {
  std::array<double, W> out{};
  std::lock_guard<std::recursive_mutex> lg(mgr->lock());
  SlotRead s;
  if (!locate(mgr, id, s)) return out;
  const uint32_t uid = id;
  ck(te_pool_read_estimates(s.pool, 1, &uid, t1, which == 0 ? out.data() : nullptr, which == 1 ? out.data() : nullptr,
                            which == 2 ? out.data() : nullptr, nullptr, nullptr));
  return out;
}
}  // namespace
Vector7d TargetInterface::getEstimatedPose() const { return readEst<7>(mgr_, id_, nullptr, 0); }
Vector6d TargetInterface::getEstimatedTwist() const { return readEst<6>(mgr_, id_, nullptr, 1); }
Vector6d TargetInterface::getEstimatedAcceleration() const { return readEst<6>(mgr_, id_, nullptr, 2); }
Vector7d TargetInterface::getEstimatedPose(const double& t1) const { return readEst<7>(mgr_, id_, &t1, 0); }
Vector6d TargetInterface::getEstimatedTwist(const double& t1) const { return readEst<6>(mgr_, id_, &t1, 1); }
Vector6d TargetInterface::getEstimatedAcceleration(const double& t1) const { return readEst<6>(mgr_, id_, &t1, 2); }

Vector7d TargetInterface::getMeasuredPose() const {
  Vector7d out{};
  std::lock_guard<std::recursive_mutex> lg(mgr_->lock());
  SlotRead s;
  if (!locate(mgr_, id_, s)) return out;
  const uint32_t uid = id_;
  ck(te_pool_read_state(s.pool, 1, &uid, nullptr, nullptr, nullptr, nullptr, nullptr, out.data()));
  return out;
}
double TargetInterface::getTime() const {
  double t = 0.0;
  std::lock_guard<std::recursive_mutex> lg(mgr_->lock());
  SlotRead s;
  if (!locate(mgr_, id_, s)) return t;
  const uint32_t uid = id_;
  ck(te_pool_read_state(s.pool, 1, &uid, nullptr, nullptr, &t, nullptr, nullptr, nullptr));
  return t;
}
long long TargetInterface::getNumberMeasurements() const {
  long long nm = 0;
  std::lock_guard<std::recursive_mutex> lg(mgr_->lock());
  SlotRead s;
  if (!locate(mgr_, id_, s)) return nm;
  const uint32_t uid = id_;
  ck(te_pool_read_state(s.pool, 1, &uid, nullptr, nullptr, nullptr, &nm, nullptr, nullptr));
  return nm;
}
double TargetInterface::getPeriodEstimate() const {   // src/target_interface.cpp:80-87
  const Vector6d tw = getEstimatedTwist();
  const double n = std::sqrt(tw[3] * tw[3] + tw[4] * tw[4] + tw[5] * tw[5]);
  if (n > 0) return 2 * M_PI / n;
  return -1.0;
}

// ----------------------------------------------------------------------------------------------
// MovingAvgFilter (utils.hpp:222-251)
// ----------------------------------------------------------------------------------------------
double MovingAvgFilter::update(double value) {
  const unsigned n = (unsigned)window_.size();
  sum_ -= window_[idx_];
  sum_ += value;
  window_[idx_] = value;
  if (!complete_ && idx_ == n - 1) complete_ = true;
  const unsigned num = complete_ ? n : idx_ + 1;
  const double res = sum_ / num;
  idx_ = (idx_ + 1) % n;
  variance_ = 0.0;
  for (unsigned k = 0; k < n; ++k) variance_ += (window_[k] - res) * (window_[k] - res);
  variance_ /= num;
  return res;
}

// ----------------------------------------------------------------------------------------------
// IntersectionSolver (src/intersection_solver.cpp:19-124)
// ----------------------------------------------------------------------------------------------
IntersectionSolver::IntersectionSolver(TargetManager::Ptr tm, const unsigned int filters_length, long long n_streams)
    : target_manager_(tm), filters_length_(filters_length), n_streams_(n_streams) {
  if (!tm) throw std::invalid_argument("IntersectionSolver needs a target manager (assert of src/intersection_solver.cpp:21)");
  if (n_streams <= 0 || n_streams > 0x7fffffffLL) throw std::invalid_argument("n_streams must be in [1, 2^31)");
  sharded_ = dynamic_cast<ShardedTargetManager*>(tm.get());
  const int G = sharded_ ? sharded_->shards() : 1;
  solvers_.assign((size_t)G, std::array<te_isolver*, 4>{nullptr, nullptr, nullptr, nullptr});
  part_.resize((size_t)G);
  for (Part& P : part_) P.moves.resize(4 * (size_t)G);
}
IntersectionSolver::~IntersectionSolver() {
  for (auto& per_shard : solvers_)
    for (te_isolver*& s : per_shard) {
      if (s) te_isolver_destroy(s);
      s = nullptr;
    }
}
TargetManager& IntersectionSolver::shardOf(int r) { return sharded_ ? sharded_->shard(r) : *target_manager_; }
te_isolver* IntersectionSolver::solverFor(int r, int type) {
  te_isolver*& s = solvers_[(size_t)r][(size_t)type];
  if (!s) {
    s = te_isolver_create(shardOf(r).poolOf(type, false), n_streams_, filters_length_);
    if (!s) throw PoolError(te_last_error());
  }
  return s;
}
double IntersectionSolver::getIntersectionTimeWithSphere(const unsigned int& id, const double& t1, const Vector3d& origin,
                                                         const double& radius) {   // :44-90
  const int s0 = 0;
  double delta = -1.0;
  query(1, &id, &s0, &t1, origin.data(), &radius, nullptr, nullptr, &delta, nullptr, nullptr);
  return delta;
}
bool IntersectionSolver::getIntersectionPoseWithSphere(const unsigned int& id, const double& t1, const double& pos_th, const double& ang_th,
                                                       const Vector3d& origin, const double& radius, Vector7d& intersection_pose) {   // :92-124
  if (!(t1 >= 0.0) || !(pos_th >= 0.0) || !(ang_th >= 0.0)) throw std::invalid_argument("t1, pos_th, ang_th must be >= 0 (:94-96)");
  intersection_pose = Vector7d{0, 0, 0, 0, 0, 0, 1};   // initPose (:99)
  const int s0 = 0;
  double delta = -1.0;
  uint8_t conv = 0;
  query(1, &id, &s0, &t1, origin.data(), &radius, &pos_th, &ang_th, &delta, intersection_pose.data(), &conv);
  return conv != 0;
}

long long IntersectionSolver::query(long long n, const unsigned* ids, const int* stream, const double* t1, const double* origin,
                                    const double* radius, const double* pos_th, const double* ang_th, double* delta, double* pose7,
                                    unsigned char* converged) {
  if (n < 0) throw std::invalid_argument("negative query count");
  if (n > 0 && (!ids || !t1 || !origin || !radius)) throw std::invalid_argument("ids, t1, origin and radius are required");
  if (pose7 && n > 0 && (!pos_th || !ang_th)) throw std::invalid_argument("thresholds are required with pose7");
  if (!stream && pose7 && n > n_streams_) throw std::invalid_argument("more queries than solver streams (stream NULL = query index)");
  if (stream)
    for (long long k = 0; k < n; ++k)
      if (stream[k] < 0 || stream[k] >= n_streams_) throw std::invalid_argument("bad stream index");
  if (pose7)
    for (long long k = 0; k < n; ++k)
      if (!(t1[k] >= 0.0) || !(pos_th[k] >= 0.0) || !(ang_th[k] >= 0.0)) throw std::invalid_argument("t1, pos_th, ang_th must be >= 0 (:94-96)");
  std::lock_guard<std::recursive_mutex> lg(target_manager_->lock());
  std::fill(phase_ms_, phase_ms_ + 4, 0.0);
  if (n == 0) return 0;
  target_manager_->flush();
  auto run = [&](long long lo, long long hi) {
    return queryRun(hi - lo, ids + lo, stream ? stream + lo : nullptr, t1 + lo, origin + 3 * lo, radius + lo, pos_th ? pos_th + lo : nullptr,
                    ang_th ? ang_th + lo : nullptr, delta ? delta + lo : nullptr, pose7 ? pose7 + 7 * lo : nullptr,
                    converged ? converged + lo : nullptr);
  };
  // only queries with pose7 touch a stream: those are cut in front of every repeated stream, as TargetManager::updateBatch cuts
  // in front of a repeated id
  if (!stream || !pose7) return run(0, n);
  if (seen_.empty()) seen_.assign((size_t)n_streams_, 0);
  auto next_gen = [&] {
    if (++gen_ == 0) {
      std::fill(seen_.begin(), seen_.end(), 0u);
      gen_ = 1;
    }
  };
  next_gen();
  long long found = 0, start = 0;
  for (long long k = 0; k < n; ++k) {
    unsigned& mark = seen_[(size_t)stream[k]];
    if (mark == gen_) {
      found += run(start, k);
      start = k;
      next_gen();
    }
    seen_[(size_t)stream[k]] = gen_;
  }
  return found + run(start, n);
}

// the model type(s) of shard r's targets: one pool in use -> every query goes to it (the kernel finds unknown ids itself); several
// -> the queries split by model type on the host
void IntersectionSolver::classify(int r, long long m, const unsigned* ids) {
  Part& P = part_[(size_t)r];
  TargetManager& M = shardOf(r);
  std::lock_guard<std::recursive_mutex> lg(M.lock());
  P.only = onlyType(M.heldTypes());
  if (P.only == -2) M.rowsByType(m, ids, P.rows);
}

// the streams shard r queries whose state lives on another shard, grouped by (model type, source); home_ then names r.  (A stream
// appears once per piece, so the shards' workers touch disjoint entries of home_.)
void IntersectionSolver::collectMoves(int r, long long m, const int* stream) {
  Part& P = part_[(size_t)r];
  const int G = (int)part_.size();
  for (auto& v : P.moves) v.clear();
  auto visit = [&](int t, long long j) {
    int& h = home_[(size_t)t * (size_t)n_streams_ + (size_t)stream[j]];
    if (h >= 0 && h != r) P.moves[(size_t)t * G + (size_t)h].push_back(stream[j]);
    h = r;
  };
  if (P.only >= 0)
    for (long long j = 0; j < m; ++j) visit(P.only, j);
  else if (P.only == -2)
    for (int t = 0; t < 4; ++t)
      for (long long j : P.rows[t]) visit(t, j);
}

long long IntersectionSolver::queryShard(int r, long long m, const unsigned* ids, const int* stream, const double* t1, const double* origin,
                                         const double* radius, const double* pos_th, const double* ang_th, double* delta, double* pose7,
                                         unsigned char* conv) {
  Part& P = part_[(size_t)r];
  std::lock_guard<std::recursive_mutex> lg(shardOf(r).lock());
  if (!pose7) stream = nullptr;   // times only: no stream is read (and stream NULL = k may exceed the streams then)
  if (P.only >= 0) {
    const long long rc = te_isolver_query(solverFor(r, P.only), m, ids, stream, t1, origin, radius, pos_th, ang_th, delta, pose7, conv);
    ck(rc);
    return rc;
  }
  static const double init_pose[7] = {0, 0, 0, 0, 0, 0, 1};
  for (long long j = 0; j < m; ++j) {   // unknown ids (all of them on a shard without targets)
    if (delta) delta[j] = -1.0;
    if (pose7) std::memcpy(pose7 + 7 * j, init_pose, sizeof(init_pose));
    if (conv) conv[j] = 0;
  }
  if (P.only == -1) return 0;
  std::vector<int> by_row;   // stream NULL = the query's row
  if (pose7 && !stream) {
    by_row.resize((size_t)m);
    std::iota(by_row.begin(), by_row.end(), 0);
    stream = by_row.data();
  }
  long long found = 0;
  std::vector<unsigned> s_ids;
  std::vector<int> s_stream;
  std::vector<double> s_t1, s_origin, s_radius, s_pth, s_ath, s_delta((size_t)m), s_pose(pose7 ? 7 * (size_t)m : 0);
  std::vector<unsigned char> s_conv(pose7 ? (size_t)m : 0);
  for (int t = 0; t < 4; ++t) {   // one sub-batch per model type
    const std::vector<long long>& rows = P.rows[t];
    if (rows.empty()) continue;
    const long long rc = te_isolver_query(solverFor(r, t), (long long)rows.size(), gatherRows<1>(ids, rows, s_ids), gatherRows<1>(stream, rows, s_stream),
                                          gatherRows<1>(t1, rows, s_t1), gatherRows<3>(origin, rows, s_origin), gatherRows<1>(radius, rows, s_radius),
                                          gatherRows<1>(pos_th, rows, s_pth), gatherRows<1>(ang_th, rows, s_ath), s_delta.data(),
                                          pose7 ? s_pose.data() : nullptr, pose7 ? s_conv.data() : nullptr);
    ck(rc);
    found += rc;
    scatterRows<1>(delta, rows, s_delta.data());
    scatterRows<7>(pose7, rows, s_pose.data());
    scatterRows<1>(pose7 ? conv : nullptr, rows, s_conv.data());
  }
  return found;
}

long long IntersectionSolver::queryRun(long long n, const unsigned* ids, const int* stream, const double* t1, const double* origin,
                                       const double* radius, const double* pos_th, const double* ang_th, double* delta, double* pose7,
                                       unsigned char* converged) {
  typedef std::chrono::steady_clock clk;
  auto ms_since = [](clk::time_point a) { return std::chrono::duration<double, std::milli>(clk::now() - a).count(); };
  const int G = (int)part_.size();
  clk::time_point t0 = clk::now();
  if (G == 1 && !sharded_) {   // a plain manager: the caller's arrays as they are
    classify(0, n, ids);
    phase_ms_[0] += ms_since(t0);
    t0 = clk::now();
    const long long found = queryShard(0, n, ids, stream, t1, origin, radius, pos_th, ang_th, delta, pose7, converged);
    phase_ms_[2] += ms_since(t0);
    return found;
  }
  // 1. route: every shard's queries in call order
  const FastMod owner_of((unsigned)G);
  const bool with_pose = pose7 != nullptr;
  const std::vector<size_t> total = sharded_->routeOnHost(
      n, ids,
      [&](int r, size_t m) {
        Part& P = part_[(size_t)r];
        P.ids.resize(m); P.where.resize(m); P.stream.resize(m); P.t1.resize(m); P.origin.resize(3 * m); P.radius.resize(m);
        P.pos_th.resize(with_pose ? m : 0); P.ang_th.resize(with_pose ? m : 0);
        P.delta.resize(m); P.pose.resize(with_pose ? 7 * m : 0); P.conv.resize(m);
      },
      [&](int, long long lo, long long hi, size_t* at) {
        for (long long k = lo; k < hi; ++k) {
          const unsigned r = owner_of(ids[k]);
          Part& P = part_[r];
          const size_t j = at[r]++;
          P.ids[j] = ids[k];
          P.where[j] = k;
          P.stream[j] = stream ? stream[k] : (int)k;
          P.t1[j] = t1[k];
          std::memcpy(&P.origin[3 * j], origin + 3 * k, 24);
          P.radius[j] = radius[k];
          if (with_pose) { P.pos_th[j] = pos_th[k]; P.ang_th[j] = ang_th[k]; }
        }
      });
  if (with_pose && home_.empty()) home_.assign(4 * (size_t)n_streams_, -1);
  sharded_->forEachShard([&](int r) {
    const long long m = (long long)total[(size_t)r];
    classify(r, m, part_[(size_t)r].ids.data());
    if (with_pose) collectMoves(r, m, part_[(size_t)r].stream.data());
  });
  phase_ms_[0] += ms_since(t0);
  // 2. move the state of every stream that changes shard, one group per (model type, source, destination), before any query
  t0 = clk::now();
  if (with_pose)
    for (int r = 0; r < G; ++r)
      for (int t = 0; t < 4; ++t)
        for (int h = 0; h < G; ++h) {
          const std::vector<int>& v = part_[(size_t)r].moves[(size_t)t * G + (size_t)h];
          if (!v.empty()) ck(te_isolver_move_streams(solverFor(h, t), solverFor(r, t), (long long)v.size(), v.data()));
        }
  phase_ms_[1] += ms_since(t0);
  // 3. every shard queries at once
  t0 = clk::now();
  sharded_->forEachShard([&](int r) {
    Part& P = part_[(size_t)r];
    const long long m = (long long)total[(size_t)r];
    P.found = m == 0 ? 0
                     : queryShard(r, m, P.ids.data(), P.stream.data(), P.t1.data(), P.origin.data(), P.radius.data(),
                                  with_pose ? P.pos_th.data() : nullptr, with_pose ? P.ang_th.data() : nullptr, P.delta.data(),
                                  with_pose ? P.pose.data() : nullptr, with_pose ? P.conv.data() : nullptr);
  });
  phase_ms_[2] += ms_since(t0);
  // 4. results into call order (rows of different shards are disjoint)
  t0 = clk::now();
  long long found = 0;
  for (const Part& P : part_) found += P.found;
  if (converged && !with_pose) std::memset(converged, 0, (size_t)n);
  sharded_->forEachShard([&](int r) {
    const Part& P = part_[(size_t)r];
    scatterRows<1>(delta, P.where, P.delta.data());
    scatterRows<7>(pose7, P.where, P.pose.data());
    scatterRows<1>(with_pose ? converged : nullptr, P.where, P.conv.data());
  });
  phase_ms_[3] += ms_since(t0);
  return found;
}

long long IntersectionSolver::earliestIntersections(long long q, const double* t1, const double* origin, const double* radius, long long k,
                                                    unsigned* ids_out, double* delta_out, long long* hits_out) {
  if (q < 0) throw std::invalid_argument("q must be >= 0");
  if (k < 0 || k > 65536) throw std::invalid_argument("k must be in [0, 65536]");
  if (q > 0 && (!t1 || !origin || !radius || !hits_out)) throw std::invalid_argument("t1, origin, radius and hits_out are required");
  if (q > 0 && k > 0 && (!ids_out || !delta_out)) throw std::invalid_argument("ids_out and delta_out are required when k > 0");
  std::lock_guard<std::recursive_mutex> lg(target_manager_->lock());
  if (q == 0) return 0;
  target_manager_->flush();
  std::vector<TargetManager*> shards;
  for (int r = 0; r < (int)solvers_.size(); ++r) shards.push_back(&shardOf(r));
  return sweep_.run(
      shards, [&](const std::function<void(int)>& f) { sharded_ ? sharded_->forEachShard(f) : f(0); }, q, k,
      [&](te_pool* p, unsigned* ids, double* delta, long long* hits) {
        return te_pool_earliest_intersections(p, q, t1, origin, radius, k, ids, delta, hits);
      },
      ids_out, delta_out, hits_out);
}

long long PoolRowMerge::run(const std::vector<TargetManager*>& shards, const std::function<void(const std::function<void(int)>&)>& each_shard,
                            long long q, long long k, const PoolQuery& query, unsigned* ids_out, double* val_out, long long* count_out) {
  const int G = (int)shards.size();
  if (lists_.size() < 4 * (size_t)G) lists_.resize(4 * (size_t)G);
  int n_lists = 0, only = -1;
  for (int r = 0; r < G; ++r) {
    const unsigned held = shards[(size_t)r]->heldTypes();
    for (int t = 0; t < 4; ++t) {
      List& L = lists_[(size_t)r * 4 + (size_t)t];
      L.used = (held >> t) & 1u;
      if (L.used) { ++n_lists; only = r * 4 + t; }
    }
  }
  auto run_pool = [&](int r, int t, unsigned* ids, double* val, long long* count) {
    TargetManager& M = *shards[(size_t)r];
    std::lock_guard<std::recursive_mutex> lk(M.lock());
    ck(query(M.poolOf(t, false), ids, val, count));
  };
  if (n_lists == 1) {   // one pool holds every target: its rows are the answer
    run_pool(only / 4, only % 4, ids_out, val_out, count_out);
  } else {
    auto run_shard = [&](int r) {
      for (int t = 0; t < 4; ++t) {
        List& L = lists_[(size_t)r * 4 + (size_t)t];
        if (!L.used) continue;
        L.ids.resize((size_t)(q * k)); L.val.resize((size_t)(q * k)); L.count.resize((size_t)q);
        run_pool(r, t, L.ids.data(), L.val.data(), L.count.data());
      }
    };
    // merge query j's sorted lists by (rank(value), id): -0.0 ranks as 0, a non-negative double's bits order like its value
    auto rank = [](double d) {
      unsigned long long b;
      std::memcpy(&b, &d, 8);
      return b == 0x8000000000000000ull ? 0ull : b;
    };
    std::vector<const List*> used;
    for (int l = 0; l < 4 * G; ++l)
      if (lists_[(size_t)l].used) used.push_back(&lists_[(size_t)l]);
    auto merge = [&](long long j, std::vector<long long>& at) {
      long long count = 0;
      for (const List* L : used) count += L->count[(size_t)j];
      count_out[j] = count;
      at.assign(used.size(), 0);
      for (long long row = 0; row < k; ++row) {
        int best = -1;
        unsigned long long best_rank = 0;
        unsigned best_id = 0;
        for (size_t l = 0; l < used.size(); ++l) {
          const List& L = *used[l];
          if (at[l] >= std::min(k, L.count[(size_t)j])) continue;
          const size_t o = (size_t)(j * k + at[l]);
          const unsigned long long rk = rank(L.val[o]);
          if (best < 0 || rk < best_rank || (rk == best_rank && L.ids[o] < best_id)) { best = (int)l; best_rank = rk; best_id = L.ids[o]; }
        }
        const size_t out = (size_t)(j * k + row);
        if (best < 0) {
          ids_out[out] = 0xFFFFFFFFu;
          val_out[out] = -1.0;
        } else {
          const size_t o = (size_t)(j * k + at[(size_t)best]++);
          ids_out[out] = used[(size_t)best]->ids[o];
          val_out[out] = used[(size_t)best]->val[o];
        }
      }
    };
    // every shard's pools at once, then the queries' merges spread over the shards' workers
    each_shard(run_shard);
    each_shard([&](int r) {
      std::vector<long long> at;
      for (long long j = r; j < q; j += G) merge(j, at);
    });
  }
  long long total = 0;
  for (long long j = 0; j < q; ++j) total += count_out[j];
  return total;
}

long long TargetManager::nearestTargets(long long q, const double* t1, const double* point, const double* radius, long long k,
                                        unsigned* ids_out, double* dist_out, long long* count_out) {
  te::check_query_args(te::NEAREST_ARGS, q, point, radius, k, ids_out, dist_out, count_out);
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  if (q == 0) return 0;
  flushLocked();
  return nearest_rows_.run(
      {this}, [](const std::function<void(int)>& f) { f(0); }, q, k,
      [&](te_pool* p, unsigned* ids, double* dist, long long* count) {
        return te_pool_nearest_targets(p, q, t1, point, radius, k, ids, dist, count);
      },
      ids_out, dist_out, count_out);
}

long long TargetManager::gatedTargets(long long q, const double* t1, const double* z, const double* gate, long long k, unsigned* ids_out,
                                      double* d2_out, long long* count_out) {
  te::check_query_args(te::GATE_ARGS, q, z, gate, k, ids_out, d2_out, count_out);
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  if (q == 0) return 0;
  flushLocked();
  return gated_rows_.run(
      {this}, [](const std::function<void(int)>& f) { f(0); }, q, k,
      [&](te_pool* p, unsigned* ids, double* d2, long long* count) { return te_pool_gated_targets(p, q, t1, z, gate, k, ids, d2, count); },
      ids_out, d2_out, count_out);
}

long long TargetManager::associate(double t1, long long q, const double* det, double gate, int K, int apply, unsigned* id_out, double* d2_out,
                                   long long* count_out) {
  te::check_assoc_args(te::ASSOC_ARGS, t1, q, det, gate, K, id_out, d2_out);
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  if (q == 0) return 0;
  flushLocked();
  return associateOver(
      {this}, [](const std::function<void(int)>& f) { f(0); }, t1, q, det, gate, K, apply, id_out, d2_out, count_out,
      [&](long long n, const unsigned* ids, const double* rec) { updateAt(t1, n, ids, rec); });
}

long long TargetManager::associateOver(const std::vector<TargetManager*>& shards, const std::function<void(const std::function<void(int)>&)>& each_shard,
                                       double t1, long long q, const double* det, double gate, int K, int apply, unsigned* id_out, double* d2_out,
                                       long long* count_out, const std::function<void(long long, const unsigned*, const double*)>& update) {
  int n_pools = 0, first = -1;   // first = shard * 4 + type of the first pool that holds targets
  for (int r = 0; r < (int)shards.size(); ++r) {
    const unsigned held = shards[(size_t)r]->heldTypes();
    for (int t = 0; t < 4; ++t)
      if ((held >> t) & 1u) {
        ++n_pools;
        if (first < 0) first = r * 4 + t;
      }
  }
  auto on_first = [&](const std::function<long long(te_pool*)>& f) {
    TargetManager& M = *shards[(size_t)(first / 4)];
    std::lock_guard<std::recursive_mutex> lk(M.lock());
    const long long rc = f(M.poolOf(first % 4, false));
    ck(rc);
    return rc;
  };
  if (n_pools == 0) {
    std::fill(id_out, id_out + q, 0xFFFFFFFFu);
    std::fill(d2_out, d2_out + q, -1.0);
    if (count_out) std::fill(count_out, count_out + q, 0LL);
    return 0;
  }
  if (n_pools == 1)   // one pool holds every target: the whole frame on its device
    return on_first([&](te_pool* p) { return te_pool_associate(p, t1, q, det, gate, K, apply, id_out, d2_out, count_out); });
  // every pool's candidate lists, merged by (d^2, id) as gatedTargets merges them; the matching on the first pool's device
  std::vector<double> z((size_t)q * 3);
  for (long long j = 0; j < q; ++j) std::memcpy(&z[(size_t)j * 3], det + 7 * (size_t)j, 24);
  std::vector<unsigned> rows_id((size_t)(q * K));
  std::vector<double> rows_d2((size_t)(q * K));
  std::vector<long long> count((size_t)q);
  assoc_rows_.run(
      shards, each_shard, q, K,
      [&](te_pool* p, unsigned* ids, double* d2, long long* cnt) { return te_pool_gated_candidates(p, t1, q, z.data(), gate, K, ids, d2, cnt); },
      rows_id.data(), rows_d2.data(), count.data());
  const long long assigned =
      on_first([&](te_pool* p) { return te_assign_greedy(p, q, K, rows_id.data(), rows_d2.data(), id_out, d2_out); });
  if (count_out) std::copy(count.begin(), count.end(), count_out);
  if (apply && assigned > 0) {
    std::vector<unsigned> ids;
    std::vector<double> rec;
    ids.reserve((size_t)assigned);
    rec.reserve((size_t)assigned * 7);
    for (long long j = 0; j < q; ++j)
      if (d2_out[j] >= 0.0) {
        ids.push_back(id_out[j]);
        rec.insert(rec.end(), det + 7 * (size_t)j, det + 7 * (size_t)j + 7);
      }
    update((long long)ids.size(), ids.data(), rec.data());
  }
  return assigned;
}

void TargetManager::updateAt(double t1, long long n, const unsigned* ids, const double* det) {
  std::lock_guard<std::recursive_mutex> lg(target_lock_);
  std::vector<long long> rows[4];
  rowsByType(n, ids, rows);
  for (int t = 0; t < 4; ++t) {
    if (rows[t].empty()) continue;
    std::vector<unsigned> t_ids;
    std::vector<double> t_det;
    ck(te_pool_update_at(poolOf(t, false), (long long)rows[t].size(), gatherRows<1>(ids, rows[t], t_ids), t1, gatherRows<7>(det, rows[t], t_det)));
  }
}

// ----------------------------------------------------------------------------------------------
// utils.hpp:273-313
// ----------------------------------------------------------------------------------------------
std::vector<std::string> splitString(const std::string& s, const std::string& delimiter) {
  std::vector<std::string> res;
  size_t start = 0, end;
  while ((end = s.find(delimiter, start)) != std::string::npos) {
    res.push_back(s.substr(start, end - start));
    start = end + delimiter.length();
  }
  res.push_back(s.substr(start));
  return res;
}
bool getId(const std::string& s, unsigned int& id) {
  auto parts = splitString(s);
  if (parts.size() == 2) {   // 'xxx_id'
    id = (unsigned)std::stoi(parts[1]);   // throws like the reference on a non-numeric suffix
    return true;
  }
  return false;
}

}  // namespace target_estimation_b200
