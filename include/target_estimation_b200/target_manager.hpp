// include/target_estimation_b200/target_manager.hpp -- host surface of the B200 target pool.
//
// Mirrors the reference's TargetManager / TargetInterface / IntersectionSolver API
// (/root/reference/include/target_estimation/target_manager.hpp:30-270, target_interface.hpp:39-283,
// intersection_solver.hpp:55-125; tick/expiry semantics of target_manager_ros.hpp:74-183) with the
// same method names, argument order, return conventions and quirks.  Storage is not one heap object per
// target: every call lands in the device-resident pools of include/te_pool.h.  Eigen is not a
// dependency of this build (absent from the image), so Vector7d / Vector6d / MatrixXd are the
// plain fixed/dynamic arrays below; INTEGRATION.md shows the Eigen::Map overloads a maintainer adds.
//
// Per-id calls (update(id,dt,meas), update(id,dt)) are queued and coalesced: the reference's
// "for every id: update(id, dt, meas)" loop of one tick becomes ONE kernel launch at the next
// getter / flush / repeated id.  Observable results are identical to immediate execution.
#pragma once
#include <array>
#include <cstdint>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "../te_pool.h"

namespace target_estimation_b200 {

typedef std::array<double, 3> Vector3d;
typedef std::array<double, 6> Vector6d;
typedef std::array<double, 7> Vector7d;

struct MatrixXd {   // dense row-major dynamic matrix (only what the API needs)
  int r = 0, c = 0;
  std::vector<double> d;
  MatrixXd() {}
  MatrixXd(int rows, int cols) : r(rows), c(cols), d((size_t)rows * cols, 0.0) {}
  double& operator()(int i, int j) { return d[(size_t)i * c + j]; }
  double operator()(int i, int j) const { return d[(size_t)i * c + j]; }
  int rows() const { return r; }
  int cols() const { return c; }
  const double* data() const { return d.data(); }
};
typedef std::vector<double> VectorXd;

class TargetManager;

// The k smallest (value, id) rows of q queries over every (shard, model type) pool that holds targets: what
// IntersectionSolver::earliestIntersections, TargetManager::nearestTargets and TargetManager::gatedTargets share.  Each pool selects
// its own rows on the device (te_pool_earliest_intersections / te_pool_nearest_targets / te_pool_gated_targets: per query, rows by
// (value, id), then id 0xFFFFFFFF / value -1, and a count); the host merges the lists of each query by (value, id) -- a candidate's
// value is a non-negative double, -0.0 ranks as 0 -- and sums the counts.  When one pool holds every target its rows are the
// answer.  The lists' buffers only grow.
class PoolRowMerge {
 public:
  // one pool's rows [q][k] and counts [q]: returns < 0 on error (te_last_error())
  typedef std::function<long long(te_pool*, unsigned* ids, double* val, long long* count)> PoolQuery;
  // each_shard(f) runs f(r) for every r < shards.size(), possibly at once; pool calls hold the shard's lock.  Returns the total count.
  long long run(const std::vector<TargetManager*>& shards, const std::function<void(const std::function<void(int)>&)>& each_shard,
                long long q, long long k, const PoolQuery& query, unsigned* ids_out, double* val_out, long long* count_out);

 private:
  struct List {   // the sorted rows of one (shard, model type) pool
    std::vector<unsigned> ids;
    std::vector<double> val;
    std::vector<long long> count;
    bool used = false;
  };
  std::vector<List> lists_;   // [shard * 4 + model type]
};

// id -> model type, ascending ids: the host registry behind getAvailableTargets / "already exists" / "does not exist".  The
// reference's std::map<unsigned, TargetInterface::Ptr> (target_manager.hpp:36) node-per-target layout costs a cache miss per
// tree level: erasing the 10 k ids that expire in one tick of a million-target pool took 10 ms.  A sorted flat vector keeps the
// map's interface for the by-id calls (binary search; appending ids in ascending order is O(1)) and adds linear-time merges
// for the batches a tick produces.
class IdRegistry {
 public:
  typedef std::pair<unsigned, uint8_t> value_type;
  typedef std::vector<value_type>::iterator iterator;
  typedef std::vector<value_type>::const_iterator const_iterator;
  iterator begin() { return v_.begin(); }
  iterator end() { return v_.end(); }
  const_iterator begin() const { return v_.begin(); }
  const_iterator end() const { return v_.end(); }
  size_t size() const { return v_.size(); }
  bool empty() const { return v_.empty(); }
  iterator find(unsigned id);
  size_t count(unsigned id) { return find(id) != v_.end() ? 1 : 0; }
  uint8_t& operator[](unsigned id);                 // inserts (type 0) if missing, like std::map
  iterator erase(iterator it) { return v_.erase(it); }
  size_t erase(unsigned id);
  template <class It> void insert(It first, It last) {   // range of (id, type) pairs in ascending id order; existing ids are kept
    std::vector<value_type> add(first, last);
    mergeSorted(add);
  }
  void insertSorted(const uint32_t* ids, size_t n, uint8_t type);   // ascending ids
  void eraseSorted(const uint32_t* ids, size_t n);                  // ascending ids; unknown ones are ignored
 private:
  void mergeSorted(const std::vector<value_type>& add);
  std::vector<value_type> v_;
};

// KalmanFilterInterface view (kalman.hpp:49-89): what test/target_manager_test.cpp:144 reads
class EstimatorView {
 public:
  EstimatorView(TargetManager* m, unsigned id) : mgr_(m), id_(id) {}
  VectorXd getState() const;
  MatrixXd getP() const;
  MatrixXd getQ() const;
  MatrixXd getR() const;
  MatrixXd getP0() const;
 private:
  TargetManager* mgr_;
  unsigned id_;
};

// TargetInterface proxy (target_interface.hpp:58-160): every getter reads the target's slot back from
// the device (a sync point).  A handle may outlive erase(); its getters then return zeros.
class TargetInterface {
 public:
  typedef std::shared_ptr<TargetInterface> Ptr;
  TargetInterface(TargetManager* m, unsigned id) : mgr_(m), id_(id), est_(m, id) {}
  void addMeasurement(const double& dt, const Vector7d& meas);
  void update(const double& dt);
  Vector7d getEstimatedPose() const;
  Vector6d getEstimatedTwist() const;
  Vector6d getEstimatedAcceleration() const;
  Vector7d getEstimatedPose(const double& t1) const;
  Vector6d getEstimatedTwist(const double& t1) const;
  Vector6d getEstimatedAcceleration(const double& t1) const;
  Vector7d getMeasuredPose() const;
  double getTime() const;
  double getPeriodEstimate() const;   // src/target_interface.cpp:80-87
  long long getNumberMeasurements() const;
  unsigned getID() const { return id_; }
  const EstimatorView* getEstimator() const { return &est_; }
 private:
  TargetManager* mgr_;
  unsigned id_;
  EstimatorView est_;
};

class TargetManager {
 public:
  typedef std::shared_ptr<TargetManager> Ptr;
  enum target_t { ANGULAR_RATES = 0, ANGULAR_VELOCITIES, UNIFORM_ACCELERATION, UNIFORM_VELOCITY };   // target_manager.hpp:38

  explicit TargetManager(int device = 0);
  explicit TargetManager(const std::string& file, int device = 0);   // throws const char* like the reference (:110-118)
  virtual ~TargetManager();

  // reference API ---------------------------------------------------------------------------
  virtual void init(const unsigned int& id, const double& dt0, const double& t0, const Vector7d& p0, const Vector6d& v0 = Vector6d{},
                    const Vector6d& a0 = Vector6d{});
  virtual void init(const target_t& type, const unsigned int& id, const double& dt0, const double& t0, const MatrixXd& Q, const MatrixXd& R,
                    const MatrixXd& P0, const Vector7d& p0, const Vector6d& v0 = Vector6d{}, const Vector6d& a0 = Vector6d{});
  void init(const std::string& file, const unsigned int& id, const double& dt0, const double& t0, const Vector7d& p0,
            const Vector6d& v0 = Vector6d{}, const Vector6d& a0 = Vector6d{});
  virtual bool update(const unsigned int& id, const double& dt, const Vector7d& meas);
  virtual bool update(const unsigned int& id, const double& dt);
  virtual void update(const double& dt);
  virtual bool erase(const unsigned int& id);
  virtual TargetInterface::Ptr getTarget(const unsigned int& id);
  virtual bool getTargetPose(const unsigned int& id, Vector7d& pose);
  virtual bool getTargetTwist(const unsigned int& id, Vector6d& twist);
  virtual bool getTargetAcceleration(const unsigned int& id, Vector6d& acc);
  virtual long long getNumberMeasurements(const unsigned int& id);
  virtual void log();
  virtual std::vector<unsigned int> getAvailableTargets();
  bool selectTargetType(const std::string& type_str, target_t& type);
  bool loadYamlFile(const std::string& file, MatrixXd& Q, MatrixXd& R, MatrixXd& P, target_t& type);

  // batched extensions (one kernel launch per call) ---------------------------------------------
  long long initBatch(long long n, const unsigned* ids, double dt0, const double* t0, const double* p0 /*[n][7]*/,
                      const double* v0 = nullptr, const double* a0 = nullptr);
  virtual long long initBatch(target_t type, const MatrixXd& Q, const MatrixXd& R, const MatrixXd& P0, long long n, const unsigned* ids, double dt0,
                              const double* t0, const double* p0, const double* v0 = nullptr, const double* a0 = nullptr,
                              const double* p0_scale = nullptr);
  // (an id may appear more than once: the records are applied in order, as the reference's sequential update() calls would --
  //  the batch is cut in front of every repeat and the pieces are launched one after the other; meas may be NULL only when no
  //  record is an UPDATE -- action NULL means UPDATE for every record -- else std::invalid_argument before any pool is stepped)
  virtual long long updateBatch(long long n, const unsigned* ids, double dt, const double* meas /*[n][7]*/, const unsigned char* action = nullptr);
  virtual long long eraseBatch(long long n, const unsigned* ids);
  virtual void getEstimatesBatch(long long n, const unsigned* ids, const double* t1, double* pose7, double* twist6, double* acc6,
                                 unsigned char* found);
  virtual void flush();
  // The k nearest targets inside a sphere at a given time, over every target of the manager (te_pool_nearest_targets on every
  // (shard, model type) pool that holds targets; the shards of a sharded manager run at once).  Query j = (t1[j], point[j][3],
  // radius[j]), t1 NULL = every target's current estimate.  The position of target i is pose7[0:3] of getEstimatesBatch({i}, {t1[j]})
  // bit for bit; dist = sqrt((dx^2 + dy^2) + dz^2), every operation rounded on its own; inside = dist <= radius[j].  count_out[j] =
  // the number of targets inside; rows 0 .. min(k, count) - 1 of ids_out[j][.] / dist_out[j][.] are those targets by (dist, id),
  // the other rows id 0xFFFFFFFF and dist -1.  The result does not depend on the shard count or on which pool holds a target.
  // Read-only; queued per-id calls are flushed first.  0 <= k <= 65536 (k == 0: counts only, ids_out / dist_out may be NULL); a
  // negative or NaN radius is an error, +inf asks for the k nearest of all.  Returns the total count.
  virtual long long nearestTargets(long long q, const double* t1 /*[q] or NULL*/, const double* point /*[q][3]*/, const double* radius,
                                   long long k, unsigned* ids_out /*[q][k]*/, double* dist_out /*[q][k]*/, long long* count_out /*[q]*/);
  // Gating: the k targets with the smallest Mahalanobis distance to a measured position, over every target of the manager
  // (te_pool_gated_targets on every (shard, model type) pool that holds targets; the shards of a sharded manager run at once).  Query
  // j = (t1[j], z[j][3], gate[j]); for target i with state x, covariance P, time t and model class (Q, R):
  //  1. p = pose7[0:3] of getEstimatesBatch({i}, {t1[j]}) bit for bit (the position nearestTargets uses); t1 NULL: the current estimate.
  //  2. C (3 x 3): P, Q, R are read through their upper triangle ((r, c) with r > c from (c, r)).  t1 NULL: C(a,b) = P(a,b), no
  //     predict, no Q.  t1 given: the position block of A(tau) P A(tau)^T + Q, tau = t1[j] - t, h = (0.5*tau)*tau, every operation
  //     rounded on its own: with the position-derivative offsets o = UV (0, 3), UA (0, 3, 6), AR (0, 6, 12), AV (0, 6) and
  //     m[u][v] = P(o_u + a, o_v + b), rows r[v] = (m[0][v] + tau*m[1][v]) + h*m[2][v], then c = (r[0] + tau*r[1]) + h*r[2] (h terms
  //     only with three offsets), C(a,b) = c + Q(a,b).
  //  3. S = C + R[0:3,0:3].
  //  4. d = p - z[j]; L00 = sqrt(S00), L10 = S10/L00, L20 = S20/L00, L11 = sqrt(S11 - L10*L10), L21 = (S21 - L20*L10)/L11,
  //     L22 = sqrt((S22 - L20*L20) - L21*L21); w0 = d0/L00, w1 = (d1 - L10*w0)/L11, w2 = ((d2 - L20*w0) - L21*w1)/L22;
  //     d^2 = (w0*w0 + w1*w1) + w2*w2.  A target whose factor does not exist (a radicand <= 0 or NaN) is never a candidate.
  //  5. inside = d^2 <= gate[j]; count_out[j] = the number of targets inside; rows 0 .. min(k, count) - 1 of ids_out[j][.] /
  //     d2_out[j][.] are those targets by (d^2, id), the other rows id 0xFFFFFFFF and d^2 -1.
  //  6. The result does not depend on the shard count or on which pool holds a target.  Read-only; queued per-id calls are flushed
  //     first.  Returns the total count.
  //  7. 0 <= k <= 65536 (k == 0: counts only, ids_out / d2_out may be NULL); a negative or NaN gate is an error, +inf asks for the k
  //     smallest distances over every target whose S has a factor.
  // Position only, for every model: for UV / UA the filter's full innovation, for AR / AV the exact position marginal of the 6-D one.
  virtual long long gatedTargets(long long q, const double* t1 /*[q] or NULL*/, const double* z /*[q][3]*/, const double* gate /*[q]*/,
                                 long long k, unsigned* ids_out /*[q][k]*/, double* d2_out /*[q][k]*/, long long* count_out /*[q]*/);
  // Association of one frame of unlabelled position detections (contract of te_pool_associate in include/te_pool.h, INTEGRATION.md
  // section 12): all q detections are stamped t1, detection j is the pose record det[j][0:7] and is gated on det[j][0:3].
  //  1. Target i is a candidate for j when t_i <= t1 (NaN never) and d^2 <= gate, d^2 bit for bit gatedTargets' for (t1, det[j][0:3]);
  //     count_out[j] (may be NULL) = the number of candidates; j's candidate list = its first min(K, count) by (d^2, id) -- when every
  //     target has t <= t1, gatedTargets(k = K)'s rows.
  //  2. Greedy on sorted edges: the edges of all candidate lists in ascending (d^2, id, j) order, each taken when neither end is
  //     taken yet.  id_out[j] / d2_out[j] = the assigned target and its d^2, 0xFFFFFFFF / -1 without one.  A detection whose K
  //     candidates all go to better edges stays unassigned.
  //  3. apply = 1: every assigned target i gets update(i, t1 - t_i, det[j]) (dt rounded once, bit for bit te_pool_step_ids with that
  //     dt); nothing else changes.  apply = 0: read-only.  Queued per-id calls are flushed first in both modes.  On a tick handle the
  //     update is a by-hand update, as updateBatch's.
  //  4. The result does not depend on the shard count, on which (shard, model type) pool holds a target, or on slot order.
  //  5. std::invalid_argument, nothing applied: t1 not finite; gate negative, NaN or +inf; K outside [1, 32]; q < 0; det, id_out or
  //     d2_out NULL while q > 0.
  // One pool holding every target runs te_pool_associate; otherwise every pool's te_pool_gated_candidates (the shards at once) are
  // merged by (d^2, id) as gatedTargets merges, te_assign_greedy runs on the first pool's device, and the assigned records go to
  // their pools' te_pool_update_at.  Returns the number of assigned detections.
  virtual long long associate(double t1, long long q, const double* det /*[q][7]*/, double gate, int K, int apply, unsigned* id_out /*[q]*/,
                              double* d2_out /*[q]*/, long long* count_out /*[q] or NULL*/);
  // One dense tick from host arrays, record k = the k-th target in denseIds() order (a homogeneous manager: getAvailableTargets()
  // order): no ids travel, nothing is looked up -- te_pool_tick_host: the copies, the step and the read-back of every target's
  // estimated position (est_pos_out [n][3], may be NULL: what the node broadcasts per tick, src/target_manager_ros.cpp:78-87) are
  // pipelined in chunks.  meas_stride 7 = poses, 3 = x y z (UV / UA).  action NULL = update(id, dt, meas) for every target.
  // updateDenseAsync enqueues the tick and returns (two ticks may be in flight; buffers must stay valid until the tick is done);
  // updateDenseWait(0) waits for all of them, (1) for all but the newest.  Returns the number of targets.
  virtual long long updateDense(double dt, const double* meas, int meas_stride, const unsigned char* action, double* est_pos_out);
  virtual long long updateDenseAsync(double dt, const double* meas, int meas_stride, const unsigned char* action, double* est_pos_out);
  virtual void updateDenseWait(int lag);
  virtual std::vector<unsigned int> denseIds();
  size_t size();   // number of targets (of this manager / shard)
  bool quiet = false;   // suppress the reference's stdout messages ("does not exist", "already exists", ...)

  // sampled logging -----------------------------------------------------------------------------
  // The reference's log() (src/target_manager.cpp:119-123 -> src/target_interface.cpp:50-55, under LOGGER_ON) publishes, per
  // target, measured_pose_, pose_internal_, twist_, acceleration_ and P_ through rt_logger (:32-40); its tests dump time / pose /
  // twist series with writeTxtFile (utils.hpp:78-120) for matlab/plot_*.m.  Here log() appends ONE batched read-back of those five
  // quantities for the watched ids to an in-memory series, and writeLog() dumps them in writeTxtFile's format.
  virtual void watch(long long n, const unsigned* ids, size_t max_samples = 1 << 20);   // n = 0: stop logging and drop the series
  size_t logSamples() const { return log_t_.size(); }
  // one sample k of watched id j: [t | measured_pose 7 | pose_internal 6 | twist 6 | acceleration 6] = 26 doubles, then P (N*N)
  bool logSample(size_t k, size_t j, double* row26, double* P, int* n_state) const;
  // <folder>time_<id>, meas_pose_<id>, est_pose_<id> (x y z roll pitch yaw), est_twist_<id>, est_acc_<id>, cov_diag_<id>:
  // one row per sample, values separated by a blank, default ostream precision (what writeTxtFile writes).  Returns #files.
  int writeLog(const std::string& folder) const;

  // access for the proxies / solver
  struct Slot { int type; };
  bool typeOf(unsigned id, int& type);
  te_pool* poolOf(int type, bool create);
  unsigned heldTypes();   // bit t set = the pool of model type t holds targets
  // the rows of a batch by model type of their id (one registry lookup per id; call order kept; unknown ids in no list)
  void rowsByType(long long n, const unsigned* ids, std::vector<long long> rows[4]);
  int device() const { return device_; }
  std::recursive_mutex& lock() { return target_lock_; }

 protected:
  struct Pending {
    std::vector<uint32_t> ids;
    std::vector<double> dt, meas;
    std::vector<uint8_t> action;
  };
  void flushLocked();
  int registerClass(int type, const MatrixXd& Q, const MatrixXd& R, const MatrixXd& P0);
  void queue(int type, unsigned id, double dt, const double* meas, int action);
  // updateBatch's arguments: meas NULL with action NULL or with an UPDATE op throws std::invalid_argument
  static void requireMeasurements(long long n, const double* meas, const unsigned char* action);
  long long updateBatchUnique(long long n, const unsigned* ids, double dt, const double* meas, const unsigned char* action);   // no id twice
  te_pool* densePool();   // the one non-empty pool of a homogeneous manager (throws otherwise)
  // associate() over the pools of `shards` (each_shard as in PoolRowMerge::run); update(n, ids, det) applies the assigned records
  long long associateOver(const std::vector<TargetManager*>& shards, const std::function<void(const std::function<void(int)>&)>& each_shard,
                          double t1, long long q, const double* det, double gate, int K, int apply, unsigned* id_out, double* d2_out,
                          long long* count_out, const std::function<void(long long, const unsigned*, const double*)>& update);
  void updateAt(double t1, long long n, const unsigned* ids, const double* det);   // te_pool_update_at of every model type's rows
  friend class ShardedTargetManager;
  PoolRowMerge nearest_rows_;
  PoolRowMerge gated_rows_;
  PoolRowMerge assoc_rows_;

  int device_;
  te_pool* pools_[4] = {nullptr, nullptr, nullptr, nullptr};
  Pending pending_[4];
  std::unordered_map<unsigned, uint8_t> pending_ids_;
  IdRegistry targets_;   // id -> model type, ascending like the reference's std::map
  std::recursive_mutex target_lock_;
  MatrixXd default_Q_, default_P_, default_R_;
  target_t default_type_ = UNIFORM_VELOCITY;
  bool default_values_loaded_ = false;
  // sampled logging: watched ids, per-sample tick time, per-sample-per-id rows
  std::vector<unsigned> log_ids_;
  size_t log_cap_ = 0;
  std::vector<double> log_t_;                  // [samples] time of the first watched target that exists (else NaN)
  std::vector<double> log_rows_;               // [samples][ids][26]
  std::vector<double> log_P_;                  // [samples][ids][18*18] (n_state^2 used)
  std::vector<int> log_n_;                     // [samples][ids] state size, 0 = id unknown at that sample
};

// utils.hpp:78-120: one value (vector) or one row (matrix) per line, "value " per column, default ostream formatting
bool writeTxtFile(const std::string& filename, const double* values, size_t rows, size_t cols);

// utils.hpp:206-265 (host copy used by nothing on the hot path; kept for API completeness)
class MovingAvgFilter {
 public:
  typedef std::shared_ptr<MovingAvgFilter> Ptr;
  explicit MovingAvgFilter(unsigned n) : sum_(0.0), variance_(0.0), window_(n, 0.0), idx_(0), complete_(false) {}
  double update(double value);
  double getVariance() const { return variance_; }
 private:
  double sum_, variance_;
  std::vector<double> window_;
  unsigned idx_;
  bool complete_;
};

// intersection_solver.hpp:55-125.  One solver STREAM = one reference solver (one pair of moving-average filters + previous
// intersection pose shared by every id queried through it, SURVEY.md H9); every query through a stream updates it in call order.
// The reference's per-id methods use stream 0.  query() is the batched form: query k goes through stream[k] (NULL = k).
// A manager holding several model types keeps one state per stream and model type (the filters live beside the pool they are
// used with; a reference solver used across model types would share them).
// Any handle works: on a ShardedTargetManager (and so a ShardedTickTargetManager) the solver keeps one te_isolver per (shard, model
// type) and the shard home[stream] that holds each stream's current state.  A call routes its queries to the owners of their ids
// (in call order), moves the state of every stream whose home is another shard to the shard that now queries it
// (te_isolver_move_streams, bit-exact), then queries all shards at once.  So the results are those of the same solver on one
// plain manager, whichever shards the ids of a stream live on.  Memory: a shard allocates its stream arrays (n_streams x
// (2 filters_length + 9) doubles + 5 bytes per model type) on its first query, so each device then holds what a single-device
// solver of the same n_streams holds.
class ShardedTargetManager;
class IntersectionSolver {
 public:
  typedef std::shared_ptr<IntersectionSolver> Ptr;
  IntersectionSolver(TargetManager::Ptr target_manager, const unsigned int filters_length = 250, long long n_streams = 1);
  ~IntersectionSolver();
  double getIntersectionTimeWithSphere(const unsigned int& id, const double& t1, const Vector3d& origin, const double& radius);
  bool getIntersectionPoseWithSphere(const unsigned int& id, const double& t1, const double& pos_th, const double& ang_th,
                                     const Vector3d& origin, const double& radius, Vector7d& intersection_pose);
  // n queries at once: delta[k] as getIntersectionTimeWithSphere, pose7[k] / converged[k] as getIntersectionPoseWithSphere through
  // stream[k] (stream NULL = k, then n <= streams() for pose queries); pose7 NULL = times only (no stream is touched, pos_th / ang_th may be NULL);
  // delta / converged may be NULL.  A stream may appear more than once: the batch is then cut in front of each repeat and the
  // pieces run in order, so a batch always equals the same queries issued one by one.  An unknown id gives -1 / initPose / false
  // and leaves its stream untouched.  Returns the number of queries whose id exists.
  long long query(long long n, const unsigned* ids, const int* stream, const double* t1, const double* origin /*[n][3]*/,
                  const double* radius, const double* pos_th, const double* ang_th, double* delta, double* pose7,
                  unsigned char* converged);
  // The k earliest sphere intercepts over every target of the manager (te_pool_earliest_intersections on every (shard, model type)
  // pool that holds targets; the shards of a sharded manager run at once).  Sphere j = (t1[j], origin[j][3], radius[j]); delta of
  // target i is bit for bit query()'s time for (i, t1[j], origin[j], radius[j]), a hit is delta >= 0 (-0.0 ranks as 0).  hits_out[j] =
  // the number of hits; rows 0 .. min(k, hits) - 1 of ids_out[j][.] / delta_out[j][.] are those hits by (delta, id), the pools' sorted
  // lists merged on the host; the other rows are id 0xFFFFFFFF and delta -1.  The result does not depend on the shard count or on
  // which pool holds a target.  Read-only: no solver stream is created or touched; queued per-id calls are flushed first.
  // 0 <= k <= 65536 (k == 0: counts only, ids_out / delta_out may be NULL).  The intercept pose of a returned target is
  // getEstimatesBatch(ids, t1 + delta).  Returns the total number of hits.
  long long earliestIntersections(long long q, const double* t1, const double* origin /*[q][3]*/, const double* radius, long long k,
                                  unsigned* ids_out /*[q][k]*/, double* delta_out /*[q][k]*/, long long* hits_out /*[q]*/);
  long long streams() const { return n_streams_; }
  // host wall time of the last query() by phase, ms: [0] routing by owner (and model type), [1] moves of stream state between
  // shards, [2] the shards' te_isolver_query calls (uploads, kernels, read-backs; all shards at once), [3] results into call order
  const double* lastPhaseMs() const { return phase_ms_; }

 private:
  struct Part {   // the queries of one shard in one call (a routed copy of the caller's rows)
    std::vector<unsigned> ids;
    std::vector<long long> where;   // caller's row
    std::vector<int> stream;
    std::vector<double> t1, origin, radius, pos_th, ang_th, delta, pose;
    std::vector<unsigned char> conv;
    int only = -1;                       // model type of the shard's targets, -1 = no target, -2 = several types (see rows)
    std::vector<long long> rows[4];      // several types: the queries of each model type (unknown ids in none)
    std::vector<std::vector<int>> moves;   // [type * G + source shard]: streams whose state comes from that shard
    long long found = 0;
  };
  long long queryRun(long long n, const unsigned* ids, const int* stream, const double* t1, const double* origin, const double* radius,
                     const double* pos_th, const double* ang_th, double* delta, double* pose7, unsigned char* converged);   // no stream twice
  void classify(int r, long long m, const unsigned* ids);
  void collectMoves(int r, long long m, const int* stream);
  long long queryShard(int r, long long m, const unsigned* ids, const int* stream, const double* t1, const double* origin,
                       const double* radius, const double* pos_th, const double* ang_th, double* delta, double* pose7, unsigned char* conv);
  TargetManager& shardOf(int r);
  te_isolver* solverFor(int r, int type);
  TargetManager::Ptr target_manager_;
  ShardedTargetManager* sharded_ = nullptr;   // the manager as a sharded one, else NULL
  unsigned filters_length_;
  long long n_streams_;
  std::vector<std::array<te_isolver*, 4>> solvers_;   // [shard][model type], created on first use
  std::vector<int> home_;                             // sharded: [type * n_streams + stream] shard of the state, -1 = fresh everywhere
  std::vector<Part> part_;
  std::vector<unsigned> seen_;                        // repeat detection: seen_[stream] == gen_ within the current piece
  unsigned gen_ = 0;
  PoolRowMerge sweep_;                                // earliestIntersections
  double phase_ms_[4] = {0, 0, 0, 0};
};

// ---------------------------------------------------------------------------------------------------
// RosTargetManager without ROS (target_manager_ros.hpp:74-183, src/target_manager_ros.cpp:6-107): the /tf
// mailbox per id, the per-tick init-on-first-sight / update / predict loop, expiry erase and the list of
// filtered poses the node broadcasts.  ros::Time stamps are (sec, nsec) pairs; ros::Time::now() is passed in.
// The mailboxes are DEVICE resident (te_pool_mailbox_*): one /tf message = one ingest call (lookup, stable sort by slot,
// Measurement::update per slot), one tick = one rebuild + one step launch + one estimate gather; host work per tick is
// proportional to the ids that appear or expire, not to the number of targets.
// ---------------------------------------------------------------------------------------------------
struct StampedPose {
  uint32_t sec = 0, nsec = 0;
  Vector7d pose{};   // geometry_msgs default-constructs to zeros
};
double toSec(uint32_t sec, uint32_t nsec);   // utils.hpp:59-62 (never contracted to an FMA)

class Measurement {   // target_manager_ros.hpp:74-134
 public:
  Measurement() : last_meas_time_(0.0), new_meas_(true) {}
  bool read(StampedPose& tr) const {
    if (new_meas_) { tr = tr_; return true; }   // new_meas_ is NOT cleared by read() (SURVEY.md H10)
    return false;
  }
  void update(const StampedPose& tr);
  double getTime() const { return last_meas_time_; }
  // the accepted stamp behind last_meas_time_, and whether the device copy of it is stale
  uint32_t acceptedSec() const { return acc_sec_; }
  uint32_t acceptedNsec() const { return acc_nsec_; }
  bool stampDirty() const { return stamp_dirty_; }
  void clearStampDirty() { stamp_dirty_ = false; }
 private:
  double last_meas_time_;
  bool new_meas_;
  StampedPose tr_;
  uint32_t acc_sec_ = 0, acc_nsec_ = 0;
  bool stamp_dirty_ = false;
};

// The node loop of RosTargetManager (target_manager_ros.hpp:136-183): what replayBag and the C-ABI's target_tick_manager_* calls
// drive, on one device (TickTargetManager) or on every GPU of the box (ShardedTickTargetManager).
class TickFrontEnd {
 public:
  virtual ~TickFrontEnd() {}
  // /tf callback (src/target_manager_ros.cpp:26-39): frame "<token>_<id>"; a frame that contains the token but does
  // not parse BREAKS the loop (the rest of the message is dropped), like the reference
  virtual void measurementCallBack(long long n, const char* const* child_frame_ids, const uint32_t* sec, const uint32_t* nsec,
                                   const double* poses) = 0;
  virtual void measurementCallBackIds(long long n, const unsigned* ids, const uint32_t* sec, const uint32_t* nsec, const double* poses) = 0;
  // RosTargetManager::update(dt) (:41-92) with ros::Time::now() = (now_sec, now_nsec).  erased (optional) receives
  // the ids removed by the expiry rule in ascending order.
  virtual void tick(const double& dt, uint32_t now_sec, uint32_t now_nsec, std::vector<unsigned>* erased = nullptr) = 0;
  // the poses the node would broadcast after the last tick: ids + [n][7]
  virtual const std::vector<unsigned>& publishedIds() const = 0;
  virtual const std::vector<double>& publishedPoses() const = 0;
  virtual void setTargetTokenName(const std::string& token_name) = 0;
  virtual void setExpirationTime(double t) = 0;
  virtual double time() const = 0;
  virtual size_t mailboxCount() = 0;   // measurements_.size() of the reference
  bool publish = true;   // gather the filtered poses every tick (the TF broadcast of :78-87)
 protected:
  // the frames of one message -> (id, stamp, pose) records, the reference's loop (:26-39): frames without the token are skipped,
  // the first frame that carries it but does not parse ends the message
  static void parseFrames(const std::string& token, long long n, const char* const* frames, const uint32_t* sec, const uint32_t* nsec,
                          const double* poses, std::vector<unsigned>& ids, std::vector<uint32_t>& s, std::vector<uint32_t>& ns,
                          std::vector<double>& p);
};

class TickTargetManager : public TargetManager, public TickFrontEnd {
 public:
  TickTargetManager(target_t type, const MatrixXd& Q, const MatrixXd& R, const MatrixXd& P, int device = 0);
  explicit TickTargetManager(const std::string& yaml_file, int device = 0);
  ~TickTargetManager() override;
  void measurementCallBack(long long n, const char* const* child_frame_ids, const uint32_t* sec, const uint32_t* nsec,
                           const double* poses) override;
  void measurementCallBackIds(long long n, const unsigned* ids, const uint32_t* sec, const uint32_t* nsec, const double* poses) override;
  void tick(const double& dt, uint32_t now_sec, uint32_t now_nsec, std::vector<unsigned>* erased = nullptr) override;
  // ascending ids + [n][7]
  const std::vector<unsigned>& publishedIds() const override { return pub_ids_; }
  const std::vector<double>& publishedPoses() const override { return pub_poses_; }
  void setTargetTokenName(const std::string& token_name) override { token_name_ = token_name; }
  void setExpirationTime(double t) override;
  double time() const override { return t_; }
  size_t mailboxCount() override;   // device mailboxes + target-less ones + host ones
 private:
  friend class ShardedTickTargetManager;
  // the pieces of the sharded node loop, each under the manager's lock
  te_pool* devicePool();   // flushes the queued by-hand calls; the tick's pool, or NULL while some id needs a host mailbox
  void ingestDev(long long n, const uint32_t* dev_ids, const uint32_t* dev_sec, const uint32_t* dev_nsec, const double* dev_poses);
  void advance(const double& dt, uint32_t now_sec, uint32_t now_nsec, std::vector<unsigned>* erased);   // tick() without the broadcast
  long long publishCount();                                  // poses the broadcast covers (every target)
  void publishInto(unsigned* ids, double* poses, long long n);   // their ascending ids and [n][7] poses
  bool foreignPossible(te_pool* pool);
  te_pool* tickPool();
  void tickForeign(const double& dt, uint32_t now_sec, uint32_t now_nsec, std::vector<unsigned>& gone_out);
  int cls_ = -1;   // model class of (Q_, R_, P_) in the pool of type_
  target_t type_;
  MatrixXd Q_, P_, R_;
  std::string token_name_;
  double t_;
  std::map<unsigned, Measurement> measurements_;   // host mailboxes: only ids that live in a pool of another model type
  double expiration_time_;
  std::vector<unsigned> pub_ids_;
  std::vector<double> pub_poses_;
  std::vector<uint32_t> gone_buf_, born_buf_;   // reusable output buffers of te_pool_mailbox_tick
  void* pub_pinned_ = nullptr;                  // storage of pub_poses_ while it is page-locked
};

// ---------------------------------------------------------------------------------------------------
// One TargetManager per GPU of the box behind the TargetManager interface (BASELINE.json north_star: "targets shard by ID across
// the 8 GPUs of one box with no collective on the hot path ... the TargetManager API stays as the host surface in C++").
// owner(id) = id mod G; shard r is an ordinary TargetManager on device devices[r] with its own pools and streams.  Per-id calls
// go to the owner (their launches coalesce per shard as in TargetManager).  The batched calls route their records to the owners
// with one parallel stable partition on the host (routeOnHost: every shard's records in the caller's order), then every shard's
// worker thread runs the shard's batched call -- so the G devices copy and step concurrently.  Results are the
// reference's: an id lives in exactly one shard, its records are applied in call order.
// The optional exchange of estimates (SURVEY.md 8(e)) is gatherEstimates(): [pose7 | twist6] records of every target, all shards,
// gathered on every device over NCCL (te_group_*), then read back from the publishing shard's device.
// ---------------------------------------------------------------------------------------------------
// id mod G without a division per record (the routing passes look at every id of a batch; a hardware divide per id cost more than
// the tick it feeds): a mask for powers of two, else Lemire's multiply-shift remainder, exact for 32-bit operands
struct FastMod {
  explicit FastMod(unsigned d) : d_(d), pow2_((d & (d - 1)) == 0), m_(~(unsigned long long)0 / d + 1) {}
  unsigned operator()(unsigned a) const {
    if (pow2_) return a & (d_ - 1);
    const unsigned long long low = m_ * a;
    return (unsigned)(((unsigned __int128)low * d_) >> 64);
  }
  unsigned d_;
  bool pow2_;
  unsigned long long m_;
};

class ShardWorkers;
class ShardedTargetManager : public TargetManager {
 public:
  // devices NULL = devices 0 .. n_shards-1; a device may repeat (several shards on one GPU: a one-GPU box still runs the
  // sharded host logic -- the estimate exchange then uses device copies, NCCL needs distinct devices)
  ShardedTargetManager(const std::string& file, int n_shards, const int* devices = nullptr);
 protected:
  // the same with shards made by make_shard(device) (a derived manager's shards are derived managers)
  ShardedTargetManager(const std::string& file, int n_shards, const int* devices, const std::function<TargetManager*(int)>& make_shard);
 public:
  ~ShardedTargetManager() override;
  int shards() const { return (int)shard_.size(); }
  int owner(unsigned id) const { return (int)(id % (unsigned)shard_.size()); }
  TargetManager& shard(int r) { return *shard_[(size_t)r]; }

  void init(const unsigned int& id, const double& dt0, const double& t0, const Vector7d& p0, const Vector6d& v0 = Vector6d{},
            const Vector6d& a0 = Vector6d{}) override;
  void init(const target_t& type, const unsigned int& id, const double& dt0, const double& t0, const MatrixXd& Q, const MatrixXd& R,
            const MatrixXd& P0, const Vector7d& p0, const Vector6d& v0 = Vector6d{}, const Vector6d& a0 = Vector6d{}) override;
  bool update(const unsigned int& id, const double& dt, const Vector7d& meas) override;
  bool update(const unsigned int& id, const double& dt) override;
  void update(const double& dt) override;
  bool erase(const unsigned int& id) override;
  TargetInterface::Ptr getTarget(const unsigned int& id) override;
  bool getTargetPose(const unsigned int& id, Vector7d& pose) override;
  bool getTargetTwist(const unsigned int& id, Vector6d& twist) override;
  bool getTargetAcceleration(const unsigned int& id, Vector6d& acc) override;
  long long getNumberMeasurements(const unsigned int& id) override;
  void log() override;
  std::vector<unsigned int> getAvailableTargets() override;   // ascending ids over all shards
  long long initBatch(target_t type, const MatrixXd& Q, const MatrixXd& R, const MatrixXd& P0, long long n, const unsigned* ids, double dt0,
                      const double* t0, const double* p0, const double* v0 = nullptr, const double* a0 = nullptr,
                      const double* p0_scale = nullptr) override;
  using TargetManager::initBatch;
  long long updateBatch(long long n, const unsigned* ids, double dt, const double* meas, const unsigned char* action = nullptr) override;
  long long eraseBatch(long long n, const unsigned* ids) override;
  void getEstimatesBatch(long long n, const unsigned* ids, const double* t1, double* pose7, double* twist6, double* acc6,
                         unsigned char* found) override;
  void flush() override;
  long long nearestTargets(long long q, const double* t1, const double* point, const double* radius, long long k, unsigned* ids_out,
                           double* dist_out, long long* count_out) override;   // every shard at once
  long long gatedTargets(long long q, const double* t1, const double* z, const double* gate, long long k, unsigned* ids_out,
                         double* d2_out, long long* count_out) override;   // every shard at once
  long long associate(double t1, long long q, const double* det, double gate, int K, int apply, unsigned* id_out, double* d2_out,
                      long long* count_out) override;   // candidates of every shard at once, updates routed by owner
  // dense ticks: the records are SHARD-MAJOR (denseIds(): shard 0's targets in ascending id, then shard 1's, ...); every shard's
  // slice is copied, stepped and read back by its own worker thread on its own device
  long long updateDense(double dt, const double* meas, int meas_stride, const unsigned char* action, double* est_pos_out) override;
  long long updateDenseAsync(double dt, const double* meas, int meas_stride, const unsigned char* action, double* est_pos_out) override;
  void updateDenseWait(int lag) override;
  std::vector<unsigned int> denseIds() override;
  void watch(long long n, const unsigned* ids, size_t max_samples = 1 << 20) override;   // forwarded to the owners

  // The optional all-gather of estimates: ids (shard-major: shard 0's targets of model type 0 in ascending id, ...) and their
  // [pose7 | twist6] records, exchanged between the devices over NCCL and read back from shard `publisher`'s device.  Either output
  // may be NULL (exchange only).  Returns the number of records; lastGatherMs() = device time of the exchange(s).
  long long gatherEstimates(std::vector<unsigned>* ids, std::vector<double>* records13, int publisher = 0);
  double lastGatherMs() const { return gather_ms_; }
  bool gatherUsesNccl();

 protected:
  void forEachShard(const std::function<void(int)>& f);   // f(r) on shard r's worker thread, all shards at once; rethrows the first error
  // The routing of a batch on the host (a parallel stable partition by owner, see updateBatch): reserve(r, m) sizes shard r's
  // staging for its m records (on r's worker thread); scatter(t, lo, hi, at) runs on router thread t for the records [lo, hi) of
  // the batch and puts record k of owner r at place at[r]++ of r's staging.  Returns the records of every shard.
  std::vector<size_t> routeOnHost(long long n, const unsigned* ids, const std::function<void(int, size_t)>& reserve,
                                  const std::function<void(int, long long, long long, size_t*)>& scatter);
  std::vector<std::vector<long long>> rowsByOwner(long long n, const unsigned* ids);   // routeOnHost: every shard's rows of the batch
  te_group* group();   // created on first use
  friend class IntersectionSolver;   // routes its queries with routeOnHost and runs them with forEachShard
  std::vector<std::unique_ptr<TargetManager>> shard_;
  std::vector<int> devices_;
  std::unique_ptr<ShardWorkers> workers_;   // one thread per shard: the shards' batched calls
  std::unique_ptr<ShardWorkers> routers_;   // the routing passes of a batch: as many threads as the host offers (at most 16)
  te_group* group_ = nullptr;
  double gather_ms_ = -1.0;
  struct Stage {   // per shard, page-locked, grow-only
    std::vector<unsigned> ids;
    double* meas = nullptr;
    unsigned char* action = nullptr;
    size_t cap = 0;
  };
  std::vector<Stage> stage_;
};

// ---------------------------------------------------------------------------------------------------
// The node loop over every GPU of the box: one TickTargetManager per shard (owner(id) = id mod G, shard r on devices[r]).  A /tf
// message is parsed on the host as a whole, then routed ON THE DEVICES (te_group_route_records: G chunk uploads in parallel, a
// stable partition by owner on every device, NCCL send / receive between them) and every shard's worker ingests its run in place
// (te_pool_mailbox_ingest_dev): host work per message is O(G) copies, not a pass over the records.  Arrival order per id is kept, so
// Measurement::update sees the records of an id in the order the single-device loop sees them.  While some shard keeps host
// mailboxes (an id lives there under another model type, created by hand) the message takes the host route instead: the router
// threads of the batched calls, then that shard's measurementCallBackIds.  TE_SHARD_HOST_ROUTE in the environment of the process
// (read when the manager is made) forces the host route -- a debugging switch.
// A tick runs every shard's tick on its worker thread at once; the erased ids of all shards come back as one ascending list, and
// the broadcast is shard-major (shard 0's targets in ascending id, then shard 1's, ...: denseIds() order), every shard writing its
// slice straight into one page-locked output.  By-hand calls, batched calls and gatherEstimates work as in ShardedTargetManager.
// ---------------------------------------------------------------------------------------------------
class ShardedTickTargetManager : public ShardedTargetManager, public TickFrontEnd {
 public:
  ShardedTickTargetManager(const std::string& yaml_file, int n_shards, const int* devices = nullptr);
  ~ShardedTickTargetManager() override;
  TickTargetManager& tickShard(int r) { return static_cast<TickTargetManager&>(*shard_[(size_t)r]); }
  void measurementCallBack(long long n, const char* const* child_frame_ids, const uint32_t* sec, const uint32_t* nsec,
                           const double* poses) override;
  void measurementCallBackIds(long long n, const unsigned* ids, const uint32_t* sec, const uint32_t* nsec, const double* poses) override;
  void tick(const double& dt, uint32_t now_sec, uint32_t now_nsec, std::vector<unsigned>* erased = nullptr) override;
  // shard-major ids + [n][7]
  const std::vector<unsigned>& publishedIds() const override { return pub_ids_; }
  const std::vector<double>& publishedPoses() const override { return pub_poses_; }
  void setTargetTokenName(const std::string& token_name) override { token_name_ = token_name; }
  void setExpirationTime(double t) override;
  double time() const override;
  size_t mailboxCount() override;   // sum over the shards

 private:
  std::string token_name_ = "target";
  bool force_host_route_ = false;
  std::vector<unsigned> pub_ids_;
  std::vector<double> pub_poses_;
  void* pub_pinned_[2] = {nullptr, nullptr};   // storage of pub_ids_ / pub_poses_ while it is page-locked
  struct HostStage {   // per shard: its records of a message on the host route
    std::vector<unsigned> ids;
    std::vector<uint32_t> sec, nsec;
    std::vector<double> poses;
  };
  std::vector<HostStage> host_stage_;
};

// utils.hpp:273-313
std::vector<std::string> splitString(const std::string& s, const std::string& delimiter = "_");
bool getId(const std::string& s, unsigned int& id);

}  // namespace target_estimation_b200
