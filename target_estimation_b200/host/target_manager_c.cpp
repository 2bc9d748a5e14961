// target_manager_c.cpp -- extern "C" wrapper of the host TargetManager: the ten symbols of the reference's
// C-ABI (/root/reference/src/target_manager_c.cpp:15-76) plus the batched extensions of
// include/target_manager_c.h.  No exception crosses the boundary.
#include "target_manager_c.h"

#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "target_estimation_b200/bag_reader.hpp"
#include "target_estimation_b200/target_manager.hpp"

using namespace target_estimation_b200;

namespace {
// the reference keeps file-static scratch vectors and copies them out even when the id is unknown
// (src/target_manager_c.cpp:8-9,39-42): an unknown id returns false and the previous value
Vector7d vector7d_tmp_{};
Vector6d vector6d_tmp_{};
thread_local std::string g_err;

template <class F, class R> R guard(R fallback, F&& f) {
  try {
    return f();
  } catch (const char* msg) {
    g_err = msg;
  } catch (const std::exception& e) {
    g_err = e.what();
  } catch (...) {
    g_err = "unknown error";
  }
  return fallback;
}
inline TargetManager* M(const target_manager_c* self) { return (TargetManager*)self; }
inline IntersectionSolver* S(const target_isolver_c* s) {
  if (!s) throw std::invalid_argument("null solver");
  return (IntersectionSolver*)s;
}
}  // namespace

extern "C" {

target_manager_c* target_manager_new_on_device(const char* file, int device) {
  return guard((target_manager_c*)nullptr, [&]() -> target_manager_c* {
    TargetManager* m = (file && file[0]) ? new TargetManager(std::string(file), device) : new TargetManager(device);
    return (target_manager_c*)m;
  });
}
target_manager_c* target_manager_new(const char* file) { return target_manager_new_on_device(file, 0); }

void target_manager_init(const target_manager_c* self, const unsigned int id, const double dt0, double p0[], const double t0) {
  guard(0, [&] {
    Vector7d p;
    std::memcpy(p.data(), p0, sizeof(double) * 7);
    M(self)->init(id, dt0, t0, p);
    return 0;
  });
}

void target_manager_update_meas(const target_manager_c* self, const unsigned int id, const double dt, double meas[]) {
  guard(0, [&] {
    Vector7d m;
    std::memcpy(m.data(), meas, sizeof(double) * 7);
    M(self)->update(id, dt, m);
    return 0;
  });
}

void target_manager_update(const target_manager_c* self, const unsigned int id, const double dt) {
  guard(0, [&] {
    M(self)->update(id, dt);
    return 0;
  });
}

bool target_manager_get_est_pose(const target_manager_c* self, const unsigned int id, double pose[]) {
  bool res = guard(false, [&] { return M(self)->getTargetPose(id, vector7d_tmp_); });
  std::memcpy(pose, vector7d_tmp_.data(), sizeof(double) * 7);
  return res;
}
bool target_manager_get_est_twist(const target_manager_c* self, const unsigned int id, double twist[]) {
  bool res = guard(false, [&] { return M(self)->getTargetTwist(id, vector6d_tmp_); });
  std::memcpy(twist, vector6d_tmp_.data(), sizeof(double) * 6);
  return res;
}
bool target_manager_get_est_acceleration(const target_manager_c* self, const unsigned int id, double acceleration[]) {
  bool res = guard(false, [&] { return M(self)->getTargetAcceleration(id, vector6d_tmp_); });
  std::memcpy(acceleration, vector6d_tmp_.data(), sizeof(double) * 6);
  return res;
}
int target_manager_get_n_measurements(const target_manager_c* self, const unsigned int id) {
  return guard(0, [&] { return (int)M(self)->getNumberMeasurements(id); });   // long long -> int like the reference (:64)
}
void target_manager_watch(const target_manager_c* self, long long n, const unsigned int* ids, long long max_samples) {
  guard(0, [&] { M(self)->watch(n, ids, max_samples > 0 ? (size_t)max_samples : (size_t)1 << 20); return 0; });
}
long long target_manager_log_samples(const target_manager_c* self) {
  return guard(-1LL, [&] { return (long long)M(self)->logSamples(); });
}
int target_manager_log_sample(const target_manager_c* self, long long k, long long j, double* row26, double* P) {
  return guard(-1, [&] {
    int n = 0;
    if (k < 0 || j < 0) return -1;
    const bool ok = M(self)->logSample((size_t)k, (size_t)j, row26, P, &n);
    return (ok || (size_t)k < M(self)->logSamples()) ? n : -1;
  });
}
int target_manager_write_log(const target_manager_c* self, const char* folder) {
  return guard(-1, [&] { return M(self)->writeLog(folder ? std::string(folder) : std::string("/tmp/")); });
}
int target_write_txt_file(const char* filename, const double* values, long long rows, long long cols) {
  return guard(-1, [&] { return target_estimation_b200::writeTxtFile(std::string(filename), values, (size_t)rows, (size_t)cols) ? 1 : 0; });
}
void target_manager_log(const target_manager_c* self) {
  guard(0, [&] { M(self)->log(); return 0; });
}
void target_manager_delete(target_manager_c* self) { delete M(self); }

// ---- batched extensions ------------------------------------------------------------------------
long long target_manager_init_batch(const target_manager_c* self, long long n, const unsigned int* ids, double dt0, const double* p0,
                                    const double* t0) {
  return guard(-1LL, [&] { return M(self)->initBatch(n, ids, dt0, t0, p0); });
}
long long target_manager_update_batch(const target_manager_c* self, long long n, const unsigned int* ids, double dt, const double* meas,
                                      const unsigned char* action) {
  return guard(-1LL, [&] { return M(self)->updateBatch(n, ids, dt, meas, action); });
}
long long target_manager_update_dense(const target_manager_c* self, double dt, const double* meas, int meas_stride, const unsigned char* action,
                                      double* est_pos_out) {
  return guard(-1LL, [&] { return M(self)->updateDense(dt, meas, meas_stride, action, est_pos_out); });
}
long long target_manager_update_dense_async(const target_manager_c* self, double dt, const double* meas, int meas_stride,
                                            const unsigned char* action, double* est_pos_out) {
  return guard(-1LL, [&] { return M(self)->updateDenseAsync(dt, meas, meas_stride, action, est_pos_out); });
}
int target_manager_update_dense_wait(const target_manager_c* self, int lag) {
  return guard(-1, [&] { M(self)->updateDenseWait(lag); return 0; });
}
long long target_manager_get_dense_ids(const target_manager_c* self, unsigned int* out, long long cap) {
  return guard(-1LL, [&] {
    auto ids = M(self)->denseIds();
    const long long n = (long long)ids.size();
    if (out && cap > 0) std::memcpy(out, ids.data(), sizeof(unsigned) * (size_t)(n < cap ? n : cap));
    return n;
  });
}
void target_manager_update_all(const target_manager_c* self, double dt) {
  guard(0, [&] { M(self)->update(dt); return 0; });
}
long long target_manager_erase_batch(const target_manager_c* self, long long n, const unsigned int* ids) {
  return guard(-1LL, [&] { return M(self)->eraseBatch(n, ids); });
}
bool target_manager_erase(const target_manager_c* self, unsigned int id) {
  return guard(false, [&] { return M(self)->erase(id); });
}
int target_manager_get_estimates_batch(const target_manager_c* self, long long n, const unsigned int* ids, const double* t1, double* pose7,
                                       double* twist6, double* acc6, unsigned char* found) {
  return guard(-1, [&] { M(self)->getEstimatesBatch(n, ids, t1, pose7, twist6, acc6, found); return 0; });
}
long long target_manager_get_ids(const target_manager_c* self, unsigned int* out, long long cap) {
  return guard(-1LL, [&] {
    auto ids = M(self)->getAvailableTargets();
    const long long n = (long long)ids.size();
    if (out && cap > 0) std::memcpy(out, ids.data(), sizeof(unsigned) * (size_t)(n < cap ? n : cap));
    return n;
  });
}
int target_manager_get_state(const target_manager_c* self, unsigned int id, double* x, double* P, double* t) {
  return guard(0, [&] {
    auto tg = M(self)->getTarget(id);
    if (!tg) return 0;
    VectorXd xs = tg->getEstimator()->getState();
    if (x) std::memcpy(x, xs.data(), sizeof(double) * xs.size());
    if (P) {
      MatrixXd Pm = tg->getEstimator()->getP();
      std::memcpy(P, Pm.data(), sizeof(double) * Pm.d.size());
    }
    if (t) *t = tg->getTime();
    return (int)xs.size();
  });
}
void target_manager_flush(const target_manager_c* self) {
  guard(0, [&] { M(self)->flush(); return 0; });
}
long long target_manager_nearest(const target_manager_c* self, long long q, const double* t1, const double* point, const double* radius, long long k,
                                 unsigned int* ids_out, double* dist_out, long long* count_out) {
  return guard(-1LL, [&] {
    if (!self) throw std::invalid_argument("null manager");
    return M(self)->nearestTargets(q, t1, point, radius, k, ids_out, dist_out, count_out);
  });
}
long long target_manager_gated(const target_manager_c* self, long long q, const double* t1, const double* z, const double* gate, long long k,
                               unsigned int* ids_out, double* d2_out, long long* count_out) {
  return guard(-1LL, [&] {
    if (!self) throw std::invalid_argument("null manager");
    return M(self)->gatedTargets(q, t1, z, gate, k, ids_out, d2_out, count_out);
  });
}
long long target_manager_associate(const target_manager_c* self, double t1, long long q, const double* det, double gate, int K, int apply,
                                   unsigned int* id_out, double* d2_out, long long* count_out) {
  return guard(-1LL, [&] {
    if (!self) throw std::invalid_argument("null manager");
    return M(self)->associate(t1, q, det, gate, K, apply, id_out, d2_out, count_out);
  });
}
const char* target_manager_last_error(void) { return g_err.c_str(); }

// ---- IntersectionSolver -------------------------------------------------------------------------------------------
target_isolver_c* target_isolver_new(const target_manager_c* m, long long n_streams, unsigned filters_length) {
  return guard((target_isolver_c*)nullptr, [&]() -> target_isolver_c* {
    if (!m) throw std::invalid_argument("null manager");
    if (n_streams <= 0) throw std::invalid_argument("n_streams must be > 0");
    if (filters_length == 0) throw std::invalid_argument("filters_length must be > 0");
    TargetManager::Ptr mp(M(m), [](TargetManager*) {});   // the caller owns the manager
    return (target_isolver_c*)new IntersectionSolver(mp, filters_length, n_streams);
  });
}
void target_isolver_delete(target_isolver_c* s) { delete (IntersectionSolver*)s; }
double target_isolver_get_time(const target_isolver_c* s, unsigned id, double t1, const double origin[3], double radius) {
  return guard(-1.0, [&] {
    if (!origin) throw std::invalid_argument("origin is required");
    return S(s)->getIntersectionTimeWithSphere(id, t1, Vector3d{origin[0], origin[1], origin[2]}, radius);
  });
}
bool target_isolver_get_pose(const target_isolver_c* s, unsigned id, double t1, double pos_th, double ang_th, const double origin[3],
                             double radius, double pose[7]) {
  return guard(false, [&] {
    if (!origin || !pose) throw std::invalid_argument("origin and pose are required");
    Vector7d p;
    const bool ok = S(s)->getIntersectionPoseWithSphere(id, t1, pos_th, ang_th, Vector3d{origin[0], origin[1], origin[2]}, radius, p);
    std::memcpy(pose, p.data(), sizeof(double) * 7);
    return ok;
  });
}
long long target_isolver_query_batch(const target_isolver_c* s, long long n, const unsigned int* ids, const int* stream, const double* t1,
                                     const double* origin, const double* radius, const double* pos_th, const double* ang_th,
                                     double* delta_out, double* pose7_out, unsigned char* converged_out) {
  return guard(-1LL, [&] { return S(s)->query(n, ids, stream, t1, origin, radius, pos_th, ang_th, delta_out, pose7_out, converged_out); });
}
long long target_isolver_earliest(const target_isolver_c* s, long long q, const double* t1, const double* origin, const double* radius, long long k,
                                  unsigned int* ids_out, double* delta_out, long long* hits_out) {
  return guard(-1LL, [&] { return S(s)->earliestIntersections(q, t1, origin, radius, k, ids_out, delta_out, hits_out); });
}
int target_isolver_last_timing(const target_isolver_c* s, double ms_out[4]) {
  return guard(-1, [&] {
    if (!ms_out) throw std::invalid_argument("ms_out is required");
    std::memcpy(ms_out, S(s)->lastPhaseMs(), sizeof(double) * 4);
    return 0;
  });
}

// ---- all GPUs of the box behind one handle --------------------------------------------------------------
target_manager_c* target_manager_new_sharded(const char* file, int n_shards, const int* devices) {
  return guard((target_manager_c*)nullptr, [&]() -> target_manager_c* {
    if (!file || !file[0]) throw std::invalid_argument("a model file is required");
    TargetManager* m = new ShardedTargetManager(std::string(file), n_shards, devices);
    return (target_manager_c*)m;
  });
}
int target_manager_shards(const target_manager_c* self) {
  return guard(-1, [&] {
    ShardedTargetManager* s = dynamic_cast<ShardedTargetManager*>(M(self));
    return s ? s->shards() : 1;
  });
}
long long target_manager_gather_estimates(const target_manager_c* self, unsigned int* ids_out, double* records_out, long long cap, int publisher) {
  return guard(-1LL, [&]() -> long long {
    ShardedTargetManager* s = dynamic_cast<ShardedTargetManager*>(M(self));
    std::vector<unsigned> ids;
    std::vector<double> rec;
    long long n = 0;
    if (s) {
      const bool want = cap > 0 && (ids_out || records_out);
      n = s->gatherEstimates(want && ids_out ? &ids : nullptr, want && records_out ? &rec : nullptr, publisher);
    } else {   // a plain manager: its own targets, ascending ids
      ids = M(self)->getAvailableTargets();
      n = (long long)ids.size();
      if (cap > 0 && records_out) {
        rec.resize((size_t)n * 13);
        std::vector<double> po((size_t)n * 7), tw((size_t)n * 6);
        M(self)->getEstimatesBatch(n, ids.data(), nullptr, po.data(), tw.data(), nullptr, nullptr);
        for (long long k = 0; k < n; ++k) {
          std::memcpy(&rec[13 * (size_t)k], &po[7 * (size_t)k], 56);
          std::memcpy(&rec[13 * (size_t)k + 7], &tw[6 * (size_t)k], 48);
        }
      }
    }
    const long long k = n < cap ? n : cap;
    if (ids_out && k > 0 && !ids.empty()) std::memcpy(ids_out, ids.data(), sizeof(unsigned) * (size_t)k);
    if (records_out && k > 0 && !rec.empty()) std::memcpy(records_out, rec.data(), sizeof(double) * 13 * (size_t)k);
    return n;
  });
}
double target_manager_last_gather_ms(const target_manager_c* self) {
  return guard(-1.0, [&] {
    ShardedTargetManager* s = dynamic_cast<ShardedTargetManager*>(M(self));
    return s ? s->lastGatherMs() : -1.0;
  });
}
int target_manager_gather_uses_nccl(const target_manager_c* self) {
  return guard(-1, [&] {
    ShardedTargetManager* s = dynamic_cast<ShardedTargetManager*>(M(self));
    return (s && s->gatherUsesNccl()) ? 1 : 0;
  });
}

// ---- tick front-end ---------------------------------------------------------------------------------
static TickFrontEnd* T(const target_manager_c* self) {
  TickFrontEnd* t = dynamic_cast<TickFrontEnd*>(M(self));
  if (!t) throw std::invalid_argument("handle is not a tick manager");
  return t;
}
target_manager_c* target_tick_manager_new(const char* file, int device) {
  return guard((target_manager_c*)nullptr, [&]() -> target_manager_c* {
    if (!file || !file[0]) throw std::invalid_argument("a model file is required");
    TargetManager* m = new TickTargetManager(std::string(file), device);
    m->quiet = true;
    return (target_manager_c*)m;
  });
}
target_manager_c* target_tick_manager_new_sharded(const char* file, int n_shards, const int* devices) {
  return guard((target_manager_c*)nullptr, [&]() -> target_manager_c* {
    if (!file || !file[0]) throw std::invalid_argument("a model file is required");
    TargetManager* m = new ShardedTickTargetManager(std::string(file), n_shards, devices);
    return (target_manager_c*)m;
  });
}
void target_tick_manager_set_expiration(const target_manager_c* self, double timeout_s) {
  guard(0, [&] { T(self)->setExpirationTime(timeout_s); return 0; });
}
void target_tick_manager_set_publish(const target_manager_c* self, int on) {
  guard(0, [&] { T(self)->publish = on != 0; return 0; });
}
void target_tick_manager_set_token(const target_manager_c* self, const char* token) {
  guard(0, [&] { T(self)->setTargetTokenName(token ? token : ""); return 0; });
}
void target_tick_manager_callback_frames(const target_manager_c* self, long long n, const char* const* frames, const unsigned int* sec,
                                         const unsigned int* nsec, const double* poses) {
  guard(0, [&] { T(self)->measurementCallBack(n, frames, sec, nsec, poses); return 0; });
}
void target_tick_manager_callback_ids(const target_manager_c* self, long long n, const unsigned int* ids, const unsigned int* sec,
                                      const unsigned int* nsec, const double* poses) {
  guard(0, [&] { T(self)->measurementCallBackIds(n, ids, sec, nsec, poses); return 0; });
}
long long target_tick_manager_update(const target_manager_c* self, double dt, unsigned int now_sec, unsigned int now_nsec,
                                     unsigned int* erased_out, long long cap) {
  return guard(-1LL, [&]() -> long long {
    std::vector<unsigned> er;
    T(self)->tick(dt, now_sec, now_nsec, &er);
    const long long n = (long long)er.size();
    if (erased_out && cap > 0) std::memcpy(erased_out, er.data(), sizeof(unsigned) * (size_t)(n < cap ? n : cap));
    return n;
  });
}
long long target_tick_manager_published(const target_manager_c* self, unsigned int* ids_out, double* poses_out, long long cap) {
  return guard(-1LL, [&]() -> long long {
    const auto& ids = T(self)->publishedIds();
    const auto& po = T(self)->publishedPoses();
    const long long n = (long long)ids.size();
    const long long k = n < cap ? n : cap;
    if (ids_out && k > 0) std::memcpy(ids_out, ids.data(), sizeof(unsigned) * (size_t)k);
    if (poses_out && k > 0) std::memcpy(poses_out, po.data(), sizeof(double) * 7 * (size_t)k);
    return n;
  });
}
double target_tick_manager_time(const target_manager_c* self) {
  return guard(-1.0, [&] { return T(self)->time(); });
}
long long target_bag_read_tf(const char* path, const char* topic, target_tf_record* out, long long cap) {
  return guard(-1LL, [&]() -> long long {
    if (!path) throw std::invalid_argument("path is NULL");
    const std::vector<TfRecord> rec = readBagTf(path, topic ? topic : "/tf");
    const long long n = (long long)rec.size();
    for (long long i = 0; i < n && i < cap && out; ++i) {
      target_tf_record& o = out[i];
      const TfRecord& r = rec[(size_t)i];
      o.rec_sec = r.rec_sec; o.rec_nsec = r.rec_nsec; o.msg = r.msg; o.seq = r.seq; o.sec = r.sec; o.nsec = r.nsec;
      std::memset(o.frame_id, 0, sizeof(o.frame_id));
      std::memset(o.child_frame_id, 0, sizeof(o.child_frame_id));
      std::strncpy(o.frame_id, r.frame_id.c_str(), sizeof(o.frame_id) - 1);
      std::strncpy(o.child_frame_id, r.child_frame_id.c_str(), sizeof(o.child_frame_id) - 1);
      std::memcpy(o.pose, r.pose, sizeof(o.pose));
    }
    return n;
  });
}
long long target_tick_manager_replay_bag(const target_manager_c* self, const char* path, const char* topic, double frequency,
                                         long long extra_ticks, long long stats_out[4]) {
  return guard(-1LL, [&]() -> long long {
    if (!path) throw std::invalid_argument("path is NULL");
    const std::vector<TfRecord> rec = readBagTf(path, topic ? topic : "/tf");
    const ReplayStats st = replayBag(*T(self), rec, frequency, extra_ticks);
    if (stats_out) { stats_out[0] = st.ticks; stats_out[1] = st.messages; stats_out[2] = st.transforms; stats_out[3] = st.erased; }
    return st.ticks;
  });
}
long long target_tick_manager_mailboxes(const target_manager_c* self) {
  return guard(-1LL, [&] { return (long long)T(self)->mailboxCount(); });
}

}  // extern "C"
