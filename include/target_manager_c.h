/* include/target_manager_c.h -- reference-facing C-ABI of the B200 target manager.
 *
 * The first ten entry points are exactly the symbols of the reference's C wrapper
 * (/root/reference/include/target_estimation/target_manager_c.h:28-37, implemented in
 * /root/reference/src/target_manager_c.cpp:15-76): same names, argument order and meaning, so
 * libtarget_c.so of this repo can be loaded in place of the reference's libtarget_c.so.
 * Differences in error behaviour, all on paths where the reference has undefined behaviour:
 *   - target_manager_new returns NULL when the YAML file cannot be loaded (the reference lets a
 *     `throw "..."` cross the extern "C" boundary, src/target_manager.cpp:115);
 *   - target_manager_init on a manager without default model is a no-op (reference: same throw).
 * Getters return false for an unknown id and then copy the previous successful value of the same
 * getter into the output, like the reference's file-static scratch vectors
 * (src/target_manager_c.cpp:8-9,39-42).
 *
 * The *_batch entry points are extensions (the reference ABI is one target per call and has no
 * erase): one call = one kernel launch over the device-resident pool.  All buffers are caller-owned
 * host memory; nothing here exposes CUDA or torch types.
 */
#ifndef TARGET_MANAGER_C_B200_H
#define TARGET_MANAGER_C_B200_H
#ifndef __cplusplus
#include <stdbool.h>
#endif

typedef void target_manager_c;

#ifdef __cplusplus
extern "C" {
#endif
/* ---- reference ABI (target_manager_c.h:28-37) ---- */
target_manager_c* target_manager_new(const char* file);
void target_manager_init(const target_manager_c* self, const unsigned int id, const double dt0, double p0[], const double t0);
void target_manager_update_meas(const target_manager_c* self, const unsigned int id, const double dt, double meas[]);
void target_manager_update(const target_manager_c* self, const unsigned int id, const double dt);
bool target_manager_get_est_pose(const target_manager_c* self, const unsigned int id, double pose[]);
bool target_manager_get_est_twist(const target_manager_c* self, const unsigned int id, double twist[]);
bool target_manager_get_est_acceleration(const target_manager_c* self, const unsigned int id, double acceleration[]);
int target_manager_get_n_measurements(const target_manager_c* self, const unsigned int id);
void target_manager_log(const target_manager_c* self);
void target_manager_delete(target_manager_c* self);

/* ---- batched extensions (not in the reference) ---- */
/* same as target_manager_new, on an explicit CUDA device */
target_manager_c* target_manager_new_on_device(const char* file, int device);
/* TargetManager::init for n ids (default model): p0 [n][7]; returns #created (existing ids skipped) */
long long target_manager_init_batch(const target_manager_c* self, long long n, const unsigned int* ids, double dt0, const double* p0,
                                    const double* t0 /* [n] or NULL = 0 */);
/* one tick: action[k] 2 = update(id,dt,meas[k]) / 1 = update(id,dt) / 0 = skip; action NULL = all 2.
 * Returns #applied (unknown ids are skipped like the reference's "does not exist").  An id may be named more than once:
 * its records are applied in order, like the reference's sequential update() calls (one launch per run of distinct ids).
 * meas NULL with action NULL or with any action 2 is an error (-1, nothing applied). */
long long target_manager_update_batch(const target_manager_c* self, long long n, const unsigned int* ids, double dt, const double* meas,
                                      const unsigned char* action);
/* one dense tick from host arrays: record k belongs to the k-th id of target_manager_get_dense_ids (a plain manager: ascending ids;
 * a sharded one: shard-major) -- no ids travel and nothing is looked up; meas [n][meas_stride] (7 = pose, 3 = x y z for the linear
 * models), action [n] or NULL = all 2, est_pos_out [n][3] or NULL = every target's estimated position after the tick.  The copies,
 * the step and the read-back are pipelined (te_pool_tick_host).  Needs a manager whose targets share one model type.  _async
 * enqueues the tick and returns (three ticks may be in flight, buffers stay valid until done); _wait(0) waits for all, (lag) for all
 * but the newest `lag` (<= 2).  Returns the number of targets, -1 on error. */
long long target_manager_update_dense(const target_manager_c* self, double dt, const double* meas, int meas_stride, const unsigned char* action,
                                      double* est_pos_out);
long long target_manager_update_dense_async(const target_manager_c* self, double dt, const double* meas, int meas_stride,
                                            const unsigned char* action, double* est_pos_out);
int target_manager_update_dense_wait(const target_manager_c* self, int lag);
long long target_manager_get_dense_ids(const target_manager_c* self, unsigned int* out, long long cap);
/* TargetManager::update(dt): predict every target */
void target_manager_update_all(const target_manager_c* self, double dt);
/* TargetManager::erase; returns #erased */
long long target_manager_erase_batch(const target_manager_c* self, long long n, const unsigned int* ids);
bool target_manager_erase(const target_manager_c* self, unsigned int id);
/* estimates for n ids: any output may be NULL; found[k] = id exists.  t1 NULL = current estimates,
 * else getEstimatedPose/Twist/Acceleration(t1[k]) */
int target_manager_get_estimates_batch(const target_manager_c* self, long long n, const unsigned int* ids, const double* t1, double* pose7,
                                       double* twist6, double* acc6, unsigned char* found);
/* getAvailableTargets: ascending ids; returns the count (call with cap 0 to size the buffer) */
long long target_manager_get_ids(const target_manager_c* self, unsigned int* out, long long cap);
/* filter state of one target: x [n], P [n*n] row-major; returns n (0 = unknown id) */
int target_manager_get_state(const target_manager_c* self, unsigned int id, double* x, double* P, double* t);
/* pending per-id calls are coalesced into one launch per tick; force them out */
void target_manager_flush(const target_manager_c* self);
/* The k nearest targets inside a sphere at a given time (TargetManager::nearestTargets), on every handle: plain, on a device,
 * sharded, tick and sharded tick.  Query j = t1[j] (t1 NULL = current estimates), point[j][3], radius[j].  A target's position is
 * pose7[0:3] of target_manager_get_estimates_batch at t1[j], bit for bit; dist = sqrt((dx^2 + dy^2) + dz^2), every operation rounded
 * on its own; inside = dist <= radius[j].  count_out[j] = the number of targets inside; rows 0 .. min(k, count_out[j]) - 1 of
 * ids_out[j][k] / dist_out[j][k] are those targets by (dist, id), the other rows id 0xFFFFFFFF and dist -1.  Read-only.  0 <= k <=
 * 65536 (k == 0: counts only, ids_out / dist_out may be NULL); the arrays may be NULL only when q == 0; a negative or NaN radius is
 * an error, +inf asks for the k nearest of all.  The pose of a returned target is target_manager_get_estimates_batch(ids, t1).
 * Returns the total count, -1 on error. */
long long target_manager_nearest(const target_manager_c* self, long long q, const double* t1, const double* point, const double* radius, long long k,
                                 unsigned int* ids_out, double* dist_out, long long* count_out);
/* Gating: the k targets with the smallest Mahalanobis distance to a measured position (TargetManager::gatedTargets, whose comment
 * states the contract operation by operation), on every handle: plain, on a device, sharded, tick and sharded tick.  Query j = t1[j]
 * (t1 NULL = current estimates and covariances), z[j][3], gate[j].  A target's position p is pose7[0:3] of
 * target_manager_get_estimates_batch at t1[j], bit for bit; its position covariance C is the position block of P (t1 NULL) or of the
 * predict step A(tau) P A(tau)^T + Q to t1[j]; S = C + R[0:3,0:3]; d^2 = (p - z)^T S^-1 (p - z) through the Cholesky factor of S,
 * every operation rounded on its own; inside = d^2 <= gate[j], and a target whose S has no factor is never inside.  count_out[j] =
 * the number of targets inside; rows 0 .. min(k, count_out[j]) - 1 of ids_out[j][k] / d2_out[j][k] are those targets by (d^2, id),
 * the other rows id 0xFFFFFFFF and d^2 -1.  Read-only.  0 <= k <= 65536 (k == 0: counts only, ids_out / d2_out may be NULL); the
 * arrays may be NULL only when q == 0; a negative or NaN gate is an error, +inf asks for the k smallest distances of all.  The pose
 * of a returned target is target_manager_get_estimates_batch(ids, t1).  Returns the total count, -1 on error. */
long long target_manager_gated(const target_manager_c* self, long long q, const double* t1, const double* z, const double* gate, long long k,
                               unsigned int* ids_out, double* d2_out, long long* count_out);
/* Association of one frame: TargetManager::associate (contract of te_pool_associate in te_pool.h, INTEGRATION.md section 12).  The q
 * detections det[q][7] are stamped t1 and gated on their positions; each is assigned at most one target, greedily by (d^2, id, j)
 * over every detection's K best candidates (1 <= K <= 32); apply = 1 updates every assigned target with its detection at t1.
 * id_out / d2_out [q] = the assigned target and its d^2 (0xFFFFFFFF / -1: none), count_out [q] (may be NULL) = the candidates.
 * Returns the number of assigned detections, -1 on error (nothing applied). */
long long target_manager_associate(const target_manager_c* self, double t1, long long q, const double* det, double gate, int K, int apply,
                                   unsigned int* id_out, double* d2_out, long long* count_out);

/* ---- all GPUs of the box behind one handle (BASELINE.json north_star: targets shard by id, no collective on the hot path) ----
 * n_shards TargetManagers, shard r on CUDA device devices[r] (NULL = devices 0 .. n_shards-1), owner(id) = id mod n_shards.  The
 * handle is a valid target_manager_c* for every function above: per-id calls go to the owner, the *_batch calls route their records
 * to the owners on the host and run on all devices at once.  target_isolver_* (below) works on it as on a plain manager. */
target_manager_c* target_manager_new_sharded(const char* file, int n_shards, const int* devices);
/* number of shards behind the handle (1 for a plain manager) */
int target_manager_shards(const target_manager_c* self);
/* The optional exchange of estimates: [pose7 | twist6] records (13 doubles) of every target of every shard, all-gathered between
 * the devices over NCCL and read back from shard `publisher`'s device, shard-major; ids_out / records_out may be NULL (exchange
 * only).  Returns the number of records (call with cap 0 to size the buffers), -1 on error.  On a plain manager: its own records. */
long long target_manager_gather_estimates(const target_manager_c* self, unsigned int* ids_out, double* records_out, long long cap, int publisher);
/* device time of the exchange inside the last gather (ms, max over the devices); 1 if it went over NCCL, 0 for device copies */
double target_manager_last_gather_ms(const target_manager_c* self);
int target_manager_gather_uses_nccl(const target_manager_c* self);

/* ---- tick front-end: RosTargetManager semantics without ROS (src/target_manager_ros.cpp:26-92) ----
 * The handle is also a valid target_manager_c* for every function above. */
target_manager_c* target_tick_manager_new(const char* file, int device);
/* The same node loop over n_shards devices (devices[r], NULL = 0 .. n_shards-1; a device may repeat), owner(id) = id mod n_shards:
 * every /tf message is routed to the owners on the devices (te_group_route_records), every shard ticks on its own device at once.
 * The handle is valid for every target_tick_manager_* and every target_manager_* call above (target_manager_shards,
 * target_manager_gather_estimates included).  Differences from a one-device handle: target_tick_manager_published lists the poses
 * shard-major (shard 0's targets in ascending id, then shard 1's, ...: target_manager_get_dense_ids order); erased ids stay one
 * ascending list. */
target_manager_c* target_tick_manager_new_sharded(const char* file, int n_shards, const int* devices);
void target_tick_manager_set_expiration(const target_manager_c* self, double timeout_s);
void target_tick_manager_set_token(const target_manager_c* self, const char* token);
/* gather the filtered poses after every tick (the TF broadcast of src/target_manager_ros.cpp:78-87; default on) or leave them on the
 * device until a getter asks */
void target_tick_manager_set_publish(const target_manager_c* self, int on);
/* /tf callback: n transforms with child frame "<token>_<id>" (frames) or already-parsed ids */
void target_tick_manager_callback_frames(const target_manager_c* self, long long n, const char* const* child_frame_ids,
                                         const unsigned int* sec, const unsigned int* nsec, const double* poses /*[n][7]*/);
void target_tick_manager_callback_ids(const target_manager_c* self, long long n, const unsigned int* ids, const unsigned int* sec,
                                      const unsigned int* nsec, const double* poses /*[n][7]*/);
/* RosTargetManager::update(dt) with ros::Time::now() = (now_sec, now_nsec); returns #targets erased by the expiry
 * rule (their ids, ascending, into erased_out up to cap), or -1 on error */
long long target_tick_manager_update(const target_manager_c* self, double dt, unsigned int now_sec, unsigned int now_nsec,
                                     unsigned int* erased_out, long long cap);
/* the filtered poses broadcast by the last tick: ascending ids (shard-major on a sharded handle) + [n][7]; returns n */
long long target_tick_manager_published(const target_manager_c* self, unsigned int* ids_out, double* poses_out, long long cap);
double target_tick_manager_time(const target_manager_c* self);
long long target_tick_manager_mailboxes(const target_manager_c* self);

/* ---- recorded /tf input: rosbag v2.0 reader + the node's loop on the recording (bag_reader.hpp) ----
 * One record per transform, in record order; `msg` groups the transforms of one TFMessage (= one callback). */
typedef struct target_tf_record {
  unsigned int rec_sec, rec_nsec;   /* receive time of the message record */
  unsigned int msg;                 /* index of the message the transform came in */
  unsigned int seq, sec, nsec;      /* header.seq, header.stamp */
  char frame_id[64], child_frame_id[64];
  double pose[7];                   /* translation xyz, rotation xyzw (target_manager_ros.hpp:36-46) */
} target_tf_record;
/* returns the number of transforms on `topic` (NULL = "/tf"), the first `cap` of them in out; -1 on error */
long long target_bag_read_tf(const char* path, const char* topic, target_tf_record* out, long long cap);
/* src/target_node.cpp:36-44 on the bag's clock at `frequency` Hz, `extra_ticks` ticks past the last message.
 * stats_out (optional): ticks, messages, transforms, erased.  Returns the number of ticks, -1 on error. */
long long target_tick_manager_replay_bag(const target_manager_c* self, const char* path, const char* topic, double frequency,
                                         long long extra_ticks, long long stats_out[4]);
/* ---- sampled logging: the reference's log() under LOGGER_ON (src/target_interface.cpp:32-40,50-55) + writeTxtFile dumps ---- */
/* watch n ids (n = 0: stop and drop the series); every target_manager_log() call then appends one batched read-back of
 * measured_pose / pose_internal / twist / acceleration / P for the watched ids (at most max_samples samples) */
void target_manager_watch(const target_manager_c* self, long long n, const unsigned int* ids, long long max_samples);
long long target_manager_log_samples(const target_manager_c* self);
/* sample k of watched id j: row26 = [t | measured_pose 7 | pose_internal 6 | twist 6 | acceleration 6], P row-major n*n (either may
 * be NULL); returns the state size n, 0 if the id did not exist at that sample, -1 on a bad index */
int target_manager_log_sample(const target_manager_c* self, long long k, long long j, double* row26, double* P);
/* <folder>time_<id>, meas_pose_<id>, est_pose_<id>, est_twist_<id>, est_acc_<id>, cov_diag_<id> in the format of writeTxtFile
 * (utils.hpp:78-120), the files matlab/plot_target_manager_test.m loads; returns the number of files written, -1 on error */
int target_manager_write_log(const target_manager_c* self, const char* folder);
/* writeTxtFile itself (utils.hpp:78-120): cols == 1 writes the vector form */
int target_write_txt_file(const char* filename, const double* values, long long rows, long long cols);
const char* target_manager_last_error(void);

/* ---- IntersectionSolver (src/intersection_solver.cpp:42-124) on any handle: plain, on-device, sharded, tick, sharded tick ----
 * One solver holds n_streams solver streams; one stream = one reference IntersectionSolver object (previous intercept pose + two
 * moving-average windows of filters_length samples), updated by every pose query through it, in call order.  The per-id calls use
 * stream 0.  On a sharded handle every stream's state follows its queries from shard to shard (moved between the devices,
 * bit-exact), so the results equal those of the same solver on a plain manager.  A manager holding several model types keeps one
 * state per stream and model type.  The solver does not own the manager: delete it before the manager.  Errors: NULL / -1 / false
 * with target_manager_last_error(). */
typedef void target_isolver_c;
target_isolver_c* target_isolver_new(const target_manager_c* m, long long n_streams, unsigned filters_length);
void target_isolver_delete(target_isolver_c* s);
/* getIntersectionTimeWithSphere: time to the first contact with the sphere, -1 = none or unknown id */
double target_isolver_get_time(const target_isolver_c* s, unsigned id, double t1, const double origin[3], double radius);
/* getIntersectionPoseWithSphere: pose[7] = intercept pose (initPose 0 0 0 0 0 0 1 if none); true once both filtered errors are
 * below the thresholds.  t1, pos_th and ang_th must be >= 0. */
bool target_isolver_get_pose(const target_isolver_c* s, unsigned id, double t1, double pos_th, double ang_th, const double origin[3],
                             double radius, double pose[7]);
/* n queries at once: query k = ids[k] through stream[k] (NULL = k, then n <= n_streams for pose queries) at t1[k], sphere origin[k][3] / radius[k],
 * thresholds pos_th[k] / ang_th[k].  delta_out[k] = the time, pose7_out[k][7] / converged_out[k] = the pose query (pose7_out NULL =
 * times only: no stream is touched and the thresholds may be NULL); any output may be NULL.  A stream named more than once is
 * updated in call order, as by the same queries one by one.  Returns the number of queries whose id exists, -1 on error. */
long long target_isolver_query_batch(const target_isolver_c* s, long long n, const unsigned int* ids, const int* stream, const double* t1,
                                     const double* origin, const double* radius, const double* pos_th, const double* ang_th,
                                     double* delta_out, double* pose7_out, unsigned char* converged_out);
/* The k earliest sphere intercepts over every target of the manager (IntersectionSolver::earliestIntersections): sphere j = t1[j],
 * origin[j][3], radius[j].  hits_out[j] = the number of targets whose time (target_isolver_query_batch's delta, bit for bit) is >= 0;
 * rows 0 .. min(k, hits_out[j]) - 1 of ids_out[j][k] / delta_out[j][k] are those targets by (delta, id), the other rows id 0xFFFFFFFF
 * and delta -1.  Read-only: no solver stream is touched.  0 <= k <= 65536 (k == 0: counts only, ids_out / delta_out may be NULL); the
 * arrays may be NULL only when q == 0.  The intercept pose of a returned target is target_manager_get_estimates_batch(ids, t1 + delta).
 * Returns the total number of hits, -1 on error. */
long long target_isolver_earliest(const target_isolver_c* s, long long q, const double* t1, const double* origin, const double* radius, long long k,
                                  unsigned int* ids_out, double* delta_out, long long* hits_out);
/* host wall time of the last query by phase, ms: routing, stream moves between shards, the shards' device queries, results into
 * call order; returns 0, -1 on error */
int target_isolver_last_timing(const target_isolver_c* s, double ms_out[4]);

#ifdef __cplusplus
}
#endif
#endif
