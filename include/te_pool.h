/* include/te_pool.h -- thin extern "C" CUDA layer under the TargetManager host surface.
 *
 * The reference keeps one heap object per target (std::map<unsigned, shared_ptr<TargetInterface>>,
 * /root/reference/include/target_estimation/target_manager.hpp:36, each owning ~13 Eigen
 * matrices, include/target_estimation/kalman.hpp:107-127).  This layer replaces that storage
 * with one device-resident pool per model type: tiles of 32 targets laid out
 * [tile][field][lane] in HBM, slots kept in ascending-id order (std::map iteration order),
 * stepped by the sm_100a kernels in target_estimation_b200/csrc.  Nothing in this header
 * exists in the reference; the reference-facing ABI is include/target_manager_c.h.
 *
 * All functions return >= 0 on success and a negative value on error (te_last_error()).
 * "host" pointers are ordinary host memory; "dev" pointers are CUDA device memory of the
 * pool's device.  There is no CPU fallback: without a CUDA device every entry point fails.
 */
#ifndef TE_POOL_H
#define TE_POOL_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct te_pool te_pool;
typedef struct te_isolver te_isolver;

/* target_t of the reference (target_manager.hpp:38) */
enum { TE_ANGULAR_RATES = 0, TE_ANGULAR_VELOCITIES = 1, TE_UNIFORM_ACCELERATION = 2, TE_UNIFORM_VELOCITY = 3 };
/* per-target action of one tick */
enum { TE_ACT_NONE = 0,      /* target untouched this tick                                      */
       TE_ACT_PREDICT = 1,   /* TargetManager::update(id,dt)       (src/target_manager.cpp:204-218) */
       TE_ACT_UPDATE = 2 };  /* TargetManager::update(id,dt,meas)  (src/target_manager.cpp:190-202) */

const char* te_last_error(void);
int te_device_count(void);
int te_model_dims(int model, int* n, int* m);           /* state / measurement dims, asserts of src/types/*.cpp */
size_t te_model_bytes_per_step(int model);                /* SURVEY.md 8(d) algorithmic bytes per target-step */

/* page-lock / unlock a host buffer the caller owns (cudaHostRegister): read-backs into it then run at PCIe speed */
int te_host_register(void* ptr, size_t bytes);
int te_host_unregister(void* ptr);
/* ---- pool lifecycle ---------------------------------------------------------------- */
te_pool* te_pool_create(int model, int device, void* cuda_stream /* cudaStream_t or NULL = own stream */);
void te_pool_destroy(te_pool* p);
int te_pool_set_stream(te_pool* p, void* cuda_stream);
int te_pool_sync(te_pool* p);
int te_pool_set_variant(te_pool* p, int variant);         /* kernel shape (warps x stages); tuning knob */
/* test hook: at most max_ctas CTAs per step launch (0 = no cap), so that a small pool walks the persistent loops of the step
   kernels (grid-stride tiles, the TMA stage ring) as many times per CTA as a bench-size pool does on the whole machine */
int te_pool_set_grid_cap(te_pool* p, int max_ctas);
int te_pool_reserve(te_pool* p, size_t n_targets);   /* both buffer generations: no later tick pays for the allocation */
long long te_pool_size(te_pool* p);
size_t te_pool_device_bytes(te_pool* p);

/* Model class = (Q, R, P0) triple, row-major, interned by content.  The reference lets every
 * target carry its own matrices (TargetManager::init(type,id,dt0,t0,Q,R,P0,...),
 * src/target_manager.cpp:144-146).  Returns the class id. */
int te_pool_register_class(te_pool* p, const double* Q, const double* R, const double* P0);
int te_pool_class_count(te_pool* p);
int te_pool_get_class(te_pool* p, int cls, double* Q, double* R, double* P0);

/* ---- add / erase (stable stream compaction; ids stay ascending) ----------------------- */
/* TargetManager::init for a batch: ids already present are skipped ("already exists",
 * src/target_manager.cpp:177-178).  cls NULL = class 0; t0 NULL = 0; v0/a0 NULL = 0;
 * p0_scale NULL = 1 (P = p0_scale * P0[cls]).  Host pointers.  Returns #targets added. */
long long te_pool_add_batch(te_pool* p, long long n, const uint32_t* ids, const uint16_t* cls, const double* t0,
                            const double* p0 /*[n][7]*/, const double* v0 /*[n][6]*/, const double* a0 /*[n][6]*/,
                            const double* p0_scale);
/* TargetManager::erase for a batch (src/target_manager.cpp:227-241).  Returns #erased. */
long long te_pool_erase_batch(te_pool* p, long long n, const uint32_t* ids);
/* ascending ids (getAvailableTargets, src/target_manager.cpp:126-133); returns pool size */
long long te_pool_ids(te_pool* p, uint32_t* out, long long cap);
int te_pool_contains(te_pool* p, uint32_t id);
/* model class of one target (-1 with te_last_error() if the id is unknown) */
int te_pool_class_of(te_pool* p, uint32_t id);

/* ---- stepping (the hot path) -------------------------------------------------------- */
/* One tick over every slot, slot order = ascending id.  dev_meas: [size][meas_stride] doubles
 * (meas_stride 7 = reference pose [x y z qx qy qz qw]; 3 = xyz only, UV/UA pools only);
 * dev_action: [size] bytes of TE_ACT_* or NULL = default_action for all.  Device pointers. */
int te_pool_step_dense(te_pool* p, double dt, const double* dev_meas, int meas_stride, const uint8_t* dev_action,
                       int default_action);
/* Replay: n_ticks consecutive dense ticks in ONE launch.  dev_meas: [n_ticks][size][meas_stride], dev_action:
 * [n_ticks][size] or NULL.  Results are bit-identical to n_ticks calls of te_pool_step_dense (same arithmetic, same
 * order); each tile stays on chip for all its ticks, so state and covariance cross HBM once per launch instead of once
 * per tick (targets are independent: temporal blocking is exact).  For batched ingestion / catch-up / offline replay. */
int te_pool_step_dense_ticks(te_pool* p, int n_ticks, double dt, const double* dev_meas, int meas_stride, const uint8_t* dev_action,
                             int default_action);
/* Live launch: the 250 Hz loop over a SMALL pool (BASELINE configs[1]: 10 000 targets) without a kernel launch per tick.  One
 * resident launch holds every target in registers (uniform-velocity / uniform-acceleration pools of at most 8 tiles per SM:
 * 37 888 targets on a B200) and applies up to max_ticks ticks AS THEY ARE RELEASED: tick k reads dev_meas[k][size][meas_stride] and
 * dev_action[k][size] (NULL = default_action) once te_pool_live_release / te_pool_live_push has released it, and writes every
 * target's estimated position to dev_pos[k][size][3] (NULL = none).  Results are bit-identical to max_ticks calls of
 * te_pool_step_dense.  te_pool_live_push copies one tick's host arrays into the rings and releases it (in order, on the pool's copy
 * stream); te_pool_live_release(upto) releases ticks whose blocks the caller has written itself.  te_pool_live_wait(ticks) spins until
 * `ticks` ticks have been applied (the last warp of a tick writes a page-locked flag) and returns the number applied -- of ticks
 * released in one burst only the last is announced (every warp applies its ticks in order, so it stands for all of them): waiting
 * for a tick inside a burst returns when the burst is done;
 * te_pool_live_end stops the launch (unreleased ticks are skipped), waits for it and returns the ticks applied.  While the launch
 * runs the pool accepts no other call, and the process must not issue anything that waits for the whole device (cudaFree,
 * cudaDeviceSynchronize, cudaStreamCreate -- measured --, a legacy-default-stream operation): it would wait for the resident
 * launch, which waits for the host.  te_pool_destroy stops a launch that is still resident. */
int te_pool_live_begin(te_pool* p, int max_ticks, double dt, double* dev_meas, int meas_stride, uint8_t* dev_action, int default_action,
                       double* dev_pos);
int te_pool_live_release(te_pool* p, int upto);
int te_pool_live_push(te_pool* p, const double* meas, const uint8_t* action);
int te_pool_live_wait(te_pool* p, int ticks);
int te_pool_live_end(te_pool* p);
/* Same with HOST buffers: host->device copies are part of the call. */
int te_pool_step_dense_host(te_pool* p, double dt, const double* meas, int meas_stride, const uint8_t* action,
                            int default_action);
/* One dense tick from HOST buffers with the per-tick result read back: meas [size][meas_stride] and action
 * [size] (or NULL) go host->device, the tick runs, and est_pos_out (host, [size][3], may be NULL) receives
 * every target's estimated position (what RosTargetManager broadcasts each tick,
 * src/target_manager_ros.cpp:78-87).  Copies and kernels are pipelined in chunks of targets over internal
 * streams.  Synchronous: returns when est_pos_out is complete. */
int te_pool_tick_host(te_pool* p, double dt, const double* meas, int meas_stride, const uint8_t* action, int default_action,
                      double* est_pos_out);
/* The same, pipelined ACROSS ticks (batched ingestion of a recorded or buffered stream at PCIe speed in both directions): the call
 * enqueues the tick and returns; up to three ticks are in flight, so the host->device copies of tick k + 1 run under the kernels of
 * tick k and the device->host read-back of tick k - 1.  meas / action / est_pos_out of a tick must stay valid (and should be
 * page-locked) until that tick is done: te_pool_tick_host_wait(p, 0) waits for every tick issued, (p, lag) for all but the newest
 * `lag` ones (lag <= 2) -- the loop "async(k); wait(2); consume est_pos_out of tick k - 2" keeps the link busy in both directions
 * (three buffers of each kind on the caller's side; wait(1) with two buffers leaves the copy-in engine idle a tenth of the time).  A
 * fourth call waits for the tick three back by itself.  Results are those of te_pool_tick_host tick by tick. */
int te_pool_tick_host_async(te_pool* p, double dt, const double* meas, int meas_stride, const uint8_t* action, int default_action,
                            double* est_pos_out);
int te_pool_tick_host_wait(te_pool* p, int lag);
/* Sparse tick by id (host buffers): op k applies action[k] with dt[k] (dt_scalar if dt NULL) and
 * meas[k][7] to ids[k]; unknown ids are skipped.  An id may appear once per call: a repeated id is detected on the device
 * before anything is stepped -- nothing is applied then and -2 is returned (the caller splits the batch, as TargetManager::
 * updateBatch does).  Returns #applied. */
long long te_pool_step_ids(te_pool* p, long long n, const uint32_t* ids, const double* dt, double dt_scalar,
                           const double* meas /*[n][7]*/, const uint8_t* action /*NULL = UPDATE*/);
/* TargetManager::update(dt): predict every target (src/target_manager.cpp:220-225). */
int te_pool_predict_all(te_pool* p, double dt);

/* ---- read-back (every getter is a device sync point) --------------------------------- */
/* ids NULL = all targets in ascending-id order (n must equal pool size).  Any output may be NULL.
 * P is row-major [n][N*N]; measured_pose is the last measurement applied through an id/host API. */
int te_pool_read_state(te_pool* p, long long n, const uint32_t* ids, double* x, double* P, double* t, long long* n_meas,
                       double* prev_rpy /*[n][3]*/, double* measured_pose /*[n][7]*/);
/* getEstimatedPose/Twist/Acceleration([t1]) (src/types/*.cpp, src/target_interface.cpp:89-140).
 * t1 NULL = current values; otherwise t1[k] per query.  found[k] = 1 if the id exists. */
int te_pool_read_estimates(te_pool* p, long long n, const uint32_t* ids, const double* t1, double* pose7, double* twist6,
                           double* acc6, double* pose6_internal, uint8_t* found);
/* Estimate records of every slot into DEVICE memory: [size][13] = pose7 | twist6 (all-gather payload). */
int te_pool_estimates_dev(te_pool* p, double* dev_out);
/* raw device views for callers that keep their own buffers (bench, all-gather) */
const uint32_t* te_pool_dev_ids(te_pool* p);

/* ---- expiry (RosTargetManager::update, src/target_manager_ros.cpp:67-72) ---------------- */
/* Record per-target last measurement stamps (toSec(sec,nsec), utils.hpp:59-62) for ids. */
int te_pool_set_stamps(te_pool* p, long long n, const uint32_t* ids, const uint32_t* sec, const uint32_t* nsec);
/* Dense form of the above for device-resident ticks: every slot whose action (dev_action[slot], or default_action when
 * NULL) is TE_ACT_UPDATE gets toSec(sec, nsec) as its last measurement stamp.  Asynchronous on the pool's stream. */
int te_pool_stamp_dense(te_pool* p, const uint8_t* dev_action, int default_action, uint32_t sec, uint32_t nsec);
/* Erase every target with last_meas_time > 0 && (now - last_meas_time) >= timeout, evaluated on
 * the device in non-contracted FP64 (bit-exact with the reference compare).  erased_out receives the
 * ascending erased ids (up to cap).  Returns #erased. */
long long te_pool_expire(te_pool* p, uint32_t now_sec, uint32_t now_nsec, double timeout, uint32_t* erased_out,
                         long long cap);

/* One whole churn tick of RosTargetManager::update (src/target_manager_ros.cpp:52-76) for a device-resident stream:
 * te_pool_step_dense(dt, dev_meas, ...) + te_pool_stamp_dense(dev_action, default_action, stamp_*) +
 * te_pool_expire(now_*, timeout, ...), with identical results (survivor state bit-identical, same erased ids, same slot
 * order), but the stable compaction is FUSED into the step: the kernel reads each tile in place and writes the
 * survivors' columns straight to their compacted slots in the pool's second buffer, so an expiry tick moves the state
 * through HBM once instead of twice.  Targets that expire at the end of this tick are not stepped (their step is
 * unobservable).  Ticks on which nothing expires run the ordinary in-place step.  Returns #erased. */
long long te_pool_step_dense_expire(te_pool* p, double dt, const double* dev_meas, int meas_stride, const uint8_t* dev_action,
                                    int default_action, uint32_t stamp_sec, uint32_t stamp_nsec, uint32_t now_sec, uint32_t now_nsec,
                                    double timeout, uint32_t* erased_out, long long cap);

/* ---- device-resident mailboxes: the node loop of RosTargetManager for pools too large for a host loop ---------------- */
/* The reference keeps one Measurement mailbox per id in a std::map (include/target_estimation/target_manager_ros.hpp:74-134,
 * 176) and walks it once per tick on the host (src/target_manager_ros.cpp:46-76).  Here every target's mailbox lives beside
 * its slot on the device: the stored stamp and pose, last_meas_time_, and new_meas_ kept as the action byte of the next tick;
 * the pose and action arrays ARE the step kernel's measurement block and action array.  Only mailboxes whose id has no
 * target yet stay on the host (a handful per tick: ids seen for the first time), where the tick promotes them.
 *
 * te_pool_mailbox_ingest = RosTargetManager::measurementCallBack (src/target_manager_ros.cpp:26-39) for records whose frame
 * names are already parsed to ids (the caller stops at the first unparsable frame, as the reference loop does): record k =
 * (ids[k], sec[k], nsec[k], poses[k][7]), host arrays, applied in arrival order per id (Measurement::update).  Synchronous. */
int te_pool_mailbox_ingest(te_pool* p, long long n, const uint32_t* ids, const uint32_t* sec, const uint32_t* nsec,
                           const double* poses /*[n][7]*/);
/* The same in two halves, so that the copy of the NEXT message runs under the current tick (the /tf callback thread hands a message
 * over as it arrives; the 71 MB of a million records take as long over PCIe as the tick of a million targets):
 * te_pool_mailbox_prefetch registers the message and returns at once; its host->device copies enter the copy stream's queue as soon
 * as the next te_pool_mailbox_tick has queued its own small uploads (the device serves ONE host-to-device queue in order) and then
 * travel under that tick's kernels, ids and stamps first.  te_pool_mailbox_ingest_prefetched -- called after the tick, or whenever
 * the message should take effect -- applies it exactly as te_pool_mailbox_ingest would (lookup against the CURRENT slots, arrival
 * order per id, first sights queued from the host arrays); lookup and sort of the records already run under the tail of the copy.
 * The record arrays must stay valid (and should be page-locked) until te_pool_mailbox_ingest_prefetched returns.  One message can
 * be in flight. */
int te_pool_mailbox_prefetch(te_pool* p, long long n, const uint32_t* ids, const uint32_t* sec, const uint32_t* nsec, const double* poses /*[n][7]*/);
int te_pool_mailbox_ingest_prefetched(te_pool* p);
/* The same for a message that is already in DEVICE memory (another CUDA stage, a NCCL receive buffer) on the pool's stream: the
 * records are used in place; only the records of unknown ids (first sights) are read back for the host's queue. */
int te_pool_mailbox_ingest_dev(te_pool* p, long long n, const uint32_t* dev_ids, const uint32_t* dev_sec, const uint32_t* dev_nsec,
                               const double* dev_poses /*[n][7]*/);
/* te_pool_mailbox_tick = RosTargetManager::update(dt) (src/target_manager_ros.cpp:41-76) without the broadcast: readable
 * mailboxes of unknown ids become targets (class cls_new, p0 = the pose, t0 = t0_new, v0 = a0 = 0) and are updated with that pose,
 * targets with a readable mailbox are updated (the flag is sticky), the others predicted; every mailbox with
 * last_meas_time > 0 && now - last_meas_time >= timeout is erased with its target.  One stable rebuild (expired slots out,
 * new ids merged in, ascending ids kept) + one step launch.  Expired targets are not stepped (unobservable).  erased_out:
 * ascending erased ids (up to cap), target-less mailboxes included, as the reference erases those too; added_out / *n_added_out:
 * ascending ids of the targets created (up to added_cap) and their number.  Returns #erased.
 * Interplay with the by-hand calls, as in the reference: a target added through te_pool_add_batch has no mailbox until its
 * first record -- the tick does not touch it (the reference's loop walks mailboxes, not targets) -- unless its id already had a
 * target-less mailbox, which then feeds it; te_pool_erase_batch keeps the erased targets' mailboxes (they become target-less,
 * so a still-readable one re-creates its target on the next tick).  Once a pool keeps mailboxes, te_pool_step_dense_expire is
 * refused (it would leave them behind). */
long long te_pool_mailbox_tick(te_pool* p, double dt, double t0_new, int cls_new, uint32_t now_sec, uint32_t now_nsec, double timeout,
                               uint32_t* erased_out, long long cap, uint32_t* added_out, long long added_cap, long long* n_added_out);
/* mailboxes alive = slots that have one + target-less ones (measurements_.size() of the reference); a device reduction + sync */
long long te_pool_mailbox_count(te_pool* p);
/* cheap upper bound of the above (no device work): enough room for the erased / added lists of the next tick */
long long te_pool_mailbox_bound(te_pool* p);
/* device views of the mailboxes in slot order: stored pose [size][7], action byte of the next tick [size] (NULL before first use) */
const double* te_pool_mailbox_dev_pose(te_pool* p);
const uint8_t* te_pool_mailbox_dev_action(te_pool* p);
/* ---- batched IntersectionSolver (src/intersection_solver.cpp) ---------------------------- */
/* n_streams independent solver states (each = one reference IntersectionSolver object: two moving
 * average filters of filters_length samples + previous intersection pose). */
te_isolver* te_isolver_create(te_pool* p, long long n_streams, unsigned filters_length);
void te_isolver_destroy(te_isolver* s);
/* query k: target ids[k] through solver stream stream[k] (NULL = k).  Each stream may appear at most
 * once per call.  delta_t[k] = getIntersectionTimeWithSphere (-1 = none); pose7/converged as
 * getIntersectionPoseWithSphere (pass pose7 NULL to only compute delta_t without touching filters).
 * Returns the number of queries whose id exists. */
int te_isolver_query(te_isolver* s, long long n, const uint32_t* ids, const int32_t* stream, const double* t1,
                     const double* origin /*[n][3]*/, const double* radius, const double* pos_th, const double* ang_th,
                     double* delta_t, double* pose7, uint8_t* converged);
/* Move the complete state of the listed streams (previous pose, both windows, both sums, window index, complete flag) from src to
 * dst: two solvers of the same model type and filters_length, usually of pools on two devices.  Afterwards stream streams[k] of dst
 * holds, byte for byte, what stream streams[k] of src held; src keeps its copy.  The streams are gathered into one block on src's
 * device (isolver_pack_streams_kernel), copied once (peer copy between devices, device copy on one), and scattered on dst's device
 * (isolver_unpack_streams_kernel).  Each solver's staging grows only when a move is larger than any before.  Synchronous. */
int te_isolver_move_streams(te_isolver* src, te_isolver* dst, long long n, const int32_t* streams);

/* The k earliest sphere intercepts over every target of the pool (read-only: no solver stream, filter or target state is touched).
 * Sphere j = (t1[j], origin[j][3], radius[j]), host arrays.  For target i, delta_ij is bit for bit te_isolver_query's delta_t for
 * (i, t1[j], origin[j], radius[j]); a hit is delta >= 0 (-0.0 is a hit and ranks as 0; -1 and NaN are not).  hits_out[j] = the
 * number of hits; rows 0 .. min(k, hits_out[j]) - 1 of ids_out[j][.] / delta_out[j][.] are those hits ordered by (delta, id), delta
 * as te_isolver_query returns it; the remaining rows are id 0xFFFFFFFF and delta -1.  0 <= k <= 65536; k == 0 gives the counts
 * only (ids_out / delta_out may then be NULL).  The targets are swept on the device in chunks of spheres sized from the pool, the
 * k-th key of every sphere is found by radix select, and only q x k rows cross to the host.  Uniform-velocity and angular-velocity
 * pools never intercept (zero t^4 coefficient) and run no kernel.  Synchronous.  Returns the total number of hits. */
long long te_pool_earliest_intersections(te_pool* p, long long q, const double* t1, const double* origin /*[q][3]*/, const double* radius,
                                         long long k, uint32_t* ids_out /*[q][k]*/, double* delta_out /*[q][k]*/, long long* hits_out /*[q]*/);
/* The k nearest targets inside a sphere, over every target of the pool (read-only).  Query j = (t1[j], point[j][3], radius[j]), host
 * arrays; t1 NULL = every target's current estimate.  The position p_i of target i is pose7[0:3] of te_pool_read_estimates at t1[j]
 * (t1 NULL: at none), bit for bit; dist_ij = sqrt_rn((dx^2 + dy^2) + dz^2) with d = p_i - point[j], every operation rounded on its
 * own in that order (no FMA).  A target is inside when dist_ij <= radius[j] (the boundary counts, NaN never does).  count_out[j] =
 * the number of targets inside; rows 0 .. min(k, count_out[j]) - 1 of ids_out[j][.] / dist_out[j][.] are those targets ordered by
 * (dist, id), the remaining rows id 0xFFFFFFFF and dist -1.  Argument rules as te_pool_earliest_intersections; a negative or NaN
 * radius is an error (radius = +inf: plain k nearest).  Every model type runs the kernels.  Synchronous.  Returns the total count. */
long long te_pool_nearest_targets(te_pool* p, long long q, const double* t1 /*[q] or NULL*/, const double* point /*[q][3]*/, const double* radius,
                                  long long k, uint32_t* ids_out /*[q][k]*/, double* dist_out /*[q][k]*/, long long* count_out /*[q]*/);
/* Gating: the k targets with the smallest Mahalanobis distance to a measured position, over every target of the pool (read-only).
 * Query j = (t1[j], z[j][3], gate[j]), host arrays.  For query j and target i, with state x, covariance P, time t, model class
 * (Q, R) and state layout of kinematic block size B:
 *  1. Position: p = pose7[0:3] of te_pool_read_estimates at t1[j], bit for bit (what te_pool_nearest_targets uses); t1 NULL: the
 *     current estimate.
 *  2. Position covariance C (3 x 3).  P, Q and R are always read through their upper triangle: entry (r, c) with r > c is taken
 *     from (c, r) (what the packed kernels keep current).
 *     t1 NULL: C(a,b) = P(a,b); no predict step, no Q.
 *     t1 given: C = the position block of the predict step A(tau) P A(tau)^T + Q with tau = t1[j] - t and h = (0.5*tau)*tau, in
 *     the operation order of predict_kinematic, every operation rounded on its own (no contraction).  Position-derivative offsets
 *     o: UV (0, 3), UA (0, 3, 6), AR (0, 6, 12), AV (0, 6) -- the position rows of AV's EKF Jacobian are [I 0 tau*I 0], and the
 *     position block of F P F^T depends only on those rows.  m[u][v] = P(o_u + a, o_v + b); rows first:
 *     r[v] = (m[0][v] + tau*m[1][v]) + h*m[2][v]; then columns: c = (r[0] + tau*r[1]) + h*r[2] (the h terms only with three
 *     offsets); C(a,b) = c + Q(a,b).
 *  3. Innovation covariance: S = C + R[0:3,0:3], the position rows and columns of the class's M x M R.
 *  4. Distance: d = p - z[j], rounded per component.  Cholesky factor, in this order: L00 = sqrt(S00); L10 = S10/L00;
 *     L20 = S20/L00; L11 = sqrt(S11 - L10*L10); L21 = (S21 - L20*L10)/L11; L22 = sqrt((S22 - L20*L20) - L21*L21).  Forward
 *     solve: w0 = d0/L00; w1 = (d1 - L10*w0)/L11; w2 = ((d2 - L20*w0) - L21*w1)/L22.  d^2 = (w0*w0 + w1*w1) + w2*w2.  A target
 *     whose factor does not exist (any radicand <= 0 or NaN) is never a candidate.
 *  5. Selection: a target is inside when d^2 <= gate[j] (the boundary counts).  count_out[j] = the number of targets inside; rows
 *     0 .. min(k, count) - 1 of ids_out[j][.] / d2_out[j][.] hold those targets ordered by (d^2, id); the remaining rows hold id
 *     0xFFFFFFFF and d^2 -1.
 *  6. The query is read-only.  Returns the total count.
 *  7. Argument rules as te_pool_nearest_targets with gate in place of radius: 0 <= k <= 65536 (k == 0: counts only, ids_out /
 *     d2_out may then be NULL); a negative or NaN gate is an error, +inf asks for the k smallest distances over every target whose
 *     S has a factor.
 * Gating is on position only, for every model: for UV / UA that is the filter's full innovation, for AR / AV the exact position
 * marginal of the 6-D innovation.  Synchronous. */
long long te_pool_gated_targets(te_pool* p, long long q, const double* t1 /*[q] or NULL*/, const double* z /*[q][3]*/, const double* gate,
                                long long k, uint32_t* ids_out /*[q][k]*/, double* d2_out /*[q][k]*/, long long* count_out /*[q]*/);

/* ---- association: one frame of unlabelled position detections (INTEGRATION.md section 12, DESIGN.md section 4.10) ---------- */
/* All q detections are stamped t1; detection j is a pose record det[j][0:7] (the record te_pool_step_ids takes) and is gated on its
 * position z_j = det[j][0:3] only.
 *  1. Candidates: target i is a candidate for detection j when t_i <= t1 (a NaN time never is: the update needs dt >= 0) and
 *     d2_ij <= gate, d2_ij being bit for bit te_pool_gated_targets' d^2 for the query (t1, z_j) (its steps 1-4).  count_out[j] = the
 *     number of candidates (count_out may be NULL).  The candidate list of j = its first min(K, count) candidates by (d^2, id): when
 *     every target has t <= t1, exactly te_pool_gated_targets(t1, z_j, gate, k = K)'s rows and count.
 *  2. Assignment, greedy on sorted edges: the edges (j, i, d^2) of all candidate lists, visited in ascending (d^2, id, j) order; an
 *     edge is taken when neither its detection nor its target is taken yet.  id_out[j] / d2_out[j] = the assigned target and its d^2,
 *     0xFFFFFFFF / -1 for a detection without one.  K bounds the work: a detection whose K candidates all go to better edges stays
 *     unassigned even when it has further candidates.
 *  3. apply = 1: every assigned target i gets update(i, t1 - t_i, det[j]) -- dt rounded once, the result bit for bit that of
 *     te_pool_step_ids with that per-row dt and measurement (t, n_meas and measured_pose change as there); other targets are not
 *     touched.  apply = 0: read-only.
 *  4. Argument errors (nothing applied): t1 not finite; gate negative, NaN or +inf (+inf has no spatial bound: te_pool_gated_targets
 *     serves it); K outside [1, 32]; q < 0; det, id_out or d2_out NULL while q > 0.
 * The candidates come from a grid index over every target's gate box (no q x size sweep), the matching runs on the device, and only
 * the detections go up and q ids, d^2 and counts come back.  Synchronous.  Returns the number of assigned detections. */
long long te_pool_associate(te_pool* p, double t1, long long q, const double* det /*[q][7]*/, double gate, int K, int apply,
                            uint32_t* id_out /*[q]*/, double* d2_out /*[q]*/, long long* count_out /*[q] or NULL*/);
/* Step 1 alone, read-only: the candidate lists of q positions z[q][3] over the pool, rows ids_out[j][.] / d2_out[j][.] by (d^2, id)
 * and rows of id 0xFFFFFFFF / d^2 -1 after them (the rows several pools' lists are merged from, as gatedTargets merges).  Argument
 * rules of te_pool_associate with z for det and ids_out for id_out.  Returns the total count. */
long long te_pool_gated_candidates(te_pool* p, double t1, long long q, const double* z /*[q][3]*/, double gate, int K,
                                   uint32_t* ids_out /*[q][K]*/, double* d2_out /*[q][K]*/, long long* count_out /*[q] or NULL*/);
/* Step 2 alone over host rows, on p's device and stream (p's targets are not read): detection j's rows ids[j][.] / d2[j][.] hold its
 * candidates by (d^2, id) with d^2 >= 0, then rows of d^2 -1 (any other layout is an error).  id_out / d2_out as te_pool_associate.
 * 1 <= K <= 32.  Returns the number of assigned detections. */
long long te_assign_greedy(te_pool* p, long long q, int K, const uint32_t* ids /*[q][K]*/, const double* d2 /*[q][K]*/, uint32_t* id_out /*[q]*/,
                           double* d2_out /*[q]*/);
/* Step 3 alone: op k = update(ids[k], t1 - t, meas[k]) with dt = t1 - t of the target computed on the device (rounded once), then
 * the path of te_pool_step_ids (same scatter, duplicate check -- -2, nothing applied -- and step launch).  Unknown ids are skipped;
 * a target with t > t1 (or a NaN t) is an error and nothing is applied.  t1 must be finite.  Returns #applied. */
long long te_pool_update_at(te_pool* p, long long n, const uint32_t* ids, double t1, const double* meas /*[n][7]*/);
/* What the pool's last te_pool_associate / te_pool_gated_candidates / te_assign_greedy call saw: out[0] = grid levels that held a
 * target, out[1] = targets on the list every detection checks directly (a non-finite gate box), out[2] = candidates over all
 * detections, out[3] = matching rounds (0 for te_pool_gated_candidates). */
int te_pool_assoc_stats(te_pool* p, long long* out /*[4]*/);

/* Dense device-resident form: one query per slot (query k = slot k = solver stream k; needs n_streams >= pool size).
 * dev_t1 NULL = each target's own time; dev_delta / dev_pose7 / dev_converged may be NULL.  Asynchronous. */
int te_isolver_query_dense(te_isolver* s, const double* dev_t1, const double* dev_origin /*[size][3]*/, const double* dev_radius,
                           double pos_th, double ang_th, double* dev_delta, double* dev_pose7, uint8_t* dev_converged);

/* ---- several pools on several devices of one box (targets shard by id: owner = id mod n, no collective on the hot path) ------ */
/* A group = the devices of the shards, in shard order, + one NCCL communicator per device created in this process
 * (ncclCommInitAll; libnccl.so.2 is loaded on first use).  Two shards on the SAME device (a one-GPU test of the sharded host
 * logic) cannot form a NCCL clique: such a group moves the records with device-to-device copies instead. */
typedef struct te_group te_group;
te_group* te_group_create(int n, const int* devices);
void te_group_destroy(te_group* g);
int te_group_size(te_group* g);
/* 1 = NCCL communicators, 0 = same-device copies (see above) */
int te_group_uses_nccl(te_group* g);
/* The optional all-gather of estimates to the publishing rank(s) (SURVEY.md 8(e)): every pool writes its [size][13] =
 * pose7 | twist6 records (te_pool_estimates_dev) on its own stream, then every device receives the records -- and the ids -- of
 * all shards, shard-major (shard 0's targets in ascending id, then shard 1's, ...): ncclAllGather when the shards hold equally
 * many targets, else one ncclBroadcast per shard inside one NCCL group (ragged all-gather, nothing padded).  pools[r] = the
 * pool of shard r (NULL = that shard has no target of this model).  counts_out[r] (optional) = records of shard r.  Asynchronous:
 * ordered on each pool's stream; te_group_sync waits.  Returns the total number of records, -1 on error. */
long long te_group_allgather_estimates(te_group* g, te_pool* const* pools, long long* counts_out);
int te_group_sync(te_group* g);
/* device views of the gathered records / ids on shard r's device (valid until the next gather) */
const double* te_group_dev_records(te_group* g, int r);
const uint32_t* te_group_dev_ids(te_group* g, int r);
/* the gathered records / ids from shard `root`'s device into host buffers ([total][13] doubles, [total] ids; either may be NULL) */
long long te_group_fetch(te_group* g, int root, double* records_out, uint32_t* ids_out, long long cap);
/* device time of the last gather (ms, max over the devices; CUDA events around the collective on every device's stream) */
double te_group_last_gather_ms(te_group* g);
/* Route one /tf message (host arrays, arrival order; should be page-locked) to the shards' devices: record k belongs to shard
 * ids[k] mod G.  The message is cut into G contiguous chunks by position; chunk c is copied to shard c's device (the G links copy at
 * once) and partitioned there by owner, stably (te_route_partition_kernel); then every shard receives its runs, [from chunk 0 | from
 * chunk 1 | ...], over grouped NCCL send / receive between distinct devices, by device copies otherwise.  Arrival order per id is
 * kept.  pools[r] = the pool of shard r (its device and stream; none may be NULL).  Asynchronous, ordered on each pool's stream like
 * te_group_allgather_estimates (the host waits only for the G x G owner counts).  Afterwards te_group_routed() gives shard r's
 * records on its own device, in arrival order: four SoA arrays that te_pool_mailbox_ingest_dev takes as they are (valid until the
 * next routed message).  counts_out[r] (optional) = records of shard r.  The buffers grow with the largest message seen and are
 * reused.  Returns n, -1 on error. */
long long te_group_route_records(te_group* g, te_pool* const* pools, long long n, const uint32_t* ids, const uint32_t* sec,
                                 const uint32_t* nsec, const double* poses /*[n][7]*/, long long* counts_out);
int te_group_routed(te_group* g, int r, long long* n, const uint32_t** dev_ids, const uint32_t** dev_sec,
                    const uint32_t** dev_nsec, const double** dev_poses);

/* ---- device micro-benchmarks behind the roofline statements (csrc/te_diag.cu; not on any product path) ---------------------- */
/* FP64 FMA rate of `device` in TFLOP/s (dependent-chain kernel, 8 chains per thread, best of 5) and the rate of a plain streaming
 * copy kernel in GB/s (read + write bytes, 1 GiB each way); either output may be NULL */
int te_diag_device_peaks(int device, double* fp64_tflops_out, double* copy_gbs_out);

#ifdef __cplusplus
}
#endif
#endif /* TE_POOL_H */
