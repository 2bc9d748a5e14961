"""Thin numpy/torch harness over include/te_pool.h.  Host arrays are numpy; device buffers are torch
CUDA tensors (torch is only plumbing: memory + streams)."""
import ctypes as C
import os

import numpy as np

from ._lib import lib, check, TeError

ANGULAR_RATES, ANGULAR_VELOCITIES, UNIFORM_ACCELERATION, UNIFORM_VELOCITY = 0, 1, 2, 3   # target_manager.hpp:38
MODEL_TYPES = {"angular_rates": 0, "angular_velocities": 1, "uniform_acceleration": 2, "uniform_velocity": 3}
ACT_NONE, ACT_PREDICT, ACT_UPDATE = 0, 1, 2

_MODELS_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "models")


def model_dims(model):
    n, m = C.c_int(), C.c_int()
    check(lib.te_model_dims(model, C.byref(n), C.byref(m)))
    return n.value, m.value


def bytes_per_step(model):
    return int(lib.te_model_bytes_per_step(model))


def load_model(name_or_path):
    """Read a models/*.yaml file the way TargetManager::loadYamlFile does (src/target_manager.cpp:18-104):
    flat lists mapped COLUMN-major (Eigen::Map<MatrixXd>), size = sqrt(len).  Returns
    (type, frequency, Q, R, P) with row-major numpy matrices M[i, j] = list[i + s*j]."""
    import yaml
    path = name_or_path
    if not os.path.exists(path):
        path = os.path.join(_MODELS_DIR, "model_%s_params.yaml" % name_or_path)
    with open(path) as f:
        node = yaml.safe_load(f)
    out = []
    for key in ("Q", "R", "P"):
        v = np.asarray(node[key], dtype=np.float64)
        s = int(np.sqrt(v.size))
        out.append(np.ascontiguousarray(v[: s * s].reshape(s, s).T))
    return MODEL_TYPES[node["type"]], float(node.get("frequency", 0.0)), out[0], out[1], out[2]


def _np(a, dtype, shape=None):
    if a is None:
        return None
    a = np.ascontiguousarray(a, dtype=dtype)
    if shape is not None:
        a = a.reshape(shape)
    return a


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _dev_ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class TargetPool:
    """One device-resident pool of targets of a single model type (include/te_pool.h)."""

    def __init__(self, model, device=0, stream=None):
        if isinstance(model, str):
            model = MODEL_TYPES[model]
        self.model = model
        self.n_state, self.n_meas_dim = model_dims(model)
        self.device = device
        self._h = lib.te_pool_create(model, device, stream)
        if not self._h:
            from ._lib import last_error
            raise TeError(last_error())

    def close(self):
        if getattr(self, "_h", None):
            lib.te_pool_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        return int(lib.te_pool_size(self._h))

    # -- configuration ---------------------------------------------------------------------
    def set_variant(self, v):
        check(lib.te_pool_set_variant(self._h, int(v)))

    def set_grid_cap(self, max_ctas):
        check(lib.te_pool_set_grid_cap(self._h, int(max_ctas)))

    def set_stream(self, stream_ptr):
        check(lib.te_pool_set_stream(self._h, stream_ptr))

    def sync(self):
        check(lib.te_pool_sync(self._h))

    def reserve(self, n):
        check(lib.te_pool_reserve(self._h, int(n)))

    def device_bytes(self):
        return int(lib.te_pool_device_bytes(self._h))

    def register_class(self, Q, R, P0):
        n, m = self.n_state, self.n_meas_dim
        Q = _np(Q, np.float64, (n, n)); R = _np(R, np.float64, (m, m)); P0 = _np(P0, np.float64, (n, n))
        return check(lib.te_pool_register_class(self._h, _ptr(Q), _ptr(R), _ptr(P0)))

    # -- add / erase -----------------------------------------------------------------------
    def add(self, ids, p0, cls=None, t0=None, v0=None, a0=None, p0_scale=None):
        ids = _np(ids, np.uint32)
        n = ids.size
        p0 = _np(p0, np.float64, (n, 7))
        cls = _np(cls, np.uint16); t0 = _np(t0, np.float64)
        v0 = _np(v0, np.float64, (n, 6)) if v0 is not None else None
        a0 = _np(a0, np.float64, (n, 6)) if a0 is not None else None
        p0_scale = _np(p0_scale, np.float64)
        return check(lib.te_pool_add_batch(self._h, n, _ptr(ids), _ptr(cls), _ptr(t0), _ptr(p0), _ptr(v0), _ptr(a0), _ptr(p0_scale)))

    def erase(self, ids):
        ids = _np(ids, np.uint32)
        return check(lib.te_pool_erase_batch(self._h, ids.size, _ptr(ids)))

    def ids(self):
        n = len(self)
        out = np.empty(n, dtype=np.uint32)
        check(lib.te_pool_ids(self._h, _ptr(out), n))
        return out

    def contains(self, id_):
        return bool(check(lib.te_pool_contains(self._h, int(id_))))

    # -- stepping --------------------------------------------------------------------------
    def step_dense(self, dt, dev_meas=None, meas_stride=7, dev_action=None, default_action=ACT_UPDATE):
        check(lib.te_pool_step_dense(self._h, float(dt), _dev_ptr(dev_meas), int(meas_stride), _dev_ptr(dev_action), int(default_action)))

    def step_dense_ticks(self, n_ticks, dt, dev_meas=None, meas_stride=7, dev_action=None, default_action=ACT_UPDATE):
        """n_ticks ticks in one launch: dev_meas [n_ticks][n][stride], dev_action [n_ticks][n] (torch CUDA tensors)"""
        check(lib.te_pool_step_dense_ticks(self._h, int(n_ticks), float(dt), _dev_ptr(dev_meas), int(meas_stride), _dev_ptr(dev_action),
                                           int(default_action)))

    # -- live launch: ticks released one by one into one resident launch (te_pool_live_*) --
    def live_begin(self, max_ticks, dt, dev_meas=None, meas_stride=7, dev_action=None, default_action=ACT_UPDATE, dev_pos=None):
        self._live_keep = (dev_meas, dev_action, dev_pos)
        check(lib.te_pool_live_begin(self._h, int(max_ticks), dt, _dev_ptr(dev_meas), meas_stride, _dev_ptr(dev_action), default_action, _dev_ptr(dev_pos)))

    def live_release(self, upto):
        return check(lib.te_pool_live_release(self._h, int(upto)))

    def live_push(self, meas, action=None):
        meas = _np(meas, np.float64); action = _np(action, np.uint8) if action is not None else None
        self._live_host = (meas, action)
        return check(lib.te_pool_live_push(self._h, _ptr(meas), _ptr(action)))

    def live_wait(self, ticks):
        return check(lib.te_pool_live_wait(self._h, int(ticks)))

    def live_end(self):
        n = check(lib.te_pool_live_end(self._h))
        self._live_keep = None
        return n

    def step_dense_host(self, dt, meas=None, action=None, default_action=ACT_UPDATE, meas_ptr=None, meas_stride=7, action_ptr=None):
        """Host buffers (numpy) or raw host pointers (pinned torch tensors: pass data_ptr())."""
        if meas is not None:
            meas = _np(meas, np.float64)
            meas_stride = meas.shape[-1] if meas.ndim == 2 else meas_stride
            meas_ptr = meas.ctypes.data
        if action is not None:
            action = _np(action, np.uint8)
            action_ptr = action.ctypes.data
        check(lib.te_pool_step_dense_host(self._h, float(dt), C.c_void_p(meas_ptr) if meas_ptr else None, int(meas_stride),
                                          C.c_void_p(action_ptr) if action_ptr else None, int(default_action)))

    def step_ids(self, ids, dt, meas=None, action=None):
        ids = _np(ids, np.uint32)
        n = ids.size
        dt_arr = None
        dt_scalar = 0.0
        if np.ndim(dt) == 0:
            dt_scalar = float(dt)
        else:
            dt_arr = _np(dt, np.float64)
        meas = _np(meas, np.float64, (n, 7)) if meas is not None else None
        action = _np(action, np.uint8)
        return check(lib.te_pool_step_ids(self._h, n, _ptr(ids), _ptr(dt_arr), dt_scalar, _ptr(meas), _ptr(action)))

    def predict_all(self, dt):
        check(lib.te_pool_predict_all(self._h, float(dt)))

    # -- read-back -------------------------------------------------------------------------
    def read_state(self, ids=None, want=("x", "P", "t", "n_meas", "prev_rpy", "measured_pose")):
        if ids is not None:
            ids = _np(ids, np.uint32)
            n = ids.size
        else:
            n = len(self)
        N = self.n_state
        out = {}
        if "x" in want: out["x"] = np.zeros((n, N))
        if "P" in want: out["P"] = np.zeros((n, N, N))
        if "t" in want: out["t"] = np.zeros(n)
        if "n_meas" in want: out["n_meas"] = np.zeros(n, dtype=np.int64)
        if "prev_rpy" in want: out["prev_rpy"] = np.zeros((n, 3))
        if "measured_pose" in want: out["measured_pose"] = np.zeros((n, 7))
        check(lib.te_pool_read_state(self._h, n, _ptr(ids), _ptr(out.get("x")), _ptr(out.get("P")), _ptr(out.get("t")),
                                     _ptr(out.get("n_meas")), _ptr(out.get("prev_rpy")), _ptr(out.get("measured_pose"))))
        return out

    def read_estimates(self, ids=None, t1=None):
        if ids is not None:
            ids = _np(ids, np.uint32)
            n = ids.size
        else:
            n = len(self)
        t1 = _np(np.broadcast_to(t1, (n,)), np.float64) if t1 is not None else None
        out = {"pose": np.zeros((n, 7)), "twist": np.zeros((n, 6)), "acc": np.zeros((n, 6)), "pose6": np.zeros((n, 6)),
               "found": np.zeros(n, dtype=np.uint8)}
        check(lib.te_pool_read_estimates(self._h, n, _ptr(ids), _ptr(t1), _ptr(out["pose"]), _ptr(out["twist"]), _ptr(out["acc"]),
                                         _ptr(out["pose6"]), _ptr(out["found"])))
        return out

    def estimates_dev(self, dev_out):
        check(lib.te_pool_estimates_dev(self._h, _dev_ptr(dev_out)))

    # -- expiry ----------------------------------------------------------------------------
    def set_stamps(self, ids, sec, nsec):
        ids = _np(ids, np.uint32); sec = _np(sec, np.uint32); nsec = _np(nsec, np.uint32)
        check(lib.te_pool_set_stamps(self._h, ids.size, _ptr(ids), _ptr(sec), _ptr(nsec)))

    def stamp_dense(self, sec, nsec, dev_action=None, default_action=ACT_UPDATE):
        check(lib.te_pool_stamp_dense(self._h, _dev_ptr(dev_action), int(default_action), int(sec), int(nsec)))

    def expire(self, now_sec, now_nsec, timeout):
        cap = len(self)
        buf = getattr(self, "_erase_buf", None)
        if buf is None or buf.size < cap:        # reusable output buffer: allocating 4 B x pool size per tick costs more than the expiry
            buf = self._erase_buf = np.empty(max(cap + cap // 4, 1), dtype=np.uint32)
        n = check(lib.te_pool_expire(self._h, int(now_sec), int(now_nsec), float(timeout), _ptr(buf), cap))
        return buf[:n].copy()

    def step_dense_expire(self, dt, dev_meas, meas_stride, dev_action, default_action, stamp, now, timeout):
        """one churn tick = step_dense + stamp_dense(stamp) + expire(now, timeout) with the compaction fused into the step;
        stamp / now are (sec, nsec) pairs.  Returns the erased ids (ascending)."""
        cap = len(self)
        buf = getattr(self, "_erase_buf", None)
        if buf is None or buf.size < cap:
            buf = self._erase_buf = np.empty(max(cap + cap // 4, 1), dtype=np.uint32)
        n = check(lib.te_pool_step_dense_expire(self._h, float(dt), _dev_ptr(dev_meas), int(meas_stride), _dev_ptr(dev_action), int(default_action),
                                                int(stamp[0]), int(stamp[1]), int(now[0]), int(now[1]), float(timeout), _ptr(buf), cap))
        return buf[:n].copy()


    # -- device-resident mailboxes: the node loop of RosTargetManager (include/te_pool.h) -------
    def mailbox_ingest(self, ids, sec, nsec, poses):
        """one /tf message: records (id, stamp, pose7) in arrival order (measurementCallBack, src/target_manager_ros.cpp:26-39)"""
        ids = _np(ids, np.uint32); sec = _np(sec, np.uint32); nsec = _np(nsec, np.uint32)
        poses = _np(poses, np.float64, (ids.size, 7))
        check(lib.te_pool_mailbox_ingest(self._h, ids.size, _ptr(ids), _ptr(sec), _ptr(nsec), _ptr(poses)))

    def mailbox_prefetch(self, ids, sec, nsec, poses):
        """start the host->device copy of the NEXT message and return (it runs under the current tick); the arrays must stay alive
        and unchanged until mailbox_ingest_prefetched() -- they are kept referenced here"""
        ids = _np(ids, np.uint32); sec = _np(sec, np.uint32); nsec = _np(nsec, np.uint32)
        poses = _np(poses, np.float64, (ids.size, 7))
        self._prefetched = (ids, sec, nsec, poses)
        check(lib.te_pool_mailbox_prefetch(self._h, ids.size, _ptr(ids), _ptr(sec), _ptr(nsec), _ptr(poses)))

    def mailbox_ingest_prefetched(self):
        check(lib.te_pool_mailbox_ingest_prefetched(self._h))
        self._prefetched = None

    def mailbox_ingest_dev(self, n, dev_ids, dev_sec, dev_nsec, dev_poses):
        """the same for a message already in device memory (torch CUDA tensors: int32/uint32 ids and stamps, float64 [n][7] poses)"""
        check(lib.te_pool_mailbox_ingest_dev(self._h, int(n), _dev_ptr(dev_ids), _dev_ptr(dev_sec), _dev_ptr(dev_nsec), _dev_ptr(dev_poses)))

    def mailbox_tick(self, dt, t0_new, now, timeout, cls_new=0, want_added=False):
        """RosTargetManager::update(dt) (src/target_manager_ros.cpp:41-76); now = (sec, nsec).  Returns (erased ids, #added), or
        (erased ids, added ids) with want_added."""
        cap = int(lib.te_pool_mailbox_bound(self._h))
        buf = getattr(self, "_erase_buf", None)
        if buf is None or buf.size < cap:
            buf = self._erase_buf = np.empty(max(cap + cap // 4, 1), dtype=np.uint32)
        added = C.c_longlong(0)
        abuf = np.empty(max(cap, 1), dtype=np.uint32) if want_added else None
        n = check(lib.te_pool_mailbox_tick(self._h, float(dt), float(t0_new), int(cls_new), int(now[0]), int(now[1]), float(timeout), _ptr(buf), cap,
                                           _ptr(abuf), cap if want_added else 0, C.byref(added)))
        if want_added:
            return buf[:n].copy(), abuf[:int(added.value)].copy()
        return buf[:n].copy(), int(added.value)

    def mailbox_count(self):
        return int(lib.te_pool_mailbox_count(self._h))

    # -- the k earliest sphere intercepts over every target (te_pool_earliest_intersections) ------
    def earliest_intersections(self, t1, origin, radius, k):
        """sphere j = (t1[j], origin[j], radius[j]); t1 and radius broadcast to q = len(origin).  Returns (hits [q], ids [q][k],
        delta [q][k]) with the hits of each sphere by (delta, id) first and rows of id 0xFFFFFFFF / delta -1 after them."""
        origin = _np(origin, np.float64).reshape(-1, 3)
        q, k = origin.shape[0], int(k)
        t1 = _np(np.broadcast_to(t1, (q,)), np.float64)
        radius = _np(np.broadcast_to(radius, (q,)), np.float64)
        hits = np.zeros(q, dtype=np.int64)
        ids = np.zeros((q, max(k, 0)), dtype=np.uint32)
        delta = np.zeros((q, max(k, 0)))
        check(lib.te_pool_earliest_intersections(self._h, q, _ptr(t1), _ptr(origin), _ptr(radius), k, _ptr(ids), _ptr(delta), _ptr(hits)))
        return hits, ids, delta

    # -- the k nearest targets inside a sphere (te_pool_nearest_targets) ------
    def nearest_targets(self, t1, point, radius, k):
        """query j = (t1[j], point[j], radius[j]); t1 (None = current estimates) and radius broadcast to q = len(point).  Returns
        (count [q], ids [q][k], dist [q][k]) with the targets inside each sphere by (dist, id) first and rows of id 0xFFFFFFFF /
        dist -1 after them."""
        point = _np(point, np.float64).reshape(-1, 3)
        q, k = point.shape[0], int(k)
        t1 = _np(np.broadcast_to(t1, (q,)), np.float64) if t1 is not None else None
        radius = _np(np.broadcast_to(radius, (q,)), np.float64)
        count = np.zeros(q, dtype=np.int64)
        ids = np.zeros((q, max(k, 0)), dtype=np.uint32)
        dist = np.zeros((q, max(k, 0)))
        check(lib.te_pool_nearest_targets(self._h, q, _ptr(t1), _ptr(point), _ptr(radius), k, _ptr(ids), _ptr(dist), _ptr(count)))
        return count, ids, dist

    # -- gating: the k smallest Mahalanobis distances to a measured position (te_pool_gated_targets) --
    def gated_targets(self, t1, z, gate, k):
        """query j = (t1[j], z[j], gate[j]); t1 (None = current estimates and covariances) and gate broadcast to q = len(z).  Returns
        (count [q], ids [q][k], d2 [q][k]) with the targets inside each gate by (d2, id) first and rows of id 0xFFFFFFFF / d2 -1 after
        them."""
        z = _np(z, np.float64).reshape(-1, 3)
        q, k = z.shape[0], int(k)
        t1 = _np(np.broadcast_to(t1, (q,)), np.float64) if t1 is not None else None
        gate = _np(np.broadcast_to(gate, (q,)), np.float64)
        count = np.zeros(q, dtype=np.int64)
        ids = np.zeros((q, max(k, 0)), dtype=np.uint32)
        d2 = np.zeros((q, max(k, 0)))
        check(lib.te_pool_gated_targets(self._h, q, _ptr(t1), _ptr(z), _ptr(gate), k, _ptr(ids), _ptr(d2), _ptr(count)))
        return count, ids, d2

    # -- association of one frame of unlabelled detections (te_pool_associate and its three steps) --
    def associate(self, t1, det, gate, K, apply=False):
        """det [q][7] pose records stamped t1, gated on det[:, 0:3]; greedy assignment over each detection's K best candidates,
        apply=True updates the assigned targets at t1.  Returns (id [q], d2 [q], count [q]) (id 0xFFFFFFFF / d2 -1: unassigned)."""
        det = _np(det, np.float64).reshape(-1, 7)
        q = det.shape[0]
        ids = np.zeros(q, dtype=np.uint32)
        d2 = np.zeros(q)
        count = np.zeros(q, dtype=np.int64)
        check(lib.te_pool_associate(self._h, float(t1), q, _ptr(det), float(gate), int(K), 1 if apply else 0, _ptr(ids), _ptr(d2), _ptr(count)))
        return ids, d2, count

    def gated_candidates(self, t1, z, gate, K):
        """the candidate lists of positions z [q][3] at t1: (count [q], ids [q][K], d2 [q][K]) as gated_targets' with k = K, over
        the targets with t <= t1"""
        z = _np(z, np.float64).reshape(-1, 3)
        q, K = z.shape[0], int(K)
        count = np.zeros(q, dtype=np.int64)
        ids = np.zeros((q, max(K, 0)), dtype=np.uint32)
        d2 = np.zeros((q, max(K, 0)))
        check(lib.te_pool_gated_candidates(self._h, float(t1), q, _ptr(z), float(gate), K, _ptr(ids), _ptr(d2), _ptr(count)))
        return count, ids, d2

    def assign_greedy(self, ids, d2):
        """greedy assignment over candidate rows ids / d2 [q][K] (each row by (d2, id), then d2 -1), on this pool's device.  Returns
        (id [q], d2 [q])."""
        ids = _np(ids, np.uint32)
        d2 = _np(d2, np.float64)
        q, K = ids.shape
        id_out = np.zeros(q, dtype=np.uint32)
        d2_out = np.zeros(q)
        check(lib.te_assign_greedy(self._h, q, K, _ptr(ids), _ptr(d2), _ptr(id_out), _ptr(d2_out)))
        return id_out, d2_out

    def update_at(self, ids, t1, meas):
        """update(id, t1 - t, meas[k]) for every id (dt from each target's own t, on the device).  Returns #applied."""
        ids = _np(ids, np.uint32)
        meas = _np(meas, np.float64, (ids.size, 7))
        return check(lib.te_pool_update_at(self._h, ids.size, _ptr(ids), float(t1), _ptr(meas)))

    def assoc_stats(self):
        """of the last association call: {levels, everywhere, candidates, rounds}"""
        out = np.zeros(4, dtype=np.int64)
        check(lib.te_pool_assoc_stats(self._h, _ptr(out)))
        return dict(zip(("levels", "everywhere", "candidates", "rounds"), (int(v) for v in out)))


class IntersectionSolver:
    """Batched IntersectionSolver: n_streams independent reference solver objects (include/te_pool.h)."""

    def __init__(self, pool, n_streams=1, filters_length=250):
        self.pool = pool
        self._h = lib.te_isolver_create(pool._h, int(n_streams), int(filters_length))
        if not self._h:
            from ._lib import last_error
            raise TeError(last_error())

    def close(self):
        if getattr(self, "_h", None):
            lib.te_isolver_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def query_dense(self, dev_origin, dev_radius, pos_th, ang_th, dev_t1=None, dev_delta=None, dev_pose=None, dev_conv=None):
        """device-resident: one query per slot (torch CUDA tensors), asynchronous on the pool's stream"""
        check(lib.te_isolver_query_dense(self._h, _dev_ptr(dev_t1), _dev_ptr(dev_origin), _dev_ptr(dev_radius), float(pos_th), float(ang_th),
                                         _dev_ptr(dev_delta), _dev_ptr(dev_pose), _dev_ptr(dev_conv)))

    def query(self, ids, t1, origin, radius, pos_th=None, ang_th=None, stream=None, with_pose=True):
        ids = _np(ids, np.uint32)
        n = ids.size
        t1 = _np(np.broadcast_to(t1, (n,)), np.float64)
        origin = _np(np.broadcast_to(origin, (n, 3)), np.float64)
        radius = _np(np.broadcast_to(radius, (n,)), np.float64)
        pos_th = _np(np.broadcast_to(pos_th, (n,)), np.float64) if pos_th is not None else None
        ang_th = _np(np.broadcast_to(ang_th, (n,)), np.float64) if ang_th is not None else None
        stream = _np(stream, np.int32)
        delta = np.zeros(n)
        pose = np.zeros((n, 7)) if with_pose else None
        conv = np.zeros(n, dtype=np.uint8) if with_pose else None
        check(lib.te_isolver_query(self._h, n, _ptr(ids), _ptr(stream), _ptr(t1), _ptr(origin), _ptr(radius), _ptr(pos_th),
                                   _ptr(ang_th), _ptr(delta), _ptr(pose), _ptr(conv)))
        return delta, pose, conv
