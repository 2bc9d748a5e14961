"""ctypes binding of include/target_manager_c.h (the reference-facing C-ABI, lib/libtarget_c.so)."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
so_path = os.path.join(_HERE, "lib", "libtarget_c.so")
if not os.path.exists(so_path):
    raise ImportError("target_estimation_b200: %s is missing -- run __graft_entry__.build()" % so_path)
clib = C.CDLL(so_path)

_p, _u, _d, _ll, _i = C.c_void_p, C.c_uint, C.c_double, C.c_longlong, C.c_int
_SIG = {
    "target_manager_new": (_p, [C.c_char_p]),
    "target_manager_new_on_device": (_p, [C.c_char_p, _i]),
    "target_manager_init": (None, [_p, _u, _d, _p, _d]),
    "target_manager_update_meas": (None, [_p, _u, _d, _p]),
    "target_manager_update": (None, [_p, _u, _d]),
    "target_manager_get_est_pose": (C.c_bool, [_p, _u, _p]),
    "target_manager_get_est_twist": (C.c_bool, [_p, _u, _p]),
    "target_manager_get_est_acceleration": (C.c_bool, [_p, _u, _p]),
    "target_manager_get_n_measurements": (_i, [_p, _u]),
    "target_manager_log": (None, [_p]),
    "target_manager_delete": (None, [_p]),
    "target_manager_init_batch": (_ll, [_p, _ll, _p, _d, _p, _p]),
    "target_manager_update_batch": (_ll, [_p, _ll, _p, _d, _p, _p]),
    "target_manager_update_all": (None, [_p, _d]),
    "target_manager_update_dense": (_ll, [_p, _d, _p, _i, _p, _p]),
    "target_manager_update_dense_async": (_ll, [_p, _d, _p, _i, _p, _p]),
    "target_manager_update_dense_wait": (_i, [_p, _i]),
    "target_manager_get_dense_ids": (_ll, [_p, _p, _ll]),
    "target_manager_erase_batch": (_ll, [_p, _ll, _p]),
    "target_manager_erase": (C.c_bool, [_p, _u]),
    "target_manager_get_estimates_batch": (_i, [_p, _ll, _p, _p, _p, _p, _p, _p]),
    "target_manager_get_ids": (_ll, [_p, _p, _ll]),
    "target_manager_get_state": (_i, [_p, _u, _p, _p, _p]),
    "target_manager_flush": (None, [_p]),
    "target_manager_nearest": (_ll, [_p, _ll, _p, _p, _p, _ll, _p, _p, _p]),
    "target_manager_gated": (_ll, [_p, _ll, _p, _p, _p, _ll, _p, _p, _p]),
    "target_manager_associate": (_ll, [_p, _d, _ll, _p, _d, _i, _i, _p, _p, _p]),
    "target_manager_last_error": (C.c_char_p, []),
    "target_manager_watch": (None, [_p, _ll, _p, _ll]),
    "target_manager_log_samples": (_ll, [_p]),
    "target_manager_log_sample": (_i, [_p, _ll, _ll, _p, _p]),
    "target_manager_write_log": (_i, [_p, C.c_char_p]),
    "target_write_txt_file": (_i, [C.c_char_p, _p, _ll, _ll]),
    "target_manager_new_sharded": (_p, [C.c_char_p, _i, _p]),
    "target_manager_shards": (_i, [_p]),
    "target_manager_gather_estimates": (_ll, [_p, _p, _p, _ll, _i]),
    "target_manager_last_gather_ms": (_d, [_p]),
    "target_manager_gather_uses_nccl": (_i, [_p]),
    "target_tick_manager_new": (_p, [C.c_char_p, _i]),
    "target_tick_manager_new_sharded": (_p, [C.c_char_p, _i, _p]),
    "target_tick_manager_set_expiration": (None, [_p, _d]),
    "target_tick_manager_set_token": (None, [_p, C.c_char_p]),
    "target_tick_manager_set_publish": (None, [_p, _i]),
    "target_tick_manager_callback_frames": (None, [_p, _ll, _p, _p, _p, _p]),
    "target_tick_manager_callback_ids": (None, [_p, _ll, _p, _p, _p, _p]),
    "target_tick_manager_update": (_ll, [_p, _d, _u, _u, _p, _ll]),
    "target_tick_manager_published": (_ll, [_p, _p, _p, _ll]),
    "target_tick_manager_time": (_d, [_p]),
    "target_tick_manager_mailboxes": (_ll, [_p]),
    "target_bag_read_tf": (_ll, [C.c_char_p, C.c_char_p, _p, _ll]),
    "target_tick_manager_replay_bag": (_ll, [_p, C.c_char_p, C.c_char_p, _d, _ll, _p]),
    "target_isolver_new": (_p, [_p, _ll, _u]),
    "target_isolver_delete": (None, [_p]),
    "target_isolver_get_time": (_d, [_p, _u, _d, _p, _d]),
    "target_isolver_get_pose": (C.c_bool, [_p, _u, _d, _d, _d, _p, _d, _p]),
    "target_isolver_query_batch": (_ll, [_p, _ll, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "target_isolver_last_timing": (_i, [_p, _p]),
    "target_isolver_earliest": (_ll, [_p, _ll, _p, _p, _p, _ll, _p, _p, _p]),
}
for _n, (_r, _a) in _SIG.items():
    _f = getattr(clib, _n)
    _f.restype = _r
    _f.argtypes = _a


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class TargetManagerC:
    """Python view of one `target_manager_c*` handle; method names follow the C symbols."""

    def __init__(self, yaml_file, device=0):
        self.h = clib.target_manager_new_on_device(yaml_file.encode() if yaml_file else None, device)
        if not self.h:
            raise RuntimeError("target_manager_new failed: %s" % clib.target_manager_last_error().decode())

    def close(self):
        if getattr(self, "h", None):
            clib.target_manager_delete(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def init(self, id_, dt0, p0, t0):
        p0 = np.ascontiguousarray(p0, dtype=np.float64)
        clib.target_manager_init(self.h, id_, dt0, _ptr(p0), t0)

    def update_meas(self, id_, dt, meas):
        meas = np.ascontiguousarray(meas, dtype=np.float64)
        clib.target_manager_update_meas(self.h, id_, dt, _ptr(meas))

    def update(self, id_, dt):
        clib.target_manager_update(self.h, id_, dt)

    def _get(self, fn, id_, k, out=None):
        out = np.zeros(k) if out is None else out
        return bool(fn(self.h, id_, _ptr(out))), out

    def get_est_pose(self, id_, out=None): return self._get(clib.target_manager_get_est_pose, id_, 7, out)
    def get_est_twist(self, id_, out=None): return self._get(clib.target_manager_get_est_twist, id_, 6, out)
    def get_est_acceleration(self, id_, out=None): return self._get(clib.target_manager_get_est_acceleration, id_, 6, out)
    def get_n_measurements(self, id_): return int(clib.target_manager_get_n_measurements(self.h, id_))

    def init_batch(self, ids, dt0, p0, t0=None):
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        p0 = np.ascontiguousarray(p0, dtype=np.float64)
        t0 = np.ascontiguousarray(t0, dtype=np.float64) if t0 is not None else None
        return int(clib.target_manager_init_batch(self.h, ids.size, _ptr(ids), dt0, _ptr(p0), _ptr(t0)))

    def update_batch(self, ids, dt, meas=None, action=None):
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        meas = np.ascontiguousarray(meas, dtype=np.float64) if meas is not None else None
        action = np.ascontiguousarray(action, dtype=np.uint8) if action is not None else None
        return int(clib.target_manager_update_batch(self.h, ids.size, _ptr(ids), dt, _ptr(meas), _ptr(action)))

    def update_all(self, dt):
        clib.target_manager_update_all(self.h, dt)

    def update_dense(self, dt, meas, action=None, est_pos_out=None, pipelined=False):
        """record k = the k-th id of dense_ids(); meas [n][7] or [n][3]; the arrays must stay alive until the tick is done"""
        meas = np.ascontiguousarray(meas, dtype=np.float64)
        action = np.ascontiguousarray(action, dtype=np.uint8) if action is not None else None
        fn = clib.target_manager_update_dense_async if pipelined else clib.target_manager_update_dense
        n = int(fn(self.h, dt, _ptr(meas), meas.shape[1], _ptr(action), _ptr(est_pos_out)))
        if n < 0:
            raise RuntimeError(clib.target_manager_last_error().decode())
        self._dense_keep = (meas, action, est_pos_out)
        return n

    def update_dense_wait(self, lag=0):
        if clib.target_manager_update_dense_wait(self.h, lag) < 0:
            raise RuntimeError(clib.target_manager_last_error().decode())

    def dense_ids(self):
        n = int(clib.target_manager_get_dense_ids(self.h, None, 0))
        out = np.zeros(max(n, 1), dtype=np.uint32)
        clib.target_manager_get_dense_ids(self.h, _ptr(out), n)
        return out[:n]

    def erase(self, id_):
        return bool(clib.target_manager_erase(self.h, id_))

    def erase_batch(self, ids):
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        return int(clib.target_manager_erase_batch(self.h, ids.size, _ptr(ids)))

    def get_estimates_batch(self, ids, t1=None):
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        n = ids.size
        t1 = np.ascontiguousarray(np.broadcast_to(t1, (n,)), dtype=np.float64) if t1 is not None else None
        pose, twist, acc, found = np.zeros((n, 7)), np.zeros((n, 6)), np.zeros((n, 6)), np.zeros(n, dtype=np.uint8)
        rc = clib.target_manager_get_estimates_batch(self.h, n, _ptr(ids), _ptr(t1), _ptr(pose), _ptr(twist), _ptr(acc), _ptr(found))
        if rc < 0:
            raise RuntimeError(clib.target_manager_last_error().decode())
        return pose, twist, acc, found

    def ids(self):
        n = int(clib.target_manager_get_ids(self.h, None, 0))
        out = np.zeros(max(n, 1), dtype=np.uint32)
        clib.target_manager_get_ids(self.h, _ptr(out), n)
        return out[:n]

    def state(self, id_, n_max=18):
        x = np.zeros(n_max); P = np.zeros(n_max * n_max); t = C.c_double()
        n = int(clib.target_manager_get_state(self.h, id_, _ptr(x), _ptr(P), C.byref(t)))
        if n == 0:
            return None
        return {"x": x[:n].copy(), "P": P[: n * n].reshape(n, n).copy(), "t": t.value}

    # -- sampled logging (the reference's log() under LOGGER_ON + writeTxtFile dumps) ----------
    def watch(self, ids, max_samples=1 << 20):
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        self._watched = ids.copy()
        clib.target_manager_watch(self.h, ids.size, _ptr(ids) if ids.size else None, max_samples)

    def log(self):
        clib.target_manager_log(self.h)

    def log_samples(self):
        return int(clib.target_manager_log_samples(self.h))

    def log_sample(self, k, j):
        """sample k of watched id j -> dict(t, measured_pose, pose_internal, twist, acceleration, P) or None if the id did not exist"""
        row, P = np.zeros(26), np.zeros(18 * 18)
        n = int(clib.target_manager_log_sample(self.h, k, j, _ptr(row), _ptr(P)))
        if n < 0:
            raise IndexError((k, j))
        if n == 0:
            return None
        return {"t": row[0], "measured_pose": row[1:8].copy(), "pose_internal": row[8:14].copy(), "twist": row[14:20].copy(),
                "acceleration": row[20:26].copy(), "P": P[: n * n].reshape(n, n).copy()}

    def write_log(self, folder="/tmp/"):
        n = int(clib.target_manager_write_log(self.h, folder.encode()))
        if n < 0:
            raise RuntimeError(clib.target_manager_last_error().decode())
        return n

    def flush(self):
        clib.target_manager_flush(self.h)

    def nearest(self, t1, point, radius, k):
        """the k nearest targets inside a sphere: query j = (t1[j], point[j], radius[j]); t1 (None = current estimates) and radius
        broadcast to q = len(point).  Returns (count [q], ids [q][k], dist [q][k]): rows past min(k, count[j]) are id 0xFFFFFFFF and
        dist -1.  The pose of a returned target is get_estimates_batch(ids, t1)."""
        point = np.ascontiguousarray(point, dtype=np.float64).reshape(-1, 3)
        q, k = point.shape[0], int(k)
        t1 = np.ascontiguousarray(np.broadcast_to(t1, (q,)), dtype=np.float64) if t1 is not None else None
        radius = np.ascontiguousarray(np.broadcast_to(radius, (q,)), dtype=np.float64)
        count = np.zeros(q, dtype=np.int64)
        ids = np.zeros((q, max(k, 0)), dtype=np.uint32)
        dist = np.zeros((q, max(k, 0)))
        if int(clib.target_manager_nearest(self.h, q, _ptr(t1), _ptr(point), _ptr(radius), k, _ptr(ids), _ptr(dist), _ptr(count))) < 0:
            raise RuntimeError(clib.target_manager_last_error().decode())
        return count, ids, dist

    def gated(self, t1, z, gate, k):
        """gating: the k targets of smallest Mahalanobis d^2 to a measured position, query j = (t1[j], z[j], gate[j]); t1 (None =
        current estimates and covariances) and gate broadcast to q = len(z).  Returns (count [q], ids [q][k], d2 [q][k]): rows past
        min(k, count[j]) are id 0xFFFFFFFF and d2 -1.  The pose of a returned target is get_estimates_batch(ids, t1)."""
        z = np.ascontiguousarray(z, dtype=np.float64).reshape(-1, 3)
        q, k = z.shape[0], int(k)
        t1 = np.ascontiguousarray(np.broadcast_to(t1, (q,)), dtype=np.float64) if t1 is not None else None
        gate = np.ascontiguousarray(np.broadcast_to(gate, (q,)), dtype=np.float64)
        count = np.zeros(q, dtype=np.int64)
        ids = np.zeros((q, max(k, 0)), dtype=np.uint32)
        d2 = np.zeros((q, max(k, 0)))
        if int(clib.target_manager_gated(self.h, q, _ptr(t1), _ptr(z), _ptr(gate), k, _ptr(ids), _ptr(d2), _ptr(count))) < 0:
            raise RuntimeError(clib.target_manager_last_error().decode())
        return count, ids, d2

    def associate(self, t1, det, gate, K, apply=False):
        """one frame of unlabelled detections det [q][7] (pose records stamped t1, gated on det[:, 0:3]): each detection is assigned at
        most one target, greedily by (d2, id, j) over its K best candidates; apply=True updates every assigned target with its
        detection at t1.  Returns (id [q], d2 [q], count [q]): id 0xFFFFFFFF / d2 -1 for an unassigned detection, count = its
        candidates."""
        det = np.ascontiguousarray(det, dtype=np.float64).reshape(-1, 7)
        q = det.shape[0]
        ids = np.zeros(q, dtype=np.uint32)
        d2 = np.zeros(q)
        count = np.zeros(q, dtype=np.int64)
        if int(clib.target_manager_associate(self.h, float(t1), q, _ptr(det), float(gate), int(K), 1 if apply else 0, _ptr(ids), _ptr(d2),
                                             _ptr(count))) < 0:
            raise RuntimeError(clib.target_manager_last_error().decode())
        return ids, d2, count


class ShardedManagerC(TargetManagerC):
    """target_manager_new_sharded: one TargetManager per device behind the same handle type (owner(id) = id mod n_shards)"""

    def __init__(self, yaml_file, n_shards, devices=None):
        dev = np.ascontiguousarray(devices, dtype=np.int32) if devices is not None else None
        self.h = clib.target_manager_new_sharded(yaml_file.encode(), int(n_shards), _ptr(dev))
        if not self.h:
            raise RuntimeError("target_manager_new_sharded failed: %s" % clib.target_manager_last_error().decode())

    def shards(self):
        return int(clib.target_manager_shards(self.h))

    def gather_estimates(self, publisher=0, fetch=True):
        """the optional all-gather of [pose7 | twist6] records: (ids, records [n][13]) read back from the publisher's device, or
        the record count only (fetch=False: exchange between the devices, nothing comes to the host)"""
        n = int(clib.target_manager_gather_estimates(self.h, None, None, 0, publisher))
        if n < 0:
            raise RuntimeError(clib.target_manager_last_error().decode())
        if not fetch:
            return n
        ids = np.zeros(max(n, 1), dtype=np.uint32); rec = np.zeros((max(n, 1), 13))
        if int(clib.target_manager_gather_estimates(self.h, _ptr(ids), _ptr(rec), n, publisher)) < 0:
            raise RuntimeError(clib.target_manager_last_error().decode())
        return ids[:n], rec[:n]

    def last_gather_ms(self):
        return float(clib.target_manager_last_gather_ms(self.h))

    def gather_uses_nccl(self):
        return int(clib.target_manager_gather_uses_nccl(self.h)) == 1


# target_tf_record of include/target_manager_c.h
TF_RECORD_DTYPE = np.dtype([("rec_sec", np.uint32), ("rec_nsec", np.uint32), ("msg", np.uint32), ("seq", np.uint32), ("sec", np.uint32),
                            ("nsec", np.uint32), ("frame_id", "S64"), ("child_frame_id", "S64"), ("pose", np.float64, (7,))], align=True)


def read_bag_tf(path, topic="/tf"):
    """every transform of a rosbag v2.0 /tf recording, in record order (target_bag_read_tf)"""
    n = int(clib.target_bag_read_tf(path.encode(), topic.encode(), None, 0))
    if n < 0:
        raise RuntimeError(clib.target_manager_last_error().decode())
    out = np.zeros(max(n, 1), dtype=TF_RECORD_DTYPE)
    clib.target_bag_read_tf(path.encode(), topic.encode(), _ptr(out), n)
    return out[:n]


class TickManagerC(TargetManagerC):
    """RosTargetManager semantics without ROS (target_tick_manager_* of include/target_manager_c.h)."""

    def __init__(self, yaml_file, device=0):
        self.h = clib.target_tick_manager_new(yaml_file.encode(), device)
        if not self.h:
            raise RuntimeError("target_tick_manager_new failed: %s" % clib.target_manager_last_error().decode())

    def set_expiration(self, t):
        clib.target_tick_manager_set_expiration(self.h, float(t))

    def set_publish(self, on):
        clib.target_tick_manager_set_publish(self.h, 1 if on else 0)

    def set_token(self, s):
        clib.target_tick_manager_set_token(self.h, s.encode())

    def callback_ids(self, ids, sec, nsec, poses):
        ids = np.ascontiguousarray(ids, dtype=np.uint32); sec = np.ascontiguousarray(sec, dtype=np.uint32)
        nsec = np.ascontiguousarray(nsec, dtype=np.uint32); poses = np.ascontiguousarray(poses, dtype=np.float64)
        clib.target_tick_manager_callback_ids(self.h, ids.size, _ptr(ids), _ptr(sec), _ptr(nsec), _ptr(poses))

    def callback_frames(self, frames, sec, nsec, poses):
        arr = (C.c_char_p * len(frames))(*[f.encode() for f in frames])
        sec = np.ascontiguousarray(sec, dtype=np.uint32); nsec = np.ascontiguousarray(nsec, dtype=np.uint32)
        poses = np.ascontiguousarray(poses, dtype=np.float64)
        clib.target_tick_manager_callback_frames(self.h, len(frames), arr, _ptr(sec), _ptr(nsec), _ptr(poses))

    def tick(self, dt, now_sec, now_nsec, cap=1 << 20):
        out = np.zeros(cap, dtype=np.uint32)
        n = int(clib.target_tick_manager_update(self.h, dt, now_sec, now_nsec, _ptr(out), cap))
        if n < 0:
            raise RuntimeError(clib.target_manager_last_error().decode())
        return out[:n].copy()

    def published(self):
        n = int(clib.target_tick_manager_published(self.h, None, None, 0))
        ids = np.zeros(max(n, 1), dtype=np.uint32); poses = np.zeros((max(n, 1), 7))
        clib.target_tick_manager_published(self.h, _ptr(ids), _ptr(poses), n)
        return ids[:n], poses[:n]

    def time(self):
        return float(clib.target_tick_manager_time(self.h))

    def replay_bag(self, path, frequency, topic="/tf", extra_ticks=0):
        """the node's loop (update; spinOnce; sleep) on a recording; returns dict(ticks, messages, transforms, erased)"""
        st = np.zeros(4, dtype=np.int64)
        if int(clib.target_tick_manager_replay_bag(self.h, path.encode(), topic.encode(), float(frequency), int(extra_ticks), _ptr(st))) < 0:
            raise RuntimeError(clib.target_manager_last_error().decode())
        return dict(zip(("ticks", "messages", "transforms", "erased"), (int(v) for v in st)))

    def mailboxes(self):
        return int(clib.target_tick_manager_mailboxes(self.h))


class ShardedTickManagerC(TickManagerC, ShardedManagerC):
    """target_tick_manager_new_sharded: the node loop over n_shards devices (owner(id) = id mod n_shards), /tf messages routed to the
    owners on the devices; published() is shard-major (dense_ids() order)"""

    def __init__(self, yaml_file, n_shards, devices=None):
        dev = np.ascontiguousarray(devices, dtype=np.int32) if devices is not None else None
        self.h = clib.target_tick_manager_new_sharded(yaml_file.encode(), int(n_shards), _ptr(dev))
        if not self.h:
            raise RuntimeError("target_tick_manager_new_sharded failed: %s" % clib.target_manager_last_error().decode())


class IntersectionSolverC:
    """target_isolver_* on any manager handle above: n_streams reference IntersectionSolver objects (the per-id calls use stream 0)"""

    def __init__(self, mgr, n_streams=1, filters_length=250):
        self.mgr = mgr   # (the solver must go before its manager)
        self.h = clib.target_isolver_new(mgr.h, int(n_streams), int(filters_length))
        if not self.h:
            raise RuntimeError("target_isolver_new failed: %s" % clib.target_manager_last_error().decode())

    def close(self):
        if getattr(self, "h", None):
            clib.target_isolver_delete(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def time(self, id_, t1, origin, radius):
        origin = np.ascontiguousarray(origin, dtype=np.float64)
        return float(clib.target_isolver_get_time(self.h, int(id_), float(t1), _ptr(origin), float(radius)))

    def pose(self, id_, t1, pos_th, ang_th, origin, radius):
        """(converged, pose7)"""
        origin = np.ascontiguousarray(origin, dtype=np.float64)
        out = np.zeros(7)
        ok = bool(clib.target_isolver_get_pose(self.h, int(id_), float(t1), float(pos_th), float(ang_th), _ptr(origin), float(radius), _ptr(out)))
        return ok, out

    def query_batch(self, ids, t1, origin, radius, pos_th=None, ang_th=None, stream=None, with_pose=True):
        """(found, delta [n], pose [n][7] or None, converged [n] or None); t1 / origin / radius / thresholds broadcast to n"""
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        n = ids.size
        t1 = np.ascontiguousarray(np.broadcast_to(t1, (n,)), dtype=np.float64)
        origin = np.ascontiguousarray(np.broadcast_to(origin, (n, 3)), dtype=np.float64)
        radius = np.ascontiguousarray(np.broadcast_to(radius, (n,)), dtype=np.float64)
        pos_th = np.ascontiguousarray(np.broadcast_to(pos_th, (n,)), dtype=np.float64) if pos_th is not None else None
        ang_th = np.ascontiguousarray(np.broadcast_to(ang_th, (n,)), dtype=np.float64) if ang_th is not None else None
        stream = np.ascontiguousarray(stream, dtype=np.int32) if stream is not None else None
        delta = np.zeros(n)
        pose = np.zeros((n, 7)) if with_pose else None
        conv = np.zeros(n, dtype=np.uint8) if with_pose else None
        found = int(clib.target_isolver_query_batch(self.h, n, _ptr(ids), _ptr(stream), _ptr(t1), _ptr(origin), _ptr(radius), _ptr(pos_th),
                                                    _ptr(ang_th), _ptr(delta), _ptr(pose), _ptr(conv)))
        if found < 0:
            raise RuntimeError(clib.target_manager_last_error().decode())
        return found, delta, pose, conv

    def earliest(self, t1, origin, radius, k):
        """the k earliest sphere intercepts over every target: sphere j = (t1[j], origin[j], radius[j]); t1 and radius broadcast to
        q = len(origin).  Returns (hits [q], ids [q][k], delta [q][k]): rows past min(k, hits[j]) are id 0xFFFFFFFF and delta -1.
        The intercept pose of a returned target is the manager's get_estimates_batch(ids, t1 + delta)."""
        origin = np.ascontiguousarray(origin, dtype=np.float64).reshape(-1, 3)
        q, k = origin.shape[0], int(k)
        t1 = np.ascontiguousarray(np.broadcast_to(t1, (q,)), dtype=np.float64)
        radius = np.ascontiguousarray(np.broadcast_to(radius, (q,)), dtype=np.float64)
        hits = np.zeros(q, dtype=np.int64)
        ids = np.zeros((q, max(k, 0)), dtype=np.uint32)
        delta = np.zeros((q, max(k, 0)))
        if int(clib.target_isolver_earliest(self.h, q, _ptr(t1), _ptr(origin), _ptr(radius), k, _ptr(ids), _ptr(delta), _ptr(hits))) < 0:
            raise RuntimeError(clib.target_manager_last_error().decode())
        return hits, ids, delta

    def last_timing(self):
        """ms of the last query by phase: routing, moves, device, results into call order"""
        ms = np.zeros(4)
        if clib.target_isolver_last_timing(self.h, _ptr(ms)) < 0:
            raise RuntimeError(clib.target_manager_last_error().decode())
        return dict(zip(("route_ms", "move_ms", "device_ms", "writeback_ms"), (float(v) for v in ms)))
