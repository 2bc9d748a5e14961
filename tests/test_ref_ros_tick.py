"""not gpu: the oracle's tick / mailbox / expiry restatement (oracle::TickTargetManager) against the REFERENCE's own
src/target_manager_ros.cpp (RosTargetManager: measurementCallBack, update(dt), Measurement mailboxes of
include/target_estimation/target_manager_ros.hpp), compiled unmodified into oracle/_ref/libref_manager.so against the roscpp /
tf / message stand-ins of oracle/eigen_standin (parameter map, a test-settable ros::Time::now(), a TransformBroadcaster that
logs).  Pins: first-sight init + update, sticky new-measurement flag, stale stamps (predict only), frames that stop the
callback loop, token filtering, expiry (erase decisions and order), the manager clock, and the poses the node broadcasts.
Skipped where neither /root/reference nor a prebuilt oracle/_ref exists."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests import orc, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "oracle", "_ref", "libref_manager.so")
DT = 1.0 / 250.0


def _lib():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s"])
    if not os.path.exists(LIB):
        pytest.skip("needs oracle/_ref/libref_manager.so, which `make -C oracle REF=<checkout of the original target_estimation project>` "
                    "builds from the original's own sources; they are not part of this repository, and this comparison has no stored form")
    orc.lib()
    L = C.CDLL(LIB, mode=C.RTLD_GLOBAL)
    if not hasattr(L, "refr_new"):
        pytest.skip("prebuilt oracle/_ref/libref_manager.so predates the ROS adapter")
    p, i, d, u, ll = C.c_void_p, C.c_int, C.c_double, C.c_uint, C.c_longlong
    L.refr_new.restype = p; L.refr_new.argtypes = [C.c_char_p, p, i, p, i, p, i]
    L.refr_set_expiration.argtypes = [p, d]
    L.refr_set_token.argtypes = [p, C.c_char_p]
    L.refr_callback.argtypes = [p, i, C.c_char_p, p, p, C.c_char_p]
    L.refr_update.restype = i; L.refr_update.argtypes = [p, d, u, u]
    L.refr_broadcast.argtypes = [i, C.c_char_p, C.c_char_p, p]
    L.refm_delete.argtypes = [p]
    L.refm_ids.restype = i; L.refm_ids.argtypes = [p, p, i]
    L.refm_state.restype = i; L.refm_state.argtypes = [p, u, p, p, p, p]
    L.refm_pose.restype = i; L.refm_pose.argtypes = [p, u, p]
    return L


def _model(name):
    y = orc.load_yaml(os.path.join(ROOT, "models", "model_%s_params.yaml" % name))
    return y["type"], y["Q"], y["R"], y["P"]


def _new_pair(L, name):
    mtype, Q, R, P = _model(name)
    Qc, Rc, Pc = orc.colmajor(Q), orc.colmajor(R), orc.colmajor(P)
    ref = L.refr_new(name.encode(), Qc.ctypes.data, Qc.size, Rc.ctypes.data, Rc.size, Pc.ctypes.data, Pc.size)
    assert ref
    O = orc.lib()
    h = O.orc_tick_new(mtype, orc.ptr(Qc), Q.shape[0], orc.ptr(Rc), R.shape[0], orc.ptr(Pc))
    return ref, h, Q.shape[0]


def _deliver(L, ref, h, frames, stamps, poses):
    fr = "\n".join(frames).encode()
    st = np.ascontiguousarray(stamps, dtype=np.uint32).reshape(-1, 2)
    ps = np.ascontiguousarray(poses, dtype=np.float64).reshape(-1, 7)
    L.refr_callback(ref, len(frames), fr, st.ctypes.data, ps.ctypes.data, b"world")
    orc.lib().orc_tick_callback(h, len(frames), fr, orc.ptr(st), orc.ptr(ps))


def _ref_ids(L, ref):
    out = np.zeros(4096, dtype=np.uint32)
    n = L.refm_ids(ref, out.ctypes.data, out.size)
    return out[:n].copy()


def _orc_ids(h):
    O = orc.lib()
    n = O.orc_num_targets(h)
    out = np.zeros(max(n, 1), dtype=np.uint32)
    O.orc_get_ids(h, orc.ptr(out), n)
    return out[:n]


def _compare_states(L, ref, h, ids, n):
    O = orc.lib()
    for id_ in ids:
        x, P = np.zeros(18), np.zeros(18 * 18)
        tt, nm = C.c_double(), C.c_longlong()
        nn = L.refm_state(ref, int(id_), x.ctypes.data, P.ctypes.data, C.byref(tt), C.byref(nm))
        assert nn == n
        xo, Po, prev = np.zeros(n), np.zeros((n, n)), np.zeros(3)
        to, no = C.c_double(), C.c_longlong()
        assert O.orc_get_state(h, int(id_), orc.ptr(xo), orc.ptr(Po), C.byref(to), C.byref(no), orc.ptr(prev))
        assert np.array_equal(x[:n], xo) and np.array_equal(P[:n * n].reshape(n, n).T, Po), id_
        assert tt.value == to.value and nm.value == no.value, id_


@pytest.mark.parametrize("name", ["uniform_velocity", "uniform_acceleration", "angular_rates", "angular_velocities"])
def test_tick_churn_matches_reference_ros_adapter(name):
    """per-tick /tf message for a changing subset of ids (new ids appear, 2 % go silent each tick, some stamps repeat), then
    update(dt) with a synthetic clock; expiry 40 ms.  Live ids, erase lists, every state and every broadcast pose must be
    bit-identical."""
    L = _lib(); O = orc.lib()
    ref, h, n = _new_pair(L, name)
    timeout = 0.04
    L.refr_set_expiration(ref, timeout); O.orc_tick_set_expiration(h, timeout)
    rng = np.random.default_rng(len(name) * 7 + 5)
    n0, ticks = 48, 70
    pool_ids = rng.choice(5000, size=n0 + ticks * 2, replace=False).astype(np.uint32)
    streams, _, _ = synth.make_streams(pool_ids.size, ticks, DT, accel=True, angular=True, seed=91)
    live = list(range(n0)); nxt = n0
    erased_total = 0
    erased = np.zeros(4096, dtype=np.uint32)
    for k in range(ticks):
        ns = 1000 * 10**9 + k * 4_000_000
        sec, nsec = ns // 10**9, ns % 10**9
        # who speaks this tick: live minus those that just went silent for good; two newcomers per tick
        gone = [j for j in live if rng.random() < 0.02]
        live = [j for j in live if j not in gone] + [nxt, nxt + 1]; nxt += 2
        speak = [j for j in live if rng.random() < 0.9]
        rng.shuffle(speak)
        frames, stamps, poses = [], [], []
        for j in speak:
            frames.append("target_%d" % pool_ids[j])
            stale = rng.random() < 0.1                      # a repeated (not newer) stamp: stored, but not a new measurement
            s_ns = ns - (8_000_000 if stale else 0)
            stamps.append((s_ns // 10**9, s_ns % 10**9)); poses.append(streams[k, j])
        frames.insert(len(frames) // 2, "camera_link"); stamps.insert(len(stamps) // 2, (sec, nsec)); poses.insert(len(poses) // 2, streams[k, 0])
        _deliver(L, ref, h, frames, stamps, poses)
        before = _ref_ids(L, ref)
        n_pub = L.refr_update(ref, DT, sec, nsec)
        n_er = O.orc_tick_update(h, DT, sec, nsec, orc.ptr(erased), erased.size)
        ids_ref, ids_orc = _ref_ids(L, ref), _orc_ids(h)
        assert np.array_equal(ids_ref, ids_orc), k
        assert n_pub == ids_ref.size
        # the reference's erase list of this tick = ids it had (or created) that are gone now; the oracle reports its own
        created = np.array(sorted(set(int(pool_ids[j]) for j in speak) - set(before.tolist())), dtype=np.uint32)
        had = np.union1d(before, created)
        assert np.array_equal(np.setdiff1d(had, ids_ref), np.sort(erased[:n_er])), k
        erased_total += n_er
        _compare_states(L, ref, h, ids_ref, n)
        # broadcast: one transform per live id in ascending order, child "<token>_filt_<id>", pose = getTargetPose, quaternion
        # normalised by tf
        child, parent, p7 = C.create_string_buffer(64), C.create_string_buffer(64), np.zeros(7)
        for i, id_ in enumerate(ids_ref):
            L.refr_broadcast(i, child, parent, p7.ctypes.data)
            assert child.value == b"target_filt_%d" % id_ and parent.value == b"world"
            po = np.zeros(7)
            assert O.orc_get_est_pose(h, int(id_), orc.ptr(po))
            q = po[3:]
            s = 1.0 / np.sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3])
            assert np.array_equal(p7[:3], po[:3]) and np.allclose(p7[3:], q * s, rtol=0, atol=4e-16), (k, id_)
    assert erased_total > 20 and O.orc_tick_time(h) == pytest.approx(ticks * DT, abs=1e-12)
    L.refm_delete(ref); O.orc_manager_delete(h)


def test_tick_mailbox_quirks_match_reference_ros_adapter():
    """the sticky flag (a silent target re-applies its last pose every tick), a frame with the token but no parsable
    '<x>_<id>' shape ends the message, frames without the token are skipped, a custom token, expiry exactly at the boundary
    (>=), and a stamp of 0 creating a mailbox but no target (it is not newer than the mailbox's initial stamp)."""
    L = _lib(); O = orc.lib()
    ref, h, n = _new_pair(L, "uniform_acceleration")
    for tok in (b"obj",):
        L.refr_set_token(ref, tok); O.orc_tick_set_token(h, tok)
    L.refr_set_expiration(ref, 0.5); O.orc_tick_set_expiration(h, 0.5)
    rng = np.random.default_rng(8)
    pose = lambda: np.concatenate([rng.normal(0, 1, 3), [0, 0, 0, 1.0]])
    erased = np.zeros(64, dtype=np.uint32)
    # tick 0: obj_5, a token-less frame (skipped), obj_7, "obj_a_b" (3 parts: stops the loop), obj_9 (never seen)
    _deliver(L, ref, h, ["obj_5", "base_link", "obj_7", "obj_a_b", "obj_9"], [(10, 0), (10, 0), (0, 0), (10, 0), (10, 0)], [pose() for _ in range(5)])
    for k in range(140):
        ns = 10 * 10**9 + k * 4_000_000
        if k == 20:   # 7 gets a real stamp once; 5 stays silent and re-applies its pose until it expires at 10.5 s exactly
            _deliver(L, ref, h, ["obj_7"], [(10, 80_000_000)], [pose()])
        if k == 30:   # an older stamp for 7: stored pose changes, flag cleared -> predict-only from here
            _deliver(L, ref, h, ["obj_7"], [(10, 40_000_000)], [pose()])
        n_pub = L.refr_update(ref, DT, ns // 10**9, ns % 10**9)
        n_er = O.orc_tick_update(h, DT, ns // 10**9, ns % 10**9, orc.ptr(erased), erased.size)
        ids_ref, ids_orc = _ref_ids(L, ref), _orc_ids(h)
        assert np.array_equal(ids_ref, ids_orc) and n_pub == ids_ref.size, k
        _compare_states(L, ref, h, ids_ref, n)
        if k == 0 or k == 19:   # stamp 0 is never "newer" than the mailbox's initial stamp 0: no measurement, no target yet
            assert ids_ref.tolist() == [5]
        if k == 20:
            assert ids_ref.tolist() == [5, 7]
        if k == 124:
            assert ids_ref.tolist() == [5, 7] and n_er == 0
        if k == 125:          # 10.5 s - 10.0 s >= 0.5 s
            assert n_er == 1 and erased[0] == 5 and ids_ref.tolist() == [7]
    L.refm_delete(ref); O.orc_manager_delete(h)
