"""-m gpu: the node loop over several devices (ShardedTickTargetManager, target_tick_manager_new_sharded of libtarget_c.so): /tf
messages routed to the owners on the devices (te_group_route_records), every shard's mailboxes, tick and expiry on its own device.

The reference runs one RosTargetManager (src/target_manager_ros.cpp:26-92): every observable of the sharded loop -- erased ids,
ids, mailboxes, clock, the broadcast poses, filter states, n_meas -- must equal that of the oracle's restatement, and bit for bit
that of a single TickTargetManager fed the same messages (same kernels, same record order per id).  Shards on one device (the
one-GPU form of these tests) exchange records by device copies; the two-GPU test covers the NCCL exchange."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests import bagfile, orc, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DT = 1.0 / 250.0


def _yaml(name):
    return os.path.join(ROOT, "models", "model_%s_params.yaml" % name)


def _devices(n_shards, distinct):
    import torch
    nd = torch.cuda.device_count()
    if distinct:
        if nd < n_shards:
            pytest.skip("needs %d GPUs" % n_shards)
        return list(range(n_shards))
    return [0] * n_shards


def _stamp(k, extra_ns=0):
    ns = 1000 * 10 ** 9 + k * 4000000 + extra_ns
    return ns // 10 ** 9, ns % 10 ** 9


def _d2h(dev_ptr, dtype, shape):
    """device memory of the current context -> a new host array (driver API: the package exposes no copy of raw pointers)"""
    out = np.empty(shape, dtype=dtype)
    if out.size:
        cu = C.CDLL("libcuda.so.1")
        assert cu.cuMemcpyDtoH_v2(out.ctypes.data_as(C.c_void_p), C.c_uint64(dev_ptr), C.c_size_t(out.nbytes)) == 0
    return out


# ---- the routing kernel ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("G", [3, 4])
def test_route_records_is_a_stable_partition(G):
    """every shard's routed arrays == numpy's stable partition of the message by id mod G, bit for bit (3 shards: the
    multiply-shift remainder; 4: the mask)"""
    import torch
    import target_estimation_b200 as te
    from target_estimation_b200._lib import check, lib
    torch.cuda.set_device(0)
    torch.cuda.synchronize()   # (the primary context is current on this thread for the driver-API read-back)
    pools = [te.TargetPool("angular_rates", device=0) for _ in range(G)]
    hp = (C.c_void_p * G)(*[p._h for p in pools])
    g = lib.te_group_create(G, (C.c_int * G)(*([0] * G)))
    assert g and lib.te_group_uses_nccl(g) == 0
    rng = np.random.default_rng(11)
    rep = rng.integers(0, 1000, 200).astype(np.uint32)
    rep[::7] = 42                                                       # one id many times in one message
    cases = {
        "empty": np.zeros(0, dtype=np.uint32),
        "fewer_than_G": np.array([7, 2], dtype=np.uint32),
        "one_owner": (np.arange(3000, dtype=np.uint32) * G + 1),
        "ragged": rng.integers(0, 2 ** 32, 10007, dtype=np.uint64).astype(np.uint32),
        "repeated": rep,
        "many_blocks": rng.integers(0, 2 ** 32, 300001, dtype=np.uint64).astype(np.uint32),
        "small_again": np.array([9, 10, 11, 12, 13], dtype=np.uint32),   # smaller than the buffers grown before it
    }
    for name, ids in cases.items():
        n = ids.size
        sec = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32)
        nsec = rng.integers(0, 10 ** 9, n).astype(np.uint32)
        poses = rng.normal(size=(n, 7))
        counts = np.zeros(G, dtype=np.int64)
        ptr = lambda a: a.ctypes.data_as(C.c_void_p)
        assert lib.te_group_route_records(g, hp, n, ptr(ids), ptr(sec), ptr(nsec), ptr(poses), ptr(counts)) == n, name
        for p in pools:
            check(lib.te_pool_sync(p._h))
        owner = ids % G
        for r in range(G):
            sel = owner == r
            m = C.c_longlong()
            pi, ps, pn, pp = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
            check(lib.te_group_routed(g, r, C.byref(m), C.byref(pi), C.byref(ps), C.byref(pn), C.byref(pp)))
            k = int(sel.sum())
            assert m.value == k == counts[r], (name, r)
            if k == 0:
                continue
            assert np.array_equal(_d2h(pi.value, np.uint32, k), ids[sel]), (name, r)
            assert np.array_equal(_d2h(ps.value, np.uint32, k), sec[sel]), (name, r)
            assert np.array_equal(_d2h(pn.value, np.uint32, k), nsec[sel]), (name, r)
            assert np.array_equal(_d2h(pp.value, np.float64, (k, 7)).view(np.uint64), poses[sel].view(np.uint64)), (name, r)
    lib.te_group_destroy(g)
    for p in pools:
        p.close()


# ---- semantics against the oracle's RosTargetManager ------------------------------------------------------------------------
@pytest.mark.parametrize("G", [1, 3])
@pytest.mark.parametrize("name", ["uniform_acceleration", "angular_velocities"])
def test_sharded_tick_semantics(name, G):
    """test_gpu_tick.py::test_tick_semantics on G shards of cuda:0: stale stamps, ids that fall silent, expire and come back,
    unrelated frames and the loop-breaking target_filt_<id> frames"""
    from target_estimation_b200.manager import ShardedTickManagerC
    path = _yaml(name)
    y = orc.load_yaml(path)
    N = y["Q"].shape[0]
    L = orc.lib()
    h = L.orc_tick_new(y["type"], orc.ptr(orc.colmajor(y["Q"])), N, orc.ptr(orc.colmajor(y["R"])), y["R"].shape[0], orc.ptr(orc.colmajor(y["P"])))
    mgr = ShardedTickManagerC(path, G, _devices(G, False))
    assert mgr.shards() == G
    timeout = 6 * DT
    L.orc_tick_set_expiration(h, timeout); mgr.set_expiration(timeout)
    rng = np.random.default_rng(5)
    n_ids = 40
    base = np.hstack([rng.normal(size=(n_ids, 3)), synth.rpy_to_quat(rng.uniform(-0.4, 0.4, (n_ids, 3)))])
    total_erased = 0
    for k in range(60):
        sec, nsec = _stamp(k)
        frames, stamps, poses = [], [], []
        for i in range(n_ids):
            silent = (i % 5 == 0 and k > 10 + i % 7) and not (i == 10 and k > 45)     # id 10 comes back after expiring
            if silent:
                continue
            stale = (i % 4 == 1 and k % 3 == 0 and k > 0)                              # resend with an old stamp -> predict only
            s = _stamp(k - 1) if stale else (sec, nsec)
            frames.append("target_%d" % i); stamps.append(s)
            poses.append(base[i] + np.r_[0.01 * k, -0.005 * k, 0.002 * k, 0, 0, 0, 0] + np.r_[rng.normal(0, 0.01, 3), 0, 0, 0, 0])
            if i == 20 and k % 9 == 4:       # the node's own output frame: ends the message for EVERY shard
                frames.append("target_filt_%d" % i); stamps.append((sec, nsec)); poses.append(base[i])
        if k % 6 == 5:                       # unrelated frames are ignored
            frames.insert(0, "camera_link"); stamps.insert(0, (sec, nsec)); poses.insert(0, base[0])
        stamps = np.array(stamps, dtype=np.uint32); poses = np.array(poses)
        L.orc_tick_callback(h, len(frames), "\n".join(frames).encode(), orc.ptr(np.ascontiguousarray(stamps)), orc.ptr(np.ascontiguousarray(poses)))
        mgr.callback_frames(frames, stamps[:, 0], stamps[:, 1], poses)
        er_ref = np.zeros(256, dtype=np.uint32)
        n_er = L.orc_tick_update(h, DT, sec, nsec, orc.ptr(er_ref), 256)
        er = mgr.tick(DT, sec, nsec)
        assert n_er == er.size and np.array_equal(er, er_ref[:n_er]), k          # one ascending list over all shards
        total_erased += n_er
        ref_ids = np.zeros(256, dtype=np.uint32)
        n_ref = L.orc_get_ids(h, orc.ptr(ref_ids), 256)
        assert np.array_equal(mgr.ids(), ref_ids[:n_ref]), k
        assert mgr.mailboxes() == L.orc_tick_mailboxes(h)
        assert mgr.time() == L.orc_tick_time(h)
        pub_ids, pub_poses = mgr.published()
        owner = pub_ids % G                                                       # shard-major, ascending inside a shard
        assert np.all(np.diff(owner) >= 0) and all(np.all(np.diff(pub_ids[owner == r].astype(np.int64)) > 0) for r in range(G))
        assert np.array_equal(np.sort(pub_ids), ref_ids[:n_ref]) and np.array_equal(pub_ids, mgr.dense_ids())
        for j in range(pub_ids.size):
            p = np.zeros(7)
            L.orc_get_est_pose(h, int(pub_ids[j]), orc.ptr(p))
            assert np.abs(pub_poses[j, :3] - p[:3]).max() <= 1e-9 * max(1.0, np.abs(p[:3]).max())
            assert min(np.abs(pub_poses[j, 3:] - p[3:]).max(), np.abs(pub_poses[j, 3:] + p[3:]).max()) <= 1e-9
    assert total_erased >= 6
    for i in mgr.ids()[::3]:
        x = np.zeros(N); P = np.zeros((N, N)); t = C.c_double(); nm = C.c_longlong()
        L.orc_get_state(h, int(i), orc.ptr(x), orc.ptr(P), C.byref(t), C.byref(nm), None)
        st = mgr.state(int(i))
        assert synth.compare_h2(st["x"][None], x[None]) <= 1.0 and synth.compare_h2(st["P"][None], P[None]) <= 1.0
        assert st["t"] == t.value and mgr.get_n_measurements(int(i)) == nm.value
    mgr.close()
    L.orc_manager_delete(h)


# ---- bit-for-bit equality with one TickTargetManager under churn -------------------------------------------------------------
def _churn_messages(n=20000, ticks=30, seed=3):
    """1 % of the speaking ids fall silent every tick (and expire 8 ticks later), as many fresh ids appear; every message is in
    shuffled order, and 50 ids are named twice -- the second record with the previous stamp (stale: the last record wins the
    stored pose, not the flag), so the arrival order per id matters"""
    rng = np.random.default_rng(seed)
    ids = (np.arange(n, dtype=np.int64) * 7 + 3)
    silent_at = np.full(n, 1 << 30, dtype=np.int64)
    next_id = int(ids.max()) + 1
    base = np.zeros((n * 2, 7)); base[:, :3] = rng.uniform(-5, 5, (n * 2, 3)); base[:, 3:] = synth.rpy_to_quat(rng.uniform(-0.4, 0.4, (n * 2, 3)))
    msgs = []
    for k in range(ticks):
        if k > 0:
            old = np.nonzero(silent_at > k)[0]
            quit_ = rng.choice(old, size=max(1, old.size // 100), replace=False)
            silent_at[quit_] = k
            fresh = np.arange(next_id, next_id + quit_.size, dtype=np.int64); next_id += quit_.size
            ids = np.concatenate([ids, fresh]); silent_at = np.concatenate([silent_at, np.full(fresh.size, 1 << 30, dtype=np.int64)])
        speak = np.nonzero(silent_at > k)[0]
        speak = speak[rng.permutation(speak.size)]
        twice = speak[:50]
        rows = np.concatenate([speak, twice])
        m_ids = ids[rows].astype(np.uint32)
        sec, nsec = _stamp(k)
        psec, pnsec = _stamp(k - 1)
        s = np.full(rows.size, sec, dtype=np.uint32); ns = np.full(rows.size, nsec, dtype=np.uint32)
        s[speak.size:] = psec; ns[speak.size:] = pnsec
        poses = base[rows % base.shape[0]].copy()
        poses[:, :3] += 0.01 * k + rng.normal(0, 0.01, (rows.size, 3))
        msgs.append((m_ids, s, ns, poses, (sec, nsec)))
    return msgs


def _equal_to_single(mgr, G, devices, msgs=None, check_every=10):
    from target_estimation_b200.manager import TickManagerC
    path = _yaml("angular_rates")
    one = TickManagerC(path, device=devices[0])
    for m in (mgr, one):
        m.set_expiration(8 * DT)
    msgs = msgs if msgs is not None else _churn_messages()
    n_erased = 0
    for k, (ids, s, ns, poses, now) in enumerate(msgs):
        mgr.callback_ids(ids, s, ns, poses)
        one.callback_ids(ids, s, ns, poses)
        ea, eb = mgr.tick(DT, *now), one.tick(DT, *now)
        assert np.array_equal(ea, eb), k
        n_erased += eb.size
        pa_ids, pa = mgr.published()
        pb_ids, pb = one.published()
        order = np.argsort(pa_ids, kind="stable")
        assert np.array_equal(pa_ids[order], pb_ids), k
        assert np.array_equal(pa[order].view(np.uint64), pb.view(np.uint64)), k      # bit for bit
        assert mgr.time() == one.time()
        if k % check_every == check_every - 1 or k == len(msgs) - 1:
            assert np.array_equal(mgr.ids(), one.ids()) and mgr.mailboxes() == one.mailboxes(), k
            for i in pb_ids[::97]:
                sa, sb = mgr.state(int(i)), one.state(int(i))
                assert np.array_equal(sa["x"].view(np.uint64), sb["x"].view(np.uint64)), (k, int(i))
                assert np.array_equal(sa["P"].view(np.uint64), sb["P"].view(np.uint64)), (k, int(i))
                assert sa["t"] == sb["t"] and mgr.get_n_measurements(int(i)) == one.get_n_measurements(int(i))
    assert n_erased > 500                         # ids did expire (about 0.6 % of the targets per tick after the first 9)
    one.close()


@pytest.mark.parametrize("G", [1, 3])
def test_churn_equals_single_manager(G):
    from target_estimation_b200.manager import ShardedTickManagerC
    dev = _devices(G, False)
    mgr = ShardedTickManagerC(_yaml("angular_rates"), G, dev)
    _equal_to_single(mgr, G, dev)
    assert not mgr.gather_uses_nccl()
    mgr.close()


def test_churn_forced_host_route_equals_single_manager(monkeypatch):
    """TE_SHARD_HOST_ROUTE (read when the manager is made) sends every message through the router threads of the host"""
    from target_estimation_b200.manager import ShardedTickManagerC
    monkeypatch.setenv("TE_SHARD_HOST_ROUTE", "1")
    dev = _devices(3, False)
    mgr = ShardedTickManagerC(_yaml("angular_rates"), 3, dev)
    _equal_to_single(mgr, 3, dev, msgs=_churn_messages(n=6000, ticks=20))
    mgr.close()


def test_churn_two_gpus_nccl():
    """two shards on two GPUs: the records travel between the devices as NCCL send / receive (skipped on a one-GPU box)"""
    from target_estimation_b200.manager import ShardedTickManagerC
    dev = _devices(2, True)
    mgr = ShardedTickManagerC(_yaml("angular_rates"), 2, dev)
    assert mgr.gather_uses_nccl()                 # the group the messages are routed over is a NCCL clique
    _equal_to_single(mgr, 2, dev)
    g_ids, g_rec = mgr.gather_estimates(publisher=1)   # the by-id surface of the handle keeps working
    assert np.array_equal(g_ids, mgr.dense_ids())
    mgr.close()


def test_foreign_model_ids_take_the_host_route(tmp_path):
    """ids created by hand under another model type keep host mailboxes: the C++ program checks the sharded loop against one
    TickTargetManager, bit for bit, on the host route"""
    lib = os.path.join(ROOT, "target_estimation_b200", "lib")
    exe = str(tmp_path / "sharded_tick_test")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "sharded_tick_test.cpp"),
                           "-o", exe, "-L", lib, "-ltarget_c", "-lte_pool", "-Wl,-rpath," + lib])
    r = subprocess.run([exe, os.path.join(ROOT, "models"), "3"], capture_output=True, text=True, timeout=600)
    print(r.stdout[-3000:], r.stderr[-2000:])
    assert r.returncode == 0 and r.stdout.strip().splitlines()[-1].startswith("ok:")


# ---- bag replay -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,freq,timeout", [("uniform_acceleration", 250.0, 1.5), ("angular_rates", 100.0, 0.6)])
def test_replay_bag_sharded_equals_single(tmp_path, name, freq, timeout):
    """target_tick_manager_replay_bag on a sharded handle (the fixture of test_gpu_replay.py) == the single-device replay"""
    from target_estimation_b200.manager import ShardedTickManagerC, TickManagerC
    rec = np.load(os.path.join(ROOT, "tests", "golden", "bag_tf_records.npz"))
    bag = str(tmp_path / "rebuilt.bag")
    bagfile.write_bag(bag, bagfile.messages_from_records(rec))
    mgr = ShardedTickManagerC(_yaml(name), 3, _devices(3, False))
    one = TickManagerC(_yaml(name))
    for m in (mgr, one):
        m.set_expiration(timeout)
    sa = mgr.replay_bag(bag, freq, extra_ticks=25)
    sb = one.replay_bag(bag, freq, extra_ticks=25)
    assert sa == sb and sa["messages"] == 572
    assert np.array_equal(mgr.ids(), one.ids()) and mgr.ids().size >= 1
    assert mgr.time() == one.time() and mgr.mailboxes() == one.mailboxes()
    pa_ids, pa = mgr.published()
    pb_ids, pb = one.published()
    order = np.argsort(pa_ids)
    assert np.array_equal(pa_ids[order], pb_ids) and np.array_equal(pa[order].view(np.uint64), pb.view(np.uint64))
    for i in one.ids():
        a, b = mgr.state(int(i)), one.state(int(i))
        assert np.array_equal(a["x"].view(np.uint64), b["x"].view(np.uint64)) and a["t"] == b["t"]
        assert mgr.get_n_measurements(int(i)) == one.get_n_measurements(int(i))
    mgr.close(); one.close()
