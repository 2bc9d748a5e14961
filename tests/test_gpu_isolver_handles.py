"""-m gpu: IntersectionSolver on every manager handle (target_isolver_* of libtarget_c.so, IntersectionSolverC).

One solver stream = one reference IntersectionSolver object.  On a sharded handle the solver keeps one te_isolver per (shard, model
type) and moves a stream's state to the shard that queries it (te_isolver_move_streams).  The kernel and its inputs are the same as
on a plain handle and the moves are exact, so every result must equal the plain handle's bit for bit, and the oracle's
(orc_isolver_*) within the tolerances of test_gpu_estimates_isolver.py.  Shards share cuda:0 unless a test says otherwise."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests import orc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DT = 1.0 / 250.0
G_ACC = 9.81
INIT_POSE = [0, 0, 0, 0, 0, 0, 1]


def _yaml(name):
    return os.path.join(ROOT, "models", "model_%s_params.yaml" % name)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64 if np.asarray(a).dtype == np.float64 else np.uint8)


def _close(a, b, tol=1e-9):
    return np.abs(a - b).max() <= tol * max(1.0, np.abs(b).max())


def _qclose(a, b, tol=1e-9):
    return min(np.abs(a - b).max(), np.abs(a + b).max()) <= tol


class Falling:
    """targets thrown sideways and falling (the geometry of tests/cpp/api_test.cpp): pose(t) = p0 + v t - g t^2 / 2 on z, identity
    attitude; measurements carry a little noise"""

    def __init__(self, n, seed):
        rng = np.random.default_rng(seed)
        self.p0 = rng.uniform(-5, 5, (n, 3)); self.p0[:, 2] += 20.0
        self.v = rng.uniform(-2, 2, (n, 3))
        self.rng = rng

    def pos(self, t, rows=slice(None)):
        p = self.p0[rows] + self.v[rows] * t
        p[..., 2] -= 0.5 * G_ACC * t * t
        return p

    def meas(self, t, rows=slice(None)):
        p = self.pos(t, rows)
        q = np.zeros(p.shape[:-1] + (4,)); q[..., 3] = 1.0
        return np.concatenate([p + self.rng.normal(0, 0.002, p.shape), q], axis=-1)

    def sphere(self, t, rows=slice(None), ahead=0.3):
        """a sphere the target reaches about `ahead` seconds after t"""
        o = self.pos(t + ahead, rows)
        return o + self.rng.normal(0, 0.05, o.shape), self.rng.uniform(0.3, 1.0, o.shape[:-1])


def _managers(name, ids, fall, shards, devices=None, oracle=True):
    """a plain and a sharded handle (and the oracle) with the same targets, initialised at t = 0"""
    from target_estimation_b200.manager import ShardedManagerC, TargetManagerC
    plain = TargetManagerC(_yaml(name), device=devices[0] if devices else 0)
    sh = ShardedManagerC(_yaml(name), shards, devices if devices else [0] * shards)
    p0 = fall.meas(0.0)
    for m in (plain, sh):
        assert m.init_batch(ids, DT, p0) == ids.size
    ref = None
    if oracle:
        ref = orc.Manager(_yaml(name))
        for j, i in enumerate(ids):
            ref.init_default(int(i), DT, p0[j], 0.0)
    return plain, sh, ref


def _step(t, ids, fall, mgrs, ref):
    meas = fall.meas(t)
    for m in mgrs:
        assert m.update_batch(ids, DT, meas) == ids.size
    if ref is not None:
        ref.step_batch(ids, DT, meas, np.full(ids.size, 2, dtype=np.uint8))


# ---- 1. per-id calls: one solver object across the ids of every shard ----------------------------------------------------------
@pytest.mark.parametrize("G", [1, 3])
@pytest.mark.parametrize("name", ["uniform_acceleration", "angular_rates", "uniform_velocity"])
def test_per_id_calls_follow_the_solver(name, G):
    from target_estimation_b200.manager import IntersectionSolverC
    n = 9
    ids = np.arange(n, dtype=np.uint32) * 4 + 1        # owners 1 2 0 1 2 0 ... on three shards
    fall = Falling(n, seed=3)
    plain, sh, ref = _managers(name, ids, fall, G)
    L = 10
    s_sh, s_pl = IntersectionSolverC(sh, 1, L), IntersectionSolverC(plain, 1, L)
    rs = orc.lib().orc_isolver_new(ref.h, L)
    t, n_found = 0.0, 0
    for k in range(250):                               # settle the filters
        t += DT
        _step(t, ids, fall, (plain, sh), ref)
    for tick in range(45):
        t += DT
        _step(t, ids, fall, (plain, sh), ref)
        for j in range(n):
            i = int(ids[(j + tick) % n])
            o, r = fall.sphere(t, (j + tick) % n)
            o = np.ascontiguousarray(o)
            d_sh, d_pl = s_sh.time(i, t, o, float(r)), s_pl.time(i, t, o, float(r))
            c_sh, p_sh = s_sh.pose(i, t, 0.05, 0.1, o, float(r))
            c_pl, p_pl = s_pl.pose(i, t, 0.05, 0.1, o, float(r))
            assert _bits(np.float64(d_sh)) == _bits(np.float64(d_pl)) and np.array_equal(_bits(p_sh), _bits(p_pl)) and c_sh == c_pl, (tick, i)
            rt = orc.lib().orc_isolver_time(rs, i, t, orc.ptr(o), float(r))
            rp = np.zeros(7)
            rc = orc.lib().orc_isolver_pose(rs, i, t, 0.05, 0.1, orc.ptr(o), float(r), orc.ptr(rp))
            if rt < 0:
                assert d_sh == -1.0
            else:
                n_found += 1
                assert abs(d_sh - rt) <= 1e-9 * max(1.0, abs(rt)), (d_sh, rt)
            assert _close(p_sh[:3], rp[:3], 1e-8) and _qclose(p_sh[3:], rp[3:], 1e-8)
            assert c_sh == bool(rc)
    if name == "uniform_velocity":
        assert n_found == 0                            # zero t^4 coefficient: always -1 (SURVEY.md H9)
    else:
        assert n_found > 200
    orc.lib().orc_isolver_delete(rs)
    s_sh.close(); s_pl.close(); sh.close(); plain.close()


# ---- 2 / 7. batched queries, stream k, interleaved with update ticks -------------------------------------------------------------
def _batched(devices, n=20000, ticks=24, L=6, n_sample=256):
    from target_estimation_b200.manager import IntersectionSolverC
    ids = (np.arange(n, dtype=np.uint32) * 3 + 7)
    fall = Falling(n, seed=11)
    plain, sh, ref = _managers("uniform_acceleration", ids, fall, len(devices), devices)
    s_sh, s_pl = IntersectionSolverC(sh, n, L), IntersectionSolverC(plain, n, L)
    rng = np.random.default_rng(5)
    sample = np.sort(rng.choice(n, n_sample, replace=False))
    refs = [orc.lib().orc_isolver_new(ref.h, L) for _ in sample]
    stream = np.arange(n, dtype=np.int32)
    t, n_conv, n_hit = 0.0, 0, 0
    for k in range(100):
        t += DT
        _step(t, ids, fall, (plain, sh), ref)
    sph_o, sph_r = fall.sphere(t, ahead=0.35)          # one sphere per target for the whole run: the filters can converge
    for tick in range(ticks):
        t += DT
        _step(t, ids, fall, (plain, sh), ref)
        # on two ticks the queries of a stream name another target (mostly on another shard): the stream's state must follow
        rows = rng.permutation(n) if tick in (8, 9) else np.arange(n)
        q_ids = ids[rows]
        origin, radius = sph_o[rows], sph_r[rows]
        fa, da, pa, ca = s_sh.query_batch(q_ids, t, origin, radius, 0.5, 0.5, stream=stream)
        fb, db, pb, cb = s_pl.query_batch(q_ids, t, origin, radius, 0.5, 0.5, stream=stream)
        assert fa == fb == n
        assert np.array_equal(_bits(da), _bits(db)) and np.array_equal(_bits(pa), _bits(pb)) and np.array_equal(ca, cb), tick
        n_conv += int(ca.sum()); n_hit += int((da >= 0).sum())
        for j, s in enumerate(sample):
            rp = np.zeros(7)
            rc = orc.lib().orc_isolver_pose(refs[j], int(q_ids[s]), t, 0.5, 0.5, orc.ptr(np.ascontiguousarray(origin[s])), float(radius[s]), orc.ptr(rp))
            assert _close(pa[s, :3], rp[:3], 1e-8) and _qclose(pa[s, 3:], rp[3:], 1e-8) and bool(ca[s]) == bool(rc), (tick, int(s))
    assert n_hit > n * ticks // 2 and n_conv > 0
    for r in refs:
        orc.lib().orc_isolver_delete(r)
    s_sh.close(); s_pl.close(); sh.close(); plain.close()


def test_batched_queries_equal_plain_handle():
    _batched([0, 0, 0])


def test_batched_queries_two_gpus():
    """item 2 with the shards on two GPUs: the moves are peer copies (skipped on a one-GPU box)"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _batched([0, 1])


# ---- 3. call order inside one batch ------------------------------------------------------------------------------------------
def test_repeated_stream_in_a_batch_equals_calls_one_by_one():
    from target_estimation_b200.manager import IntersectionSolverC
    n = 6
    ids = np.arange(n, dtype=np.uint32) + 3            # 3 4 5 6 7 8: owners 0 1 2 0 1 2
    fall = Falling(n, seed=2)
    plain, sh, _ = _managers("uniform_acceleration", ids, fall, 3, oracle=False)
    b_sh, one_sh, b_pl = IntersectionSolverC(sh, 2, 5), IntersectionSolverC(sh, 2, 5), IntersectionSolverC(plain, 2, 5)
    t = 0.0
    for k in range(200):
        t += DT
        _step(t, ids, fall, (plain, sh), None)
    for tick in range(12):
        t += DT
        _step(t, ids, fall, (plain, sh), None)
        q = np.array([3, 4, 5, 6], dtype=np.uint32) if tick % 2 == 0 else np.array([8, 7, 6, 5], dtype=np.uint32)
        st = np.array([0, 0, 0, 1], dtype=np.int32)   # stream 0 three times, on three shards
        origin, radius = fall.sphere(t, q - 3)
        _, da, pa, ca = b_sh.query_batch(q, t, origin, radius, 0.05, 0.1, stream=st)
        _, db, pb, cb = b_pl.query_batch(q, t, origin, radius, 0.05, 0.1, stream=st)
        assert np.array_equal(_bits(da), _bits(db)) and np.array_equal(_bits(pa), _bits(pb)) and np.array_equal(ca, cb), tick
        for k in range(q.size):
            _, d1, p1, c1 = one_sh.query_batch(q[k:k + 1], t, origin[k:k + 1], radius[k:k + 1], 0.05, 0.1, stream=st[k:k + 1])
            assert _bits(d1[0]) == _bits(da[k]) and np.array_equal(_bits(p1[0]), _bits(pa[k])) and c1[0] == ca[k], (tick, k)
    b_sh.close(); one_sh.close(); b_pl.close(); sh.close(); plain.close()


# ---- 4. the state follows the stream ----------------------------------------------------------------------------------------------
def test_stream_alternating_between_shards():
    """one stream, ids 0 and 1 (two shards, the same trajectory) in turn for 300 calls: longer than the window, so it wraps"""
    from target_estimation_b200.manager import IntersectionSolverC
    ids = np.array([0, 1], dtype=np.uint32)
    fall = Falling(2, seed=4)
    fall.p0[1] = fall.p0[0]; fall.v[1] = fall.v[0]
    plain, sh, _ = _managers("uniform_acceleration", ids, fall, 3, oracle=False)
    s_sh, s_pl = IntersectionSolverC(sh, 1, 50), IntersectionSolverC(plain, 1, 50)
    t = 0.0
    for k in range(150):
        t += DT
        _step(t, ids, fall, (plain, sh), None)
    n_conv = 0
    o, r = fall.sphere(t, 0, ahead=0.6)
    o = np.ascontiguousarray(o)
    for call in range(300):
        if call % 3 == 0:
            t += DT
            _step(t, ids, fall, (plain, sh), None)
        i = call % 2
        ca, pa = s_sh.pose(int(ids[i]), t, 0.05, 0.1, o, float(r))
        cb, pb = s_pl.pose(int(ids[i]), t, 0.05, 0.1, o, float(r))
        assert ca == cb and np.array_equal(_bits(pa), _bits(pb)), call
        n_conv += ca
    assert 0 < n_conv < 300                            # the filters start unconverged and do converge
    s_sh.close(); s_pl.close(); sh.close(); plain.close()


class _IsolverState(C.Structure):   # te::IsolverState (csrc/te_kernels.cuh)
    _fields_ = [("n_streams", C.c_longlong), ("L", C.c_uint), ("prev_pose", C.c_void_p), ("pos_win", C.c_void_p), ("ang_win", C.c_void_p),
                ("pos_sum", C.c_void_p), ("ang_sum", C.c_void_p), ("idx", C.c_void_p), ("complete", C.c_void_p),
                ("pos_th_all", C.c_double), ("ang_th_all", C.c_double)]


class _Isolver(C.Structure):        # the head of struct te_isolver (csrc/te_pool_internal.cuh)
    _fields_ = [("pool", C.c_void_p), ("st", _IsolverState)]


def _state_arrays(h):
    st = _Isolver.from_address(h).st
    S, L = st.n_streams, st.L
    return [(st.prev_pose, np.float64, (S, 7)), (st.pos_win, np.float64, (L, S)), (st.ang_win, np.float64, (L, S)), (st.pos_sum, np.float64, S),
            (st.ang_sum, np.float64, S), (st.idx, np.uint32, S), (st.complete, np.uint8, S)]


def _read_state(h):
    cu = C.CDLL("libcuda.so.1")
    out = []
    for ptr, dt, shape in _state_arrays(h):
        a = np.empty(shape, dtype=dt)
        assert cu.cuMemcpyDtoH_v2(a.ctypes.data_as(C.c_void_p), C.c_uint64(ptr), C.c_size_t(a.nbytes)) == 0
        out.append(a)
    return out


def _write_state(h, arrays):
    cu = C.CDLL("libcuda.so.1")
    for (ptr, _, _), a in zip(_state_arrays(h), arrays):
        a = np.ascontiguousarray(a)
        assert cu.cuMemcpyHtoD_v2(C.c_uint64(ptr), a.ctypes.data_as(C.c_void_p), C.c_size_t(a.nbytes)) == 0


def _stream_cols(arrays, s):
    pp, pw, aw, ps, as_, ix, cp = arrays
    return [np.ascontiguousarray(a) for a in (pp[s], pw[:, s], aw[:, s], ps[s], as_[s], ix[s], cp[s])]


def test_move_streams_round_trip_is_byte_exact():
    """te_isolver_move_streams directly: random state on A, random stream subsets A -> B -> A; A's bytes stay as they were, B's
    listed streams equal A's, B's other streams keep their own bytes"""
    import torch
    import target_estimation_b200 as te
    from target_estimation_b200._lib import lib
    torch.cuda.set_device(0)
    torch.cuda.synchronize()   # (the primary context is current on this thread for the driver-API copies)
    S, L = 3000, 13
    pools = [te.TargetPool("uniform_acceleration", device=0) for _ in range(2)]
    sa, sb = te.IntersectionSolver(pools[0], S, L), te.IntersectionSolver(pools[1], S, L)
    rng = np.random.default_rng(17)

    def random_state():
        return [rng.normal(size=(S, 7)), rng.normal(size=(L, S)), rng.normal(size=(L, S)), rng.normal(size=S), rng.normal(size=S),
                rng.integers(0, L, S).astype(np.uint32), rng.integers(0, 2, S).astype(np.uint8)]

    _write_state(sa._h, random_state())
    _write_state(sb._h, random_state())
    a0 = _read_state(sa._h)
    for size in (1, 7, 1000, 2999, 3000, 50):          # the last is smaller than the staging grown before it
        sub = np.sort(rng.choice(S, size, replace=False)).astype(np.int32) if size % 2 else rng.choice(S, size, replace=False).astype(np.int32)
        b_before = _read_state(sb._h)
        assert lib.te_isolver_move_streams(sa._h, sb._h, sub.size, sub.ctypes.data_as(C.c_void_p)) == 0
        b1 = _read_state(sb._h)
        for x, y in zip(_stream_cols(b1, sub), _stream_cols(a0, sub)):
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), size
        rest = np.setdiff1d(np.arange(S), sub)
        for x, y in zip(_stream_cols(b1, rest), _stream_cols(b_before, rest)):
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), size
        assert lib.te_isolver_move_streams(sb._h, sa._h, sub.size, sub.ctypes.data_as(C.c_void_p)) == 0
        for x, y in zip(_read_state(sa._h), a0):
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), size
    bad = np.array([S], dtype=np.int32)
    assert lib.te_isolver_move_streams(sa._h, sb._h, 1, bad.ctypes.data_as(C.c_void_p)) == -1
    assert lib.te_isolver_move_streams(sa._h, sa._h, 1, bad.ctypes.data_as(C.c_void_p)) == -1
    sa.close(); sb.close()
    for p in pools:
        p.close()


# ---- 5. unknown and erased ids -----------------------------------------------------------------------------------------------
def test_unknown_and_erased_ids_leave_the_stream_untouched():
    from target_estimation_b200.manager import IntersectionSolverC
    n = 6
    ids = np.arange(n, dtype=np.uint32)
    fall = Falling(n, seed=8)
    plain, sh, _ = _managers("uniform_acceleration", ids, fall, 3, oracle=False)
    s_sh, s_pl = IntersectionSolverC(sh, 1, 8), IntersectionSolverC(plain, 1, 8)
    t = 0.0
    for k in range(200):
        t += DT
        _step(t, ids, fall, (plain, sh), None)
    o, r = fall.sphere(t, 0)
    o = np.ascontiguousarray(o)
    seq = [0, 1, 99, 2, 100, 3, 4, 5, 101, 1, 2]      # 99 .. 101 never existed
    for round_ in range(3):
        if round_ == 1:
            assert plain.erase_batch(np.array([1, 2], dtype=np.uint32)) == 2 and sh.erase_batch(np.array([1, 2], dtype=np.uint32)) == 2
        for i in seq:
            gone = i >= 99 or (round_ >= 1 and i in (1, 2))
            ca, pa = s_sh.pose(i, t, 0.05, 0.1, o, float(r))
            cb, pb = s_pl.pose(i, t, 0.05, 0.1, o, float(r))
            da, db = s_sh.time(i, t, o, float(r)), s_pl.time(i, t, o, float(r))
            assert ca == cb and np.array_equal(_bits(pa), _bits(pb)) and da == db, (round_, i)
            if gone:
                assert da == -1.0 and not ca and list(pa) == INIT_POSE
        found, d, _, _ = s_sh.query_batch(np.array(seq, dtype=np.uint32), t, o, r, with_pose=False)
        assert found == sum(1 for i in seq if not (i >= 99 or (round_ >= 1 and i in (1, 2))))
    s_sh.close(); s_pl.close(); sh.close(); plain.close()


# ---- 6. the sharded node loop ------------------------------------------------------------------------------------------------
def test_sharded_node_loop_equals_tick_manager():
    """the churn loop of test_gpu_sharded_tick.py on ShardedTickManagerC and TickManagerC, a batched query over the published ids
    every few ticks: bit for bit"""
    from target_estimation_b200.manager import IntersectionSolverC, ShardedTickManagerC, TickManagerC
    from tests.test_gpu_sharded_tick import _churn_messages
    path = _yaml("angular_rates")
    mgr, one = ShardedTickManagerC(path, 3, [0, 0, 0]), TickManagerC(path, device=0)
    for m in (mgr, one):
        m.set_expiration(8 * DT)
    msgs = _churn_messages(n=6000, ticks=24)
    S = 8000
    s_sh, s_one = IntersectionSolverC(mgr, S, 20), IntersectionSolverC(one, S, 20)
    rng = np.random.default_rng(1)
    for k, (ids, s, ns, poses, now) in enumerate(msgs):
        for m in (mgr, one):
            m.callback_ids(ids, s, ns, poses)
        assert np.array_equal(mgr.tick(DT, *now), one.tick(DT, *now))
        if k % 4 != 3:
            continue
        pub_ids, pub = one.published()
        n = pub_ids.size
        assert n <= S
        origin = pub[:, :3] + rng.normal(0, 0.3, (n, 3))
        radius = rng.uniform(0.2, 1.0, n)
        stream = rng.permutation(S)[:n].astype(np.int32)
        t1 = one.time()
        fa, da, pa, ca = s_sh.query_batch(pub_ids, t1, origin, radius, 0.5, 0.5, stream=stream)
        fb, db, pb, cb = s_one.query_batch(pub_ids, t1, origin, radius, 0.5, 0.5, stream=stream)
        assert fa == fb == n
        assert np.array_equal(_bits(da), _bits(db)) and np.array_equal(_bits(pa), _bits(pb)) and np.array_equal(ca, cb), k
    s_sh.close(); s_one.close(); mgr.close(); one.close()


# ---- 8. the C++ class on a ShardedTargetManager ------------------------------------------------------------------------------
def test_cpp_isolver_on_sharded_manager(tmp_path):
    lib = os.path.join(ROOT, "target_estimation_b200", "lib")
    exe = str(tmp_path / "isolver_sharded_test")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "isolver_sharded_test.cpp"),
                           "-o", exe, "-L", lib, "-ltarget_c", "-lte_pool", "-Wl,-rpath," + lib])
    r = subprocess.run([exe, os.path.join(ROOT, "models"), "3"], capture_output=True, text=True, timeout=600)
    print(r.stdout[-3000:], r.stderr[-2000:])
    assert r.returncode == 0 and r.stdout.strip().splitlines()[-1].startswith("ok:")
