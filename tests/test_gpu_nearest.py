"""-m gpu: the k nearest targets inside a sphere at a given time (TargetManagerC.nearest, target_manager_nearest,
te_pool_nearest_targets).

A target's position is pose7[0:3] of get_estimates_batch at t1, and its distance to the point is rounded operation by operation in
a fixed order, so every check compares bit for bit with the brute force a caller has without the query: get_estimates_batch over
every id, the distance in numpy in that order, and np.lexsort((ids, dist)) over dist <= radius."""
import os
import subprocess

import numpy as np
import pytest

from tests.test_gpu_isolver_handles import DT, Falling, _bits, _managers, _step, _yaml

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NO_ID = 0xFFFFFFFF
MODELS = ["uniform_acceleration", "angular_rates", "uniform_velocity", "angular_velocities"]


def distance(pos, point):
    """sqrt((dx^2 + dy^2) + dz^2) with d = pos - point, each numpy operation rounded on its own: the order the kernel uses"""
    d = pos - point
    return np.sqrt((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2])


def brute(mgr, t1, point, radius, k):
    """(count, ids [q][k], dist [q][k]) from get_estimates_batch over every id of the manager for every query"""
    ids = mgr.ids()
    point = np.asarray(point, dtype=np.float64).reshape(-1, 3)
    q = point.shape[0]
    radius = np.broadcast_to(np.asarray(radius, dtype=np.float64), (q,))
    when = [None] * q if t1 is None else list(np.broadcast_to(np.asarray(t1, dtype=np.float64), (q,)))
    count = np.zeros(q, dtype=np.int64)
    out_ids = np.full((q, k), NO_ID, dtype=np.uint32)
    out_d = np.full((q, k), -1.0)
    last, pos = (), None
    for j in range(q):
        key = None if when[j] is None else _bits(np.float64(when[j])).tobytes()
        if key != last:
            pose, _, _, found = mgr.get_estimates_batch(ids, when[j])
            assert found.all()
            last, pos = key, pose[:, :3]
        dist = distance(pos, point[j])
        inside = dist <= radius[j]
        count[j] = int(inside.sum())
        ii, dd = ids[inside], dist[inside]
        order = np.lexsort((ii, dd))[:k]
        out_ids[j, :order.size] = ii[order]
        out_d[j, :order.size] = dd[order]
    return count, out_ids, out_d


def same(a, b):
    """two (count, ids, dist) results, bit for bit"""
    return np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(_bits(a[2]), _bits(b[2]))


def falling(name, n, shards, ticks, seed=11, devices=None):
    ids = np.arange(n, dtype=np.uint32) * 3 + 5
    fall = Falling(n, seed=seed)
    plain, sh, _ = _managers(name, ids, fall, shards, devices, oracle=False)
    t = 0.0
    for _ in range(ticks):
        t += DT
        _step(t, ids, fall, (plain, sh), None)
    return ids, fall, plain, sh, t


def points(fall, t, q, rng, spread=0.3):
    """q points near the positions of random targets at t"""
    rows = rng.choice(fall.p0.shape[0], q, replace=False)
    return fall.pos(t, rows) + rng.normal(0, spread, (q, 3))


# ---- 1. every model, every shape = brute force, bit for bit ---------------------------------------------------------------------
@pytest.mark.parametrize("name", MODELS)
def test_nearest_equals_brute_force(name):
    n = 20000
    ids, fall, plain, sh, t = falling(name, n, 3, 100)
    rng = np.random.default_rng(2)
    for q in (1, 7, 64):
        point = points(fall, t, q, rng)
        t1 = t + 0.01 * (np.arange(q) // 3 % 3)                # runs of three equal t1; a run may come back to an earlier t1
        for when in (t1, None):
            for radius in (rng.uniform(1.0, 2.0, q), np.full(q, np.inf)):
                full = brute(plain, when, point, radius, n)
                count = full[0]
                if np.isinf(radius[0]):
                    assert np.all(count == n)
                else:
                    assert count.min() > 0 and count.max() < 0.2 * n, count
                for k in (0, 1, 100, 1000, int(count.max()) + 7):
                    ref = (count, full[1][:, :k], full[2][:, :k]) if k <= n else \
                        (count, np.pad(full[1], ((0, 0), (0, k - n)), constant_values=NO_ID), np.pad(full[2], ((0, 0), (0, k - n)), constant_values=-1.0))
                    assert same(plain.nearest(when, point, radius, k), ref), (q, when is None, radius[0], k)
                    assert same(sh.nearest(when, point, radius, k), ref), (q, when is None, radius[0], k)
    plain.close(); sh.close()


# ---- 2. ties: equal distance under different ids -------------------------------------------------------------------------------
@pytest.mark.parametrize("G", [1, 3])
def test_ties_come_out_by_ascending_id(G):
    """groups of three targets with identical histories: ids 3g + 5, 3g + 6, 3g + 7 (on three different shards when G = 3)"""
    from target_estimation_b200.manager import ShardedManagerC, TargetManagerC
    n_groups = 3000
    n = 3 * n_groups
    ids = np.arange(n, dtype=np.uint32) + 5
    fall = Falling(n_groups, seed=6)
    grp = np.arange(n) // 3
    mgr = TargetManagerC(_yaml("uniform_acceleration")) if G == 1 else ShardedManagerC(_yaml("uniform_acceleration"), G, [0] * G)
    assert mgr.init_batch(ids, DT, fall.meas(0.0)[grp]) == n
    t = 0.0
    for _ in range(100):
        t += DT
        assert mgr.update_batch(ids, DT, fall.meas(t)[grp]) == n
    rng = np.random.default_rng(4)
    point = points(fall, t, 5, rng)
    radius = rng.uniform(2.0, 2.5, 5)
    count, r_ids, r_d = brute(mgr, t, point, radius, n)
    assert np.all(count % 3 == 0) and count.min() >= 9
    for j in range(5):
        d = r_d[j, :count[j]]
        assert np.array_equal(d[0::3], d[1::3]) and np.array_equal(d[0::3], d[2::3])   # the groups do tie
    for k in (1, 2, 4, 5, 3 * int(count.min() // 6) + 1, 3 * int(count.min() // 3) - 1):
        got = mgr.nearest(t, point, radius, k)
        assert same(got, (count, r_ids[:, :k], r_d[:, :k])), k
        rows = min(k, int(count.min()))
        assert np.all(np.diff(got[1][:, :rows].astype(np.int64), axis=1)[np.diff(got[2][:, :rows], axis=1) == 0] > 0)
    mgr.close()


# ---- 3. the boundary counts as inside ------------------------------------------------------------------------------------------
def test_boundary_counts_as_inside():
    ids, fall, plain, sh, t = falling("uniform_velocity", 3000, 3, 50)
    pos = plain.get_estimates_batch(ids, t)[0][:, :3]
    rng = np.random.default_rng(17)
    rows = rng.choice(ids.size, 8, replace=False)
    point = pos[rows] + rng.normal(0, 0.5, (8, 3))
    radius = np.array([distance(pos[r:r + 1], point[j])[0] for j, r in enumerate(rows)])   # target rows[j] lies on sphere j
    below = np.nextafter(radius, 0.0)
    for m in (plain, sh):
        count, got_ids, got_d = m.nearest(t, point, radius, 3000)
        assert same((count, got_ids, got_d), brute(plain, t, point, radius, 3000))
        c_below, ids_below, d_below = m.nearest(t, point, below, 3000)
        assert same((c_below, ids_below, d_below), brute(plain, t, point, below, 3000))
        for j, r in enumerate(rows):
            at = np.nonzero(got_ids[j, :count[j]] == ids[r])[0]
            assert at.size == 1 and got_d[j, at[0]] == radius[j]                     # dist == radius: inside
            assert ids[r] not in ids_below[j, :c_below[j]] and c_below[j] < count[j]   # one ulp less: outside
    plain.close(); sh.close()


# ---- 4. every handle gives the same answer -------------------------------------------------------------------------------------
def _handles_after_churn(devices):
    """plain, sharded over `devices` and sharded with G = 1, fed the same records"""
    from target_estimation_b200.manager import ShardedManagerC, TargetManagerC
    path = _yaml("angular_rates")
    mgrs = (TargetManagerC(path, device=devices[0]), ShardedManagerC(path, len(devices), devices), ShardedManagerC(path, 1, [devices[0]]))
    plain, sh = mgrs[0], mgrs[1]
    ids = np.arange(30000, dtype=np.uint32) * 3 + 5
    fall = Falling(ids.size, seed=11)
    p0, t = fall.meas(0.0), 0.0
    for m in mgrs:
        assert m.init_batch(ids, DT, p0) == ids.size
    for _ in range(100):
        t += DT
        meas = fall.meas(t)
        for m in mgrs:
            assert m.update_batch(ids, DT, meas) == ids.size
    rng = np.random.default_rng(9)
    rows = np.arange(ids.size)                                # the trajectory (row of fall) of each id
    for rnd in range(3):                                      # churn: erase a few percent, add as many fresh ids, keep stepping
        gone = np.sort(rng.choice(ids, 900, replace=False))
        for m in mgrs:
            assert m.erase_batch(gone) == gone.size
        keep = ~np.isin(ids, gone)
        fresh = np.arange(900, dtype=np.uint32) * 3 + int(ids.max()) + 1
        p0 = fall.meas(t)[rows[~keep]]
        for m in mgrs:
            assert m.init_batch(fresh, DT, p0, t0=np.full(fresh.size, t)) == fresh.size
        rows = np.concatenate([rows[keep], rows[~keep]])
        ids = np.concatenate([ids[keep], fresh])
        order = np.argsort(ids)
        ids, rows = ids[order], rows[order]
        for _ in range(20):
            t += DT
            meas = fall.meas(t)[rows]
            for m in mgrs:
                assert m.update_batch(ids, DT, meas) == ids.size
    point = points(fall, t, 16, rng)
    for when in (t + 0.05, None):
        for radius in (rng.uniform(1.0, 2.0, 16), np.inf):
            ref = brute(plain, when, point, radius, 500)
            assert ref[0].min() > 0
            for m in mgrs:
                assert same(m.nearest(when, point, radius, 500), ref)
    assert same(sh.nearest(t, point, 1.5, 500), brute(sh, t, point, 1.5, 500))
    for m in mgrs:
        m.close()


def test_plain_and_sharded_handles_after_churn():
    _handles_after_churn([0, 0, 0])


def test_plain_and_sharded_handles_two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _handles_after_churn([0, 1])


def test_tick_and_sharded_tick_handles_after_churn():
    from target_estimation_b200.manager import ShardedTickManagerC, TickManagerC
    from tests.test_gpu_sharded_tick import _churn_messages
    path = _yaml("angular_velocities")
    mgr, one = ShardedTickManagerC(path, 3, [0, 0, 0]), TickManagerC(path, device=0)
    for m in (mgr, one):
        m.set_expiration(8 * DT)
    rng = np.random.default_rng(3)
    checked = 0
    for k, (ids, s, ns, poses, now) in enumerate(_churn_messages(n=20000, ticks=24)):
        for m in (mgr, one):
            m.callback_ids(ids, s, ns, poses)
        assert np.array_equal(mgr.tick(DT, *now), one.tick(DT, *now))
        if k % 6 != 5:
            continue
        pub_ids, pub = one.published()
        rows = rng.choice(pub_ids.size, 8, replace=False)
        point, radius = pub[rows, :3] + rng.normal(0, 0.05, (8, 3)), rng.uniform(0.3, 0.6, 8)
        for when in (one.time() + 0.05, None):
            ref = brute(one, when, point, radius, 300)
            assert ref[0].sum() > 0
            assert same(one.nearest(when, point, radius, 300), ref) and same(mgr.nearest(when, point, radius, 300), ref), k
            checked += 1
    assert checked == 8
    mgr.close(); one.close()


# ---- 5. mixed-model managers (C++) -----------------------------------------------------------------------------------------------
def test_cpp_nearest_on_mixed_model_managers(tmp_path):
    lib = os.path.join(ROOT, "target_estimation_b200", "lib")
    exe = str(tmp_path / "nearest_test")
    subprocess.check_call(["g++", "-O1", "-ffp-contract=off", "-std=c++17", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "nearest_test.cpp"), "-o", exe, "-L", lib, "-ltarget_c", "-lte_pool",
                           "-Wl,-rpath," + lib])
    r = subprocess.run([exe, os.path.join(ROOT, "models"), "3"], capture_output=True, text=True, timeout=600)
    print(r.stdout[-3000:], r.stderr[-2000:])
    assert r.returncode == 0 and r.stdout.strip().splitlines()[-1].startswith("ok:")


# ---- 6. read-only --------------------------------------------------------------------------------------------------------------
def test_query_leaves_filters_mailboxes_and_solver_streams_alone():
    """filter states and mailbox counts are byte-identical before and after a query, and a twin manager that is never queried ticks
    to the same published poses; a solver's pose queries around a query give what the same queries give on the twin"""
    from target_estimation_b200.manager import IntersectionSolverC, ShardedTickManagerC, TickManagerC
    from tests.test_gpu_sharded_tick import _churn_messages
    path = _yaml("uniform_acceleration")
    for make in (lambda: TickManagerC(path, device=0), lambda: ShardedTickManagerC(path, 3, [0, 0, 0])):
        a, b = make(), make()
        for m in (a, b):
            m.set_expiration(8 * DT)
        sa, sb = IntersectionSolverC(a, 300, 10), IntersectionSolverC(b, 300, 10)
        rng = np.random.default_rng(5)
        stream = np.arange(300, dtype=np.int32)
        for k, (ids, s, ns, poses, now) in enumerate(_churn_messages(n=6000, ticks=14)):
            for m in (a, b):
                m.callback_ids(ids, s, ns, poses)
            if k >= 2:
                live = a.ids()
                sample = live[::41]
                before = [a.state(int(i)) for i in sample]
                mail = a.mailboxes()
                q_ids = live[:300]
                o, r = rng.normal(0, 3, (300, 3)), rng.uniform(1.0, 3.0, 300)
                ra1, rb1 = (x.query_batch(q_ids, a.time(), o, r, 0.5, 0.5, stream=stream) for x in (sa, sb))
                point = a.published()[1][rng.choice(live.size, 4, replace=False), :3]
                assert a.nearest(a.time() + 0.02, point, 1.0, 50)[0].sum() > 0
                assert a.nearest(None, point, np.inf, 1000)[0].sum() == 4 * live.size
                after = [a.state(int(i)) for i in sample]
                for x, y in zip(before, after):
                    assert np.array_equal(_bits(x["x"]), _bits(y["x"])) and np.array_equal(_bits(x["P"]), _bits(y["P"])) and x["t"] == y["t"]
                assert a.mailboxes() == mail == b.mailboxes()
                ra2, rb2 = (x.query_batch(q_ids, a.time(), o, r, 0.5, 0.5, stream=stream) for x in (sa, sb))
                for ra, rb in ((ra1, rb1), (ra2, rb2)):
                    assert ra[0] == rb[0] and np.array_equal(_bits(ra[1]), _bits(rb[1])) and np.array_equal(_bits(ra[2]), _bits(rb[2]))
                    assert np.array_equal(ra[3], rb[3])
            assert np.array_equal(a.tick(DT, *now), b.tick(DT, *now))
            pa, pb = a.published(), b.published()
            assert np.array_equal(pa[0], pb[0]) and np.array_equal(_bits(pa[1]), _bits(pb[1]))
        sa.close(); sb.close(); a.close(); b.close()


def test_pool_entry_and_empty_manager():
    import target_estimation_b200 as te
    from target_estimation_b200.manager import TargetManagerC
    m = TargetManagerC(_yaml("angular_velocities"))
    count, got_ids, got_d = m.nearest(0.0, np.zeros((3, 3)), np.inf, 4)
    assert not count.any() and np.all(got_ids == NO_ID) and np.all(got_d == -1.0)
    ids = np.arange(1, 4, dtype=np.uint32)
    p0 = np.zeros((3, 7)); p0[:, 6] = 1.0
    assert m.init_batch(ids, DT, p0) == 3 and m.erase_batch(ids) == 3
    assert m.nearest(None, np.zeros((2, 3)), np.inf, 4)[0].sum() == 0
    m.close()
    # the pool entry point directly: equal to the pool's own read-back
    _, Q, R, P0 = te.load_model("angular_rates")[1:]
    fall = Falling(4000, seed=5)
    pool = te.TargetPool("angular_rates")
    pool.register_class(Q, R, P0)
    pids = np.arange(4000, dtype=np.uint32) * 2
    pool.add(pids, fall.meas(0.0))
    t = 0.0
    for _ in range(40):
        t += DT
        pool.step_ids(pids, DT, fall.meas(t))
    point = points(fall, t, 6, np.random.default_rng(8))
    for when in (t + 0.03, None):
        count, got_ids, got_d = pool.nearest_targets(when, point, 1.5, 50)
        pos = pool.read_estimates(pids, when)["pose"][:, :3]
        for j in range(6):
            dist = distance(pos, point[j])
            inside = dist <= 1.5
            order = np.lexsort((pids[inside], dist[inside]))[:50]
            assert count[j] == inside.sum() and count[j] > 0
            assert np.array_equal(got_ids[j, :order.size], pids[inside][order])
            assert np.array_equal(_bits(got_d[j, :order.size]), _bits(dist[inside][order]))
            assert np.all(got_ids[j, order.size:] == NO_ID) and np.all(got_d[j, order.size:] == -1.0)
    pool.close()


# ---- 7. scale: every target is a candidate ----------------------------------------------------------------------------------------
def test_one_mi_targets_sixteen_queries_radius_inf():
    from target_estimation_b200.manager import TargetManagerC
    n = 1 << 20
    ids = np.arange(n, dtype=np.uint32)
    fall = Falling(n, seed=31)
    m = TargetManagerC(_yaml("uniform_acceleration"))
    assert m.init_batch(ids, DT, fall.meas(0.0)) == n
    t = 0.0
    for _ in range(30):
        t += DT
        assert m.update_batch(ids, DT, fall.meas(t)) == n
    point = points(fall, t, 16, np.random.default_rng(5), spread=2.0)
    ref = brute(m, t + 0.05, point, np.inf, 10000)
    assert np.all(ref[0] == n)
    assert same(m.nearest(t + 0.05, point, np.inf, 10000), ref)
    m.close()
