"""-m gpu: the k earliest sphere intercepts over every target (IntersectionSolverC.earliest, target_isolver_earliest,
te_pool_earliest_intersections).

The reference answers "when does target id reach this sphere?" one id at a time; the sweep answers "which targets reach it first?"
over the whole manager.  Its delta is the time query's delta bit for bit, so every check compares it with the brute force: a
times-only query_batch over every id and sphere, ranked with np.lexsort((ids, delta)) over the hits (delta >= 0)."""
import os
import subprocess

import numpy as np
import pytest

from tests import orc
from tests.test_gpu_isolver_handles import DT, Falling, _bits, _managers, _step, _yaml

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NO_ID = 0xFFFFFFFF


def brute(solver, ids, t1, origin, radius, k):
    """(hits, ids [q][k], delta [q][k]) from query_batch over every id of `ids` for every sphere"""
    origin = np.asarray(origin, dtype=np.float64).reshape(-1, 3)
    q, n = origin.shape[0], ids.size
    t1 = np.broadcast_to(np.asarray(t1, dtype=np.float64), (q,))
    radius = np.broadcast_to(np.asarray(radius, dtype=np.float64), (q,))
    hits = np.zeros(q, dtype=np.int64)
    out_ids = np.full((q, k), NO_ID, dtype=np.uint32)
    out_d = np.full((q, k), -1.0)
    for j in range(q):
        _, d, _, _ = solver.query_batch(ids, t1[j], origin[j], radius[j], with_pose=False)
        hit = d >= 0
        hits[j] = int(hit.sum())
        ii, dd = ids[hit], d[hit]
        order = np.lexsort((ii, dd))[:k]
        out_ids[j, :order.size] = ii[order]
        out_d[j, :order.size] = dd[order]
    return hits, out_ids, out_d


def same(a, b):
    """two (hits, ids, delta) results, bit for bit"""
    return np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(_bits(a[2]), _bits(b[2]))


def spheres(fall, t, q, rng, radius=(1.0, 1.6)):
    """q spheres on the future paths of random targets (about 0.3 s ahead): a few percent of the targets reach each"""
    rows = rng.choice(fall.p0.shape[0], q, replace=False)
    o = fall.pos(t + 0.3, rows) + rng.normal(0, 0.1, (q, 3))
    return o, rng.uniform(radius[0], radius[1], q)


def falling(name, n, shards, ticks, seed=11, devices=None, oracle=False):
    ids = np.arange(n, dtype=np.uint32) * 3 + 5
    fall = Falling(n, seed=seed)
    plain, sh, ref = _managers(name, ids, fall, shards, devices, oracle=oracle)
    t = 0.0
    for _ in range(ticks):
        t += DT
        _step(t, ids, fall, (plain, sh), ref)
    return ids, fall, plain, sh, ref, t


# ---- 1. ranking = brute force, bit for bit -------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["uniform_acceleration", "angular_rates"])
def test_ranking_equals_brute_force(name):
    from target_estimation_b200.manager import IntersectionSolverC
    ids, fall, plain, sh, _, t = falling(name, 50000, 3, 250)
    s_pl, s_sh = IntersectionSolverC(plain, 1, 10), IntersectionSolverC(sh, 1, 10)
    rng = np.random.default_rng(2)
    for q in (1, 7, 64):
        origin, radius = spheres(fall, t, q, rng)
        t1 = np.full(q, t)
        if q == 7:
            t1[3:5] += 0.01                                   # several runs of equal t1 in one chunk
        ref_full = brute(s_pl, ids, t1, origin, radius, 65536)
        hits = ref_full[0]
        assert hits.min() > 0 and hits.max() < 0.2 * ids.size, hits
        for k in (0, 1, 100, 1000, int(hits.max()) + 7):
            ref = (hits, ref_full[1][:, :k], ref_full[2][:, :k])
            got = s_pl.earliest(t1, origin, radius, k)
            assert same(got, ref), (q, k)
            assert same(s_sh.earliest(t1, origin, radius, k), ref), (q, k)
    s_pl.close(); s_sh.close(); plain.close(); sh.close()


# ---- 2. ties: equal delta under different ids --------------------------------------------------------------------------------
@pytest.mark.parametrize("G", [1, 3])
def test_ties_come_out_by_ascending_id(G):
    """groups of three targets with identical histories: ids 3g + 5, 3g + 6, 3g + 7 (on three different shards when G = 3)"""
    from target_estimation_b200.manager import IntersectionSolverC, ShardedManagerC, TargetManagerC
    n_groups = 3000
    n = 3 * n_groups
    ids = np.arange(n, dtype=np.uint32) + 5
    fall = Falling(n_groups, seed=6)
    grp = np.arange(n) // 3
    mgr = TargetManagerC(_yaml("uniform_acceleration")) if G == 1 else ShardedManagerC(_yaml("uniform_acceleration"), G, [0] * G)
    assert mgr.init_batch(ids, DT, fall.meas(0.0)[grp]) == n
    t = 0.0
    for _ in range(200):
        t += DT
        assert mgr.update_batch(ids, DT, fall.meas(t)[grp]) == n
    s = IntersectionSolverC(mgr, 1, 10)
    rng = np.random.default_rng(4)
    origin, radius = spheres(fall, t, 5, rng, radius=(1.5, 2.0))
    hits, r_ids, r_d = brute(s, ids, t, origin, radius, 65536)
    assert np.all(hits % 3 == 0) and hits.min() >= 9
    for j in range(5):
        d = r_d[j, :hits[j]]
        assert np.array_equal(d[0::3], d[1::3]) and np.array_equal(d[0::3], d[2::3])   # the groups do tie
    for k in (1, 2, 4, 5, 3 * int(hits.min() // 6) + 1, 3 * int(hits.min() // 3) - 1):
        got = s.earliest(t, origin, radius, k)
        assert same(got, (hits, r_ids[:, :k], r_d[:, :k])), k
        rows = min(k, int(hits.min()))
        assert np.all(np.diff(got[1][:, :rows].astype(np.int64), axis=1)[np.diff(got[2][:, :rows], axis=1) == 0] > 0)
    s.close(); mgr.close()


# ---- 3. every handle gives the same answer -------------------------------------------------------------------------------------
def _plain_and_sharded(devices):
    from target_estimation_b200.manager import IntersectionSolverC
    ids, fall, plain, sh, _, t = falling("uniform_acceleration", 30000, len(devices), 150, devices=devices)
    rng = np.random.default_rng(9)
    rows = np.arange(ids.size)                                # the trajectory (row of fall) of each id
    for rnd in range(3):                                      # churn: erase a few percent, add as many fresh ids, keep stepping
        gone = np.sort(rng.choice(ids, 900, replace=False))
        for m in (plain, sh):
            assert m.erase_batch(gone) == gone.size
        keep = ~np.isin(ids, gone)
        fresh = np.arange(900, dtype=np.uint32) * 3 + int(ids.max()) + 1
        p0 = fall.meas(t)[rows[~keep]]
        for m in (plain, sh):
            assert m.init_batch(fresh, DT, p0, t0=np.full(fresh.size, t)) == fresh.size
        rows = np.concatenate([rows[keep], rows[~keep]])
        ids = np.concatenate([ids[keep], fresh])
        order = np.argsort(ids)
        ids, rows = ids[order], rows[order]
        for _ in range(40):
            t += DT
            meas = fall.meas(t)[rows]
            for m in (plain, sh):
                assert m.update_batch(ids, DT, meas) == ids.size
    s_pl, s_sh = IntersectionSolverC(plain, 1, 10), IntersectionSolverC(sh, 1, 10)
    origin, radius = spheres(fall, t, 16, rng)
    ref = brute(s_pl, ids, t, origin, radius, 500)
    assert ref[0].min() > 0
    a, b = s_pl.earliest(t, origin, radius, 500), s_sh.earliest(t, origin, radius, 500)
    assert same(a, ref) and same(b, ref)
    assert same(b, brute(s_sh, ids, t, origin, radius, 500))
    s_pl.close(); s_sh.close(); plain.close(); sh.close()


def test_plain_and_sharded_handles_after_churn():
    _plain_and_sharded([0, 0, 0])


def test_plain_and_sharded_handles_two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _plain_and_sharded([0, 1])


def test_tick_and_sharded_tick_handles_after_churn():
    from target_estimation_b200.manager import IntersectionSolverC, ShardedTickManagerC, TickManagerC
    from tests.test_gpu_sharded_tick import _churn_messages
    path = _yaml("angular_rates")
    mgr, one = ShardedTickManagerC(path, 3, [0, 0, 0]), TickManagerC(path, device=0)
    for m in (mgr, one):
        m.set_expiration(8 * DT)
    s_sh, s_one = IntersectionSolverC(mgr, 1, 10), IntersectionSolverC(one, 1, 10)
    rng = np.random.default_rng(3)
    n_hits = 0
    for k, (ids, s, ns, poses, now) in enumerate(_churn_messages(n=20000, ticks=24)):
        for m in (mgr, one):
            m.callback_ids(ids, s, ns, poses)
        assert np.array_equal(mgr.tick(DT, *now), one.tick(DT, *now))
        if k % 6 != 5:
            continue
        pub_ids, pub = one.published()
        rows = rng.choice(pub_ids.size, 8, replace=False)
        origin, radius = pub[rows, :3] + rng.normal(0, 0.2, (8, 3)), rng.uniform(0.2, 0.6, 8)
        t1 = one.time()
        ref = brute(s_one, one.ids(), t1, origin, radius, 300)
        a, b = s_one.earliest(t1, origin, radius, 300), s_sh.earliest(t1, origin, radius, 300)
        assert same(a, ref) and same(b, ref), k
        n_hits += int(ref[0].sum())
    assert n_hits > 0
    s_sh.close(); s_one.close(); mgr.close(); one.close()


# ---- 4. mixed-model managers (C++) -----------------------------------------------------------------------------------------------
def test_cpp_sweep_on_mixed_model_managers(tmp_path):
    lib = os.path.join(ROOT, "target_estimation_b200", "lib")
    exe = str(tmp_path / "sweep_test")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "sweep_test.cpp"),
                           "-o", exe, "-L", lib, "-ltarget_c", "-lte_pool", "-Wl,-rpath," + lib])
    r = subprocess.run([exe, os.path.join(ROOT, "models"), "3"], capture_output=True, text=True, timeout=600)
    print(r.stdout[-3000:], r.stderr[-2000:])
    assert r.returncode == 0 and r.stdout.strip().splitlines()[-1].startswith("ok:")


# ---- 5. unit checks ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["uniform_velocity", "angular_velocities"])
def test_no_acceleration_never_hits(name):
    from target_estimation_b200.manager import IntersectionSolverC
    ids, fall, plain, sh, _, t = falling(name, 2000, 3, 50)
    for m in (plain, sh):
        s = IntersectionSolverC(m, 1, 10)
        origin, radius = spheres(fall, t, 4, np.random.default_rng(1), radius=(3.0, 4.0))
        hits, got_ids, got_d = s.earliest(t, origin, radius, 10)
        assert not hits.any() and np.all(got_ids == NO_ID) and np.all(got_d == -1.0)
        assert brute(s, ids, t, origin, radius, 1)[0].sum() == 0
        s.close()
    plain.close(); sh.close()


def test_empty_manager_and_pool_entry():
    import target_estimation_b200 as te
    from target_estimation_b200.manager import IntersectionSolverC, TargetManagerC
    m = TargetManagerC(_yaml("uniform_acceleration"))
    s = IntersectionSolverC(m, 1, 10)
    hits, got_ids, got_d = s.earliest(0.0, np.zeros((3, 3)), 1.0, 4)
    assert not hits.any() and np.all(got_ids == NO_ID) and np.all(got_d == -1.0)
    ids = np.arange(1, 4, dtype=np.uint32)
    p0 = np.zeros((3, 7)); p0[:, 6] = 1.0
    assert m.init_batch(ids, DT, p0) == 3 and m.erase_batch(ids) == 3
    assert s.earliest(0.0, np.zeros((2, 3)), 1.0, 4)[0].sum() == 0
    s.close(); m.close()
    # the pool entry point directly: equal to the pool's own batched time query
    _, Q, R, P0 = te.load_model("uniform_acceleration")[1:]
    fall = Falling(4000, seed=5)
    pool = te.TargetPool("uniform_acceleration")
    pool.register_class(Q, R, P0)
    pids = np.arange(4000, dtype=np.uint32) * 2
    pool.add(pids, fall.meas(0.0))
    t = 0.0
    for _ in range(60):
        t += DT
        pool.step_ids(pids, DT, fall.meas(t))
    solver = te.IntersectionSolver(pool, 1, 10)
    origin, radius = spheres(fall, t, 6, np.random.default_rng(8))
    hits, got_ids, got_d = pool.earliest_intersections(t, origin, radius, 50)
    for j in range(6):
        d, _, _ = solver.query(pids, t, origin[j], radius[j], with_pose=False)
        hit = d >= 0
        order = np.lexsort((pids[hit], d[hit]))[:50]
        assert hits[j] == hit.sum() and hits[j] > 0
        assert np.array_equal(got_ids[j, :order.size], pids[hit][order]) and np.array_equal(_bits(got_d[j, :order.size]), _bits(d[hit][order]))
        assert np.all(got_ids[j, order.size:] == NO_ID) and np.all(got_d[j, order.size:] == -1.0)
    solver.close(); pool.close()


def test_hits_match_the_oracle_and_lie_on_the_sphere():
    from target_estimation_b200.manager import IntersectionSolverC
    ids, fall, plain, sh, ref, t = falling("uniform_acceleration", 2000, 3, 200, oracle=True)
    rng = np.random.default_rng(12)
    origin, radius = spheres(fall, t, 8, rng, radius=(2.0, 3.0))
    rs = orc.lib().orc_isolver_new(ref.h, 10)
    n_checked = 0
    for m in (plain, sh):
        s = IntersectionSolverC(m, 1, 10)
        hits, got_ids, got_d = s.earliest(t, origin, radius, 256)
        for j in range(8):
            rows = min(256, int(hits[j]))
            sel = got_ids[j, :rows]
            d = got_d[j, :rows]
            pose, _, _, found = m.get_estimates_batch(sel, t + d)
            assert found.all()
            dist = np.linalg.norm(pose[:, :3] - origin[j], axis=1)
            assert np.all(np.abs(dist - radius[j]) <= 1e-6 * radius[j]), j
            for i, dj in zip(sel[:32], d[:32]):
                rt = orc.lib().orc_isolver_time(rs, int(i), t, orc.ptr(np.ascontiguousarray(origin[j])), float(radius[j]))
                assert abs(dj - rt) <= 1e-9 * max(1.0, abs(rt)), (j, int(i), dj, rt)
                n_checked += 1
        s.close()
    assert n_checked >= 256
    orc.lib().orc_isolver_delete(rs)
    plain.close(); sh.close()


def test_solver_streams_are_untouched():
    from target_estimation_b200.manager import IntersectionSolverC
    ids, fall, plain, sh, _, t = falling("uniform_acceleration", 3000, 3, 150)
    rng = np.random.default_rng(21)
    origin, radius = spheres(fall, t, 4, rng)
    q_ids = ids[:500]
    q_o, q_r = fall.sphere(t, slice(0, 500))
    for m in (plain, sh):
        a, b = IntersectionSolverC(m, 500, 10), IntersectionSolverC(m, 500, 10)
        stream = np.arange(500, dtype=np.int32)
        for step in range(3):
            ra = a.query_batch(q_ids, t, q_o, q_r, 0.5, 0.5, stream=stream)
            if step == 1:
                assert a.earliest(t, origin, radius, 100)[0].sum() > 0
            rb = b.query_batch(q_ids, t, q_o, q_r, 0.5, 0.5, stream=stream)
            assert ra[0] == rb[0] and np.array_equal(_bits(ra[1]), _bits(rb[1])) and np.array_equal(_bits(ra[2]), _bits(rb[2]))
            assert np.array_equal(ra[3], rb[3]), step
        a.close(); b.close()
    plain.close(); sh.close()


# ---- 6. scale ---------------------------------------------------------------------------------------------------------------
def test_one_mi_targets_sixteen_spheres():
    from target_estimation_b200.manager import IntersectionSolverC, TargetManagerC
    n = 1 << 20
    ids = np.arange(n, dtype=np.uint32)
    fall = Falling(n, seed=31)
    m = TargetManagerC(_yaml("uniform_acceleration"))
    assert m.init_batch(ids, DT, fall.meas(0.0)) == n
    t = 0.0
    for _ in range(30):
        t += DT
        assert m.update_batch(ids, DT, fall.meas(t)) == n
    s = IntersectionSolverC(m, 1, 10)
    origin, radius = spheres(fall, t, 16, np.random.default_rng(5))
    ref = brute(s, ids, t, origin, radius, 1000)
    assert ref[0].min() > 1000
    assert same(s.earliest(t, origin, radius, 1000), ref)
    s.close(); m.close()
