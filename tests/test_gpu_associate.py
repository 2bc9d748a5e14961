"""-m gpu: association of one frame of unlabelled detections (te_pool_associate, te_pool_gated_candidates, te_assign_greedy,
te_pool_update_at, TargetManagerC.associate).

The candidate rows must be gatedTargets' rows bit for bit (the gating contract of include/te_pool.h, restated in numpy by
tests/test_gpu_gate.py), the assignment must be the greedy on the edges sorted by (d2, id, j) -- restated below as a plain
sequential loop -- and an applied frame must leave every target as te_pool_step_ids with dt = t1 - t would."""
import numpy as np
import pytest

from tests.test_gpu_gate import CHI2, MODELS, NO_ID, _bits, brute_pool, dense_classes, dense_pool, dense_yaml, near, same
from tests.test_gpu_isolver_handles import DT, Falling

pytestmark = pytest.mark.gpu


def greedy(ids, d2):
    """the contract's assignment over candidate rows ids / d2 [q][K] (d2 -1 = no row): edges visited by (d2, id, j)"""
    q, K = ids.shape
    j = np.repeat(np.arange(q), K)
    ii, dd = ids.ravel(), d2.ravel()
    ok = dd >= 0
    j, ii, dd = j[ok], ii[ok], dd[ok]
    order = np.lexsort((j, ii, dd))
    out_id = np.full(q, NO_ID, dtype=np.uint32)
    out_d2 = np.full(q, -1.0)
    taken = set()
    for e in order:
        if out_id[j[e]] != NO_ID or ii[e] in taken:
            continue
        out_id[j[e]], out_d2[j[e]] = ii[e], dd[e]
        taken.add(ii[e])
    return out_id, out_d2


def same_assignment(got, ref):
    return np.array_equal(got[0], ref[0]) and np.array_equal(_bits(got[1]), _bits(ref[1]))


def frame(pool, ids, t, q, rng, clutter=0.1, sigma=0.003):
    """q detections near targets, a tenth of them clutter around the scene, as pose records"""
    n_near = q - int(clutter * q)
    z = near(pool, ids, t, n_near, rng, sigma) if n_near else np.zeros((0, 3))
    lo, hi = z.min(axis=0) if n_near else np.zeros(3), z.max(axis=0) if n_near else np.ones(3)
    z = np.concatenate([z, rng.uniform(lo - 1, hi + 1, (q - n_near, 3))])[rng.permutation(q)]
    det = np.zeros((q, 7))
    det[:, :3] = z
    det[:, 6] = 1.0
    return det


def check_frame(pool, name, cls, Q, R, t1, det, gate, K):
    """candidates = gatedTargets(k = K) bit for bit and the assignment = the greedy restatement; returns the assignment"""
    ref = pool.gated_targets(t1, det[:, :3], gate, K)
    cand = pool.gated_candidates(t1, det[:, :3], gate, K)
    assert same(cand, ref)
    got = pool.associate(t1, det, gate, K)
    assert np.array_equal(got[2], ref[0])
    assert same_assignment(got, greedy(ref[1], ref[2]))
    assert same_assignment(pool.assign_greedy(ref[1], ref[2]), got)
    return got


# ---- 1. every model, 8 dense SPD classes in every warp -----------------------------------------------------------------------------
@pytest.mark.parametrize("name", MODELS)
def test_associate_equals_gated_rows_and_greedy(name):
    n = 20000
    pool, ids, cls, Q, R, fall, t = dense_pool(name, n, 100)
    rng = np.random.default_rng(5)
    t1 = t + 0.02
    for q in (1, 7, 2000):
        det = frame(pool, ids, t1, q, rng)
        wide = brute_pool(name, pool, cls, Q, R, t1, det[:1, :3], np.inf, n)[2][0, n // 20]   # a gate that takes 5 % of the targets
        for gate in (CHI2, wide):
            for K in (1, 4, 32):
                check_frame(pool, name, cls, Q, R, t1, det, gate, K)
    # gatedTargets itself is the numpy contract (tests/test_gpu_gate.py); one frame of it here too
    det = frame(pool, ids, t1, 7, rng)
    assert same(pool.gated_candidates(t1, det[:, :3], CHI2, 32), brute_pool(name, pool, cls, Q, R, t1, det[:, :3], CHI2, 32))
    pool.close()


# ---- 2. the index under stress, against gatedTargets ------------------------------------------------------------------------------
def scaled_classes(scales, inf_class=False, no_factor=False):
    """uniform-velocity classes with position sigma s (diagonal), one with near-singular coupled P0 (condition ~1e8), optionally one of
    infinite position variance and one whose S has no factor"""
    out = []
    for s in scales:
        Q = np.eye(6) * 1e-4 * s * s
        R = np.eye(3) * 1e-2 * s * s
        P0 = np.eye(6) * s * s
        out.append((Q, R, P0))
    u = np.array([1.0, 1.0, 1.0]) / np.sqrt(3)
    C = np.eye(3) * 1e-8 + np.outer(u, u)                          # condition number ~1e8
    P0 = np.zeros((6, 6)); P0[:3, :3] = C; P0[3:, 3:] = np.eye(3)
    out.append((np.zeros((6, 6)), np.zeros((3, 3)), P0))
    if inf_class:
        P0 = np.eye(6); P0[0, 0] = P0[1, 1] = P0[2, 2] = np.inf
        out.append((np.zeros((6, 6)), np.eye(3), P0))
    if no_factor:
        out.append((np.zeros((6, 6)), np.zeros((3, 3)), np.zeros((6, 6))))
    return out


def stress_pool(center, n=6000, seed=3, **kw):
    import target_estimation_b200 as te
    rng = np.random.default_rng(seed)
    classes = scaled_classes(10.0 ** np.arange(-6, 4), **kw)
    pool = te.TargetPool("uniform_velocity")
    for c, (Q, R, P0) in enumerate(classes):
        assert pool.register_class(Q, R, P0) == c
    ids = np.arange(n, dtype=np.uint32) * 2 + 1
    cls = np.arange(n) % len(classes)
    p = np.zeros((n, 7)); p[:, 6] = 1.0
    p[:, :3] = center + rng.normal(0, 50, (n, 3)) * (rng.random((n, 1)) < 0.5) + rng.normal(0, 1e-3, (n, 3))
    t0 = np.where(np.arange(n) % 7 == 3, 2.0, 0.5)                # every seventh target is later than the frame: never a candidate
    pool.add(ids, p, cls=cls.astype(np.uint16), t0=t0)
    return pool, ids, p, t0


@pytest.mark.parametrize("center", [0.0, 1e9])
def test_index_stress_equals_gated_rows(center):
    pool, ids, p, t0 = stress_pool(center, inf_class=True, no_factor=True)
    rng = np.random.default_rng(4)
    t1 = 1.0
    late = ids[t0 > t1]
    det = np.zeros((300, 7)); det[:, 6] = 1.0
    det[:, :3] = p[rng.choice(ids.size, 300), :3] + rng.normal(0, 1e-3, (300, 3)) * rng.choice([1e-9, 1e-3, 1.0, 1e3], (300, 1))
    for gate in (CHI2, 1e-6, 1e4):
        for K in (1, 32):
            cnt, cid, cd2 = pool.gated_candidates(t1, det[:, :3], gate, K)
            # with every late target erased from a twin, the rows are gatedTargets' rows
            assert not np.isin(cid, late).any()
            got = pool.associate(t1, det, gate, K)
            assert same_assignment(got, greedy(cid, cd2))
            assert np.array_equal(got[2], cnt)
            st = pool.assoc_stats()
            assert st["everywhere"] > 0 and st["levels"] > 1
    pool.erase(late)
    for gate in (CHI2, 1e4):
        ref = pool.gated_targets(t1, det[:, :3], gate, 32)
        assert same(pool.gated_candidates(t1, det[:, :3], gate, 32), ref)
    pool.close()


def test_every_detection_on_one_point_and_gate_zero():
    pool, ids, p, t0 = stress_pool(0.0)
    keep = ids[t0 <= 1.0]
    pool.erase(ids[t0 > 1.0])
    pos = pool.read_estimates(keep, 1.0)["pose"][:, :3]
    det = np.zeros((64, 7)); det[:, 6] = 1.0
    det[:, :3] = pos[17]                                          # every detection exactly on one target's position at t1
    for gate in (0.0, CHI2):
        for K in (1, 8):
            ref = pool.gated_targets(1.0, det[:, :3], gate, K)
            assert same(pool.gated_candidates(1.0, det[:, :3], gate, K), ref)
            got = pool.associate(1.0, det, gate, K)
            assert same_assignment(got, greedy(ref[1], ref[2]))
            assert got[0][0] != NO_ID and np.all(got[0][1:] != got[0][0])   # identical detections: the lowest j wins
            if gate == 0.0:
                assert ref[0][0] >= 1 and got[1][0] == 0.0
    # the exact boundary: a gate equal to a candidate's d2 keeps it
    z = pos[5] + 0.01
    ref = pool.gated_targets(1.0, z[None], np.inf, 4)
    b = ref[2][0, 2]
    cand = pool.gated_candidates(1.0, z[None], b, 4)
    assert cand[0][0] == 3 and np.array_equal(cand[1][0, :3], ref[1][0, :3])
    pool.close()


# ---- 3. ties ---------------------------------------------------------------------------------------------------------------------
def test_ties_resolve_by_id_then_by_detection():
    import target_estimation_b200 as te
    pool = te.TargetPool("uniform_velocity")
    pool.register_class(np.eye(6) * 1e-3, np.eye(3) * 1e-2, np.eye(6))
    ids = np.array([40, 7, 19, 3], dtype=np.uint32)
    p = np.zeros((4, 7)); p[:, 6] = 1.0
    p[:, 0] = [1.0, -1.0, 1.0, -1.0]                             # two pairs at equal distance from the origin
    pool.add(ids, p)
    det = np.zeros((3, 7)); det[:, 6] = 1.0                       # three identical detections at the origin
    got = pool.associate(0.0, det, 100.0, 4)
    assert list(got[0]) == [3, 7, 19] and got[1][0] == got[1][1] == got[1][2]
    assert same_assignment(got, greedy(*pool.gated_targets(0.0, det[:, :3], 100.0, 4)[1:]))
    pool.close()


# ---- 4. apply = 1 ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", MODELS)
def test_apply_equals_step_ids_with_per_target_dt(name):
    a, ids, cls, Q, R, fall, t = dense_pool(name, 8000, 60)
    b = dense_pool(name, 8000, 60)[0]
    rng = np.random.default_rng(8)
    m = fall.meas(t + 2 * DT)[::3]
    for pool in (a, b):                                           # targets at different times
        pool.step_ids(ids[::3], 2 * DT, m)
    t1 = t + 5 * DT
    det = frame(a, ids, t1, 1500, rng)
    before = a.read_state()
    ro = a.associate(t1, det, CHI2, 8, apply=False)
    assert all(np.array_equal(_bits(v), _bits(before[k])) for k, v in a.read_state().items())
    got = a.associate(t1, det, CHI2, 8, apply=True)
    assert same_assignment(got, ro) and np.array_equal(got[2], ro[2])
    hit = got[0] != NO_ID
    t_b = b.read_state(got[0][hit], want=("t",))["t"]
    assert b.step_ids(got[0][hit], t1 - t_b, det[hit]) == hit.sum()
    sa, sb = a.read_state(), b.read_state()
    for k in sa:
        assert np.array_equal(_bits(sa[k]), _bits(sb[k])), k
    untouched = ~np.isin(ids, got[0][hit])
    assert np.array_equal(_bits(sa["x"][untouched]), _bits(before["x"][untouched]))
    a.close(); b.close()


# ---- 5. handles after churn -----------------------------------------------------------------------------------------------------
def _states(m, ids):
    out = [m.state(int(i)) for i in ids]
    return {k: np.stack([np.asarray(s[k]) for s in out]) for k in out[0]}


def test_handles_equal_plain_manager(tmp_path):
    from target_estimation_b200.manager import ShardedManagerC, ShardedTickManagerC, TargetManagerC, TickManagerC
    name = "uniform_acceleration"
    path, Q, R = dense_yaml(tmp_path, name, 21)
    mgrs = (TargetManagerC(path), ShardedManagerC(path, 3, [0, 0, 0]), ShardedManagerC(path, 1, [0]), TickManagerC(path, device=0),
            ShardedTickManagerC(path, 3, [0, 0, 0]))
    ids = np.arange(3000, dtype=np.uint32) * 3 + 5
    fall = Falling(ids.size, seed=11)
    t = 0.0
    p0 = fall.meas(0.0)
    for m in mgrs:
        assert m.init_batch(ids, DT, p0) == ids.size
    rng = np.random.default_rng(9)
    for _ in range(40):
        t += DT
        meas = fall.meas(t)
        for m in mgrs:
            assert m.update_batch(ids, DT, meas) == ids.size
    gone = np.sort(rng.choice(ids, 90, replace=False))            # churn
    for m in mgrs:
        assert m.erase_batch(gone) == gone.size
    ids = ids[~np.isin(ids, gone)]
    part = ids[::4]
    meas = fall.meas(t + DT)[: part.size]
    for m in mgrs:                                                # targets at different times
        assert m.update_batch(part, DT, meas) == part.size
    t1 = t + 3 * DT
    pos = mgrs[0].get_estimates_batch(ids, t1)[0][:, :3]
    det = np.zeros((800, 7)); det[:, 6] = 1.0
    det[:, :3] = pos[rng.choice(ids.size, 800, replace=False)] + rng.normal(0, 0.003, (800, 3))
    ref = mgrs[0].associate(t1, det, CHI2, 8)
    rows = mgrs[0].gated(t1, det[:, :3], CHI2, 8)
    assert np.array_equal(ref[2], rows[0]) and same_assignment(ref, greedy(rows[1], rows[2]))
    for m in mgrs[1:]:
        got = m.associate(t1, det, CHI2, 8)
        assert same_assignment(got, ref) and np.array_equal(got[2], ref[2])
    for m in mgrs:
        got = m.associate(t1, det, CHI2, 8, apply=True)
        assert same_assignment(got, ref)
    want = _states(mgrs[0], ids)
    for m in mgrs[1:]:
        st = _states(m, ids)
        for k in want:
            assert np.array_equal(_bits(np.asarray(st[k], dtype=np.float64)), _bits(np.asarray(want[k], dtype=np.float64))), k
    for m in mgrs:
        m.close()


# ---- 6. scale: 1 Mi targets, 1 Mi detections + 10 % clutter -------------------------------------------------------------------------
def test_one_mi_by_one_mi():
    import target_estimation_b200 as te
    n = 1 << 20
    Q, R, P0 = (m[0] for m in dense_classes("uniform_acceleration", 1, 31))
    pool = te.TargetPool("uniform_acceleration")
    pool.register_class(Q, R, P0)
    rng = np.random.default_rng(12)
    ids = np.arange(n, dtype=np.uint32) * 2 + 1
    p = np.zeros((n, 7)); p[:, 6] = 1.0
    p[:, :3] = rng.uniform(-2000, 2000, (n, 3))
    pool.add(ids, p)
    t1 = 0.05
    q = n + n // 10
    det = np.zeros((q, 7)); det[:, 6] = 1.0
    det[:n, :3] = pool.read_estimates(ids, t1)["pose"][:, :3] + rng.normal(0, 0.3, (n, 3))
    det[n:, :3] = rng.uniform(-2000, 2000, (q - n, 3))
    det = det[rng.permutation(q)]
    K = 8
    cnt, cid, cd2 = pool.gated_candidates(t1, det[:, :3], CHI2, K)
    sample = rng.choice(q, 4096, replace=False)
    assert same((cnt[sample], cid[sample], cd2[sample]), pool.gated_targets(t1, det[sample, :3], CHI2, K))
    got = pool.associate(t1, det, CHI2, K)
    assert np.array_equal(got[2], cnt)
    assert same_assignment(got, greedy(cid, cd2))
    assert (got[0] != NO_ID).sum() > n // 2
    pool.close()


# ---- 7. mixed model types: the multi-pool merge and te_assign_greedy, from C++ ---------------------------------------------------
def test_cpp_associate_on_mixed_model_managers(tmp_path):
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lib = os.path.join(root, "target_estimation_b200", "lib")
    exe = str(tmp_path / "associate_test")
    subprocess.check_call(["g++", "-O1", "-ffp-contract=off", "-std=c++17", "-I", os.path.join(root, "include"),
                           os.path.join(root, "tests", "cpp", "associate_test.cpp"), "-o", exe, "-L", lib, "-ltarget_c", "-lte_pool",
                           "-Wl,-rpath," + lib])
    for G in ("1", "3"):
        r = subprocess.run([exe, os.path.join(root, "models"), G], capture_output=True, text=True, timeout=600)
        print(r.stdout[-3000:], r.stderr[-2000:])
        assert r.returncode == 0 and r.stdout.strip().splitlines()[-1].startswith("ok:")
