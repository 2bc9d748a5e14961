"""-m gpu: gating -- the k targets with the smallest Mahalanobis distance to a measured position (TargetManagerC.gated,
target_manager_gated, te_pool_gated_targets).

The query's d^2 is defined operation by operation (include/te_pool.h), so every check compares bit for bit with the numpy
restatement of that contract: x, P, t from read_state / TargetManagerC.state, Q and R the registered class matrices, the position
from get_estimates_batch / read_estimates at t1, the formula in the documented order, and np.lexsort((ids, d2)) over d2 <= gate.
The filters run dense random SPD classes (full off-diagonals in Q, R and P0), several of them in every warp."""
import os
import subprocess

import numpy as np
import pytest

from tests.test_gpu_isolver_handles import DT, Falling, _bits

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NO_ID = 0xFFFFFFFF
MODELS = ["uniform_acceleration", "angular_rates", "uniform_velocity", "angular_velocities"]
OFFSETS = {"uniform_velocity": (0, 3), "uniform_acceleration": (0, 3, 6), "angular_rates": (0, 6, 12), "angular_velocities": (0, 6)}
CHI2 = 11.34   # the 99 % quantile of the chi-square distribution with 3 degrees of freedom


# ---- the contract in numpy ---------------------------------------------------------------------------------------------------------
def dense_spd(rng, ref):
    """a random dense SPD matrix with the diagonal magnitudes of ref, bitwise symmetric"""
    d = np.diag(ref).copy()
    s = np.sqrt(np.where(d > 0, d, d.max() * 1e-6))
    a = rng.normal(size=ref.shape)
    x = (a @ a.T / ref.shape[0] + 0.5 * np.eye(ref.shape[0])) * s[:, None] * s[None, :]
    return (x + x.T) / 2


def dense_classes(name, n_cls, seed):
    """n_cls dense SPD (Q, R, P0) classes, stacked: Q [c][N][N], R [c][M][M], P0 [c][N][N]"""
    import target_estimation_b200 as te
    _, _, Q, R, P0 = te.load_model(name)
    rng = np.random.default_rng(seed)
    cl = [(dense_spd(rng, Q), dense_spd(rng, R), dense_spd(rng, P0)) for _ in range(n_cls)]
    return tuple(np.stack([c[i] for c in cl]) for i in range(3))


def pos_cov(name, P, t, cls, Q, t1):
    """C of the contract for every target, {(a, b): [n]} for a >= b; P [n][N][N] and Q [classes][N][N] read through the upper triangle"""
    def pu(i, j):
        return P[:, min(i, j), max(i, j)]
    if t1 is None:
        return {(a, b): pu(a, b) for a in range(3) for b in range(a + 1)}
    off = OFFSETS[name]
    tau = np.float64(t1) - t
    h = (0.5 * tau) * tau
    C = {}
    for a in range(3):
        for b in range(a + 1):
            r = []
            for ov in off:
                x = pu(off[0] + a, ov + b) + tau * pu(off[1] + a, ov + b)
                if len(off) == 3:
                    x = x + h * pu(off[2] + a, ov + b)
                r.append(x)
            c = r[0] + tau * r[1]
            if len(off) == 3:
                c = c + h * r[2]
            C[a, b] = c + Q[cls, b, a]
    return C


def mahalanobis2(C, R, cls, d):
    """d^2 through the Cholesky factor of S = C + R[0:3, 0:3] in the documented order; NaN where the factor does not exist"""
    S = {(a, b): C[a, b] + R[cls, b, a] for (a, b) in C}
    with np.errstate(all="ignore"):
        l00 = np.sqrt(S[0, 0])
        l10 = S[1, 0] / l00
        l20 = S[2, 0] / l00
        rad1 = S[1, 1] - l10 * l10
        l11 = np.sqrt(rad1)
        l21 = (S[2, 1] - l20 * l10) / l11
        rad2 = (S[2, 2] - l20 * l20) - l21 * l21
        l22 = np.sqrt(rad2)
        w0 = d[:, 0] / l00
        w1 = (d[:, 1] - l10 * w0) / l11
        w2 = ((d[:, 2] - l20 * w0) - l21 * w1) / l22
        d2 = (w0 * w0 + w1 * w1) + w2 * w2
    return np.where((S[0, 0] > 0) & (rad1 > 0) & (rad2 > 0), d2, np.nan)


def brute(name, ids, P, t, cls, Q, R, positions, t1, z, gate, k):
    """(count, ids [q][k], d2 [q][k]) of the contract; positions(t1) = every target's position at t1 (None: now)"""
    z = np.asarray(z, dtype=np.float64).reshape(-1, 3)
    q = z.shape[0]
    gate = np.broadcast_to(np.asarray(gate, dtype=np.float64), (q,))
    when = [None] * q if t1 is None else list(np.broadcast_to(np.asarray(t1, dtype=np.float64), (q,)))
    count = np.zeros(q, dtype=np.int64)
    out_ids = np.full((q, k), NO_ID, dtype=np.uint32)
    out_d = np.full((q, k), -1.0)
    last = ()
    for j in range(q):
        key = None if when[j] is None else _bits(np.float64(when[j])).tobytes()
        if key != last:
            C, pos, last = pos_cov(name, P, t, cls, Q, when[j]), positions(when[j]), key
        d2 = mahalanobis2(C, R, cls, pos - z[j])
        inside = d2 <= gate[j]
        count[j] = int(inside.sum())
        ii, dd = ids[inside], d2[inside]
        order = np.lexsort((ii, dd))[:k]
        out_ids[j, :order.size] = ii[order]
        out_d[j, :order.size] = dd[order]
    return count, out_ids, out_d


def brute_pool(name, pool, cls, Q, R, t1, z, gate, k):
    ids = pool.ids()
    st = pool.read_state(ids, want=("P", "t"))
    return brute(name, ids, st["P"], st["t"], cls, Q, R, lambda w: pool.read_estimates(ids, w)["pose"][:, :3], t1, z, gate, k)


def brute_mgr(name, mgr, Q, R, t1, z, gate, k):
    """a manager of one class (the YAML's): the state one id at a time"""
    ids = mgr.ids()
    st = [mgr.state(int(i)) for i in ids]
    P, t = np.stack([s["P"] for s in st]), np.array([s["t"] for s in st])
    cls = np.zeros(ids.size, dtype=np.int64)

    def positions(w):
        pose, _, _, found = mgr.get_estimates_batch(ids, w)
        assert found.all()
        return pose[:, :3]
    return brute(name, ids, P, t, cls, Q[None], R[None], positions, t1, z, gate, k)


def same(a, b):
    """two (count, ids, d2) results, bit for bit"""
    return np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(_bits(a[2]), _bits(b[2]))


def pad(ref, k):
    count, ids, d2 = ref
    if k <= ids.shape[1]:
        return count, ids[:, :k], d2[:, :k]
    w = ((0, 0), (0, k - ids.shape[1]))
    return count, np.pad(ids, w, constant_values=NO_ID), np.pad(d2, w, constant_values=-1.0)


def dense_pool(name, n, ticks, seed=11, n_cls=8):
    """a pool of n falling targets over n_cls dense classes, interleaved (slot s holds class s % n_cls: every warp holds all of them),
    after `ticks` updates"""
    import target_estimation_b200 as te
    Q, R, P0 = dense_classes(name, n_cls, seed)
    pool = te.TargetPool(name)
    for c in range(n_cls):
        assert pool.register_class(Q[c], R[c], P0[c]) == c
    ids = np.arange(n, dtype=np.uint32) * 3 + 5
    cls = np.arange(n) % n_cls
    fall = Falling(n, seed=seed)
    pool.add(ids, fall.meas(0.0), cls=cls)
    t = 0.0
    for _ in range(ticks):
        t += DT
        pool.step_ids(ids, DT, fall.meas(t))
    return pool, ids, cls, Q, R, fall, t


def near(pool, ids, t, q, rng, sigma=0.003):
    """q measured positions close to random targets"""
    rows = rng.choice(ids.size, q, replace=False)
    return pool.read_estimates(ids[rows], t)["pose"][:, :3] + rng.normal(0, sigma, (q, 3))


def dense_yaml(tmp_path, name, seed):
    """a model file of one dense SPD class, in the loader's column-major lists (the matrices are symmetric)"""
    Q, R, P0 = (m[0] for m in dense_classes(name, 1, seed))
    path = str(tmp_path / ("dense_%s.yaml" % name))
    with open(path, "w") as f:
        f.write("type: %s\nfrequency: 250.0\n" % name)
        for key, m in (("Q", Q), ("R", R), ("P", P0)):
            f.write("%s: [%s]\n" % (key, ", ".join("%.17e" % v for v in m.T.ravel())))
    return path, Q, R


# ---- 1. pools of every model, dense classes: every shape = brute force, bit for bit ----------------------------------------------
@pytest.mark.parametrize("name", MODELS)
def test_gated_equals_brute_force(name):
    n = 20000
    pool, ids, cls, Q, R, fall, t = dense_pool(name, n, 100)
    rng = np.random.default_rng(2)
    inside_chi2 = 0
    for q in (1, 7, 64):
        z = near(pool, ids, t, q, rng)
        t1 = t + 0.01 * (np.arange(q) // 3 % 3)                 # runs of three equal t1; a run may come back to an earlier t1
        for when in (t1, None):
            full_inf = brute_pool(name, pool, cls, Q, R, when, z, np.inf, n)
            assert np.all(full_inf[0] == n)
            wide = full_inf[2][:, n // 20]                        # a gate that takes 5 % of the targets
            for gate in (np.full(q, CHI2), wide, np.full(q, np.inf)):
                full = full_inf if np.isinf(gate[0]) else brute_pool(name, pool, cls, Q, R, when, z, gate, n)
                count = full[0]
                if gate is wide:
                    assert np.all(count >= n // 20 + 1) and np.all(count < n // 10)
                if gate[0] == CHI2:
                    inside_chi2 += int(count.sum())
                for k in (0, 1, 100, int(count.max()) + 7):
                    assert same(pool.gated_targets(when, z, gate, k), pad(full, k)), (q, when is None, gate[0], k)
    assert inside_chi2 > 0
    pool.close()


# ---- 2. the contract is the filter's own predict: twin pools stepped with one predict of dt = tau ------------------------------
@pytest.mark.parametrize("name", MODELS)
def test_contract_matches_the_filter_predict(name):
    import target_estimation_b200 as te
    n, tau = 5000, 0.013
    pool, ids, cls, Q, R, fall, t = dense_pool(name, n, 100, seed=4)
    twin = dense_pool(name, n, 100, seed=4)[0]
    before = pool.read_state(ids, want=("x", "P", "t"))
    assert np.array_equal(_bits(before["P"]), _bits(twin.read_state(ids, want=("P",))["P"]))
    t1 = t + tau
    C = pos_cov(name, before["P"], before["t"], cls, Q, t1)
    assert twin.step_ids(ids, tau, None, np.full(n, te.ACT_PREDICT, dtype=np.uint8)) == n
    after = twin.read_state(ids, want=("x", "P", "t"))
    Pp = after["P"][:, :3, :3]
    scale = np.abs(Pp).reshape(n, 9).max(axis=1)
    for (a, b), c in C.items():
        assert np.all(np.abs(c - Pp[:, a, b]) <= 1e-12 * scale), (a, b)
    z = near(pool, ids, t1, 16, np.random.default_rng(6))
    count, got_ids, got_d2 = pool.gated_targets(t1, z, np.inf, n)
    assert np.all(count == n)
    S = Pp + R[cls][:, :3, :3]
    row = np.searchsorted(ids, got_ids)
    for j in range(16):
        d = after["x"][:, :3] - z[j]
        ref = np.einsum("ni,ni->n", d, np.linalg.solve(S, d[:, :, None])[:, :, 0])
        assert np.all(np.abs(got_d2[j] - ref[row[j]]) <= 1e-9 * ref[row[j]]), j
    pool.close(); twin.close()


# ---- 3. every handle, dense-SPD model file: each equals the brute force, sharded equals plain --------------------------------------
def test_plain_and_sharded_handles_after_churn(tmp_path):
    from target_estimation_b200.manager import ShardedManagerC, TargetManagerC
    name = "uniform_acceleration"
    path, Q, R = dense_yaml(tmp_path, name, 21)
    mgrs = (TargetManagerC(path), ShardedManagerC(path, 3, [0, 0, 0]), ShardedManagerC(path, 1, [0]))
    ids = np.arange(3000, dtype=np.uint32) * 3 + 5
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
    rows = np.arange(ids.size)
    for _ in range(3):                                        # churn: erase a few percent, add as many fresh ids, keep stepping
        gone = np.sort(rng.choice(ids, 90, replace=False))
        for m in mgrs:
            assert m.erase_batch(gone) == gone.size
        keep = ~np.isin(ids, gone)
        fresh = np.arange(90, dtype=np.uint32) * 3 + int(ids.max()) + 1
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
    z = mgrs[0].get_estimates_batch(ids[rng.choice(ids.size, 16, replace=False)], t)[0][:, :3] + rng.normal(0, 0.003, (16, 3))
    for when in (t + 0.05, None):
        for gate in (CHI2, np.inf):
            ref = brute_mgr(name, mgrs[0], Q, R, when, z, gate, 500)
            for m in mgrs:
                assert same(m.gated(when, z, gate, 500), ref), (when is None, gate)
    assert same(mgrs[1].gated(t, z, 1e4, 500), brute_mgr(name, mgrs[1], Q, R, t, z, 1e4, 500))
    for m in mgrs:
        m.close()


def test_tick_and_sharded_tick_handles_after_churn(tmp_path):
    from target_estimation_b200.manager import ShardedTickManagerC, TickManagerC
    from tests.test_gpu_sharded_tick import _churn_messages
    name = "angular_velocities"
    path, Q, R = dense_yaml(tmp_path, name, 22)
    mgr, one = ShardedTickManagerC(path, 3, [0, 0, 0]), TickManagerC(path, device=0)
    for m in (mgr, one):
        m.set_expiration(8 * DT)
    rng = np.random.default_rng(3)
    checked = 0
    for k, (ids, s, ns, poses, now) in enumerate(_churn_messages(n=3000, ticks=24)):
        for m in (mgr, one):
            m.callback_ids(ids, s, ns, poses)
        assert np.array_equal(mgr.tick(DT, *now), one.tick(DT, *now))
        if k % 6 != 5:
            continue
        pub_ids, pub = one.published()
        z = pub[rng.choice(pub_ids.size, 8, replace=False), :3] + rng.normal(0, 0.003, (8, 3))
        for when in (one.time() + 0.05, None):
            for gate in (CHI2, np.inf):
                ref = brute_mgr(name, one, Q, R, when, z, gate, 300)
                assert same(one.gated(when, z, gate, 300), ref) and same(mgr.gated(when, z, gate, 300), ref), (k, gate)
            checked += 1
    assert checked == 8
    mgr.close(); one.close()


# ---- 4. ties: identical histories come out by ascending id ----------------------------------------------------------------------
@pytest.mark.parametrize("G", [1, 3])
def test_ties_come_out_by_ascending_id(G, tmp_path):
    """groups of three targets with identical histories: ids 3g + 5, 3g + 6, 3g + 7 (on three different shards when G = 3)"""
    from target_estimation_b200.manager import ShardedManagerC, TargetManagerC
    name = "uniform_acceleration"
    path, Q, R = dense_yaml(tmp_path, name, 23)
    n_groups = 1000
    n = 3 * n_groups
    ids = np.arange(n, dtype=np.uint32) + 5
    fall = Falling(n_groups, seed=6)
    grp = np.arange(n) // 3
    mgr = TargetManagerC(path) if G == 1 else ShardedManagerC(path, G, [0] * G)
    assert mgr.init_batch(ids, DT, fall.meas(0.0)[grp]) == n
    t = 0.0
    for _ in range(100):
        t += DT
        assert mgr.update_batch(ids, DT, fall.meas(t)[grp]) == n
    rng = np.random.default_rng(4)
    z = mgr.get_estimates_batch(ids[rng.choice(n, 5, replace=False)], t)[0][:, :3] + rng.normal(0, 0.5, (5, 3))
    full = brute_mgr(name, mgr, Q, R, t, z, np.inf, n)
    gate = full[2][:, 299]                                    # 300 rows: 100 whole groups (ties never straddle: d2 of groups differ)
    count, r_ids, r_d = brute_mgr(name, mgr, Q, R, t, z, gate, n)
    assert np.all(count % 3 == 0) and count.min() >= 9
    for j in range(5):
        d = r_d[j, :count[j]]
        assert np.array_equal(d[0::3], d[1::3]) and np.array_equal(d[0::3], d[2::3])   # the groups do tie
    for k in (1, 2, 4, 5, 3 * int(count.min() // 6) + 1, 3 * int(count.min() // 3) - 1):
        got = mgr.gated(t, z, gate, k)
        assert same(got, (count, r_ids[:, :k], r_d[:, :k])), k
        rows = min(k, int(count.min()))
        assert np.all(np.diff(got[1][:, :rows].astype(np.int64), axis=1)[np.diff(got[2][:, :rows], axis=1) == 0] > 0)
    mgr.close()


# ---- 5. the boundary counts; a class whose S has no factor never does ------------------------------------------------------------
def test_exact_boundary_counts_as_inside():
    name = "uniform_velocity"
    pool, ids, cls, Q, R, fall, t = dense_pool(name, 3000, 50)
    rng = np.random.default_rng(17)
    z = near(pool, ids, t, 8, rng, sigma=0.05)
    full = brute_pool(name, pool, cls, Q, R, t, z, np.inf, 3000)
    at = rng.integers(0, 200, 8)
    gate = full[2][np.arange(8), at]                          # the d2 of row at[j] of query j
    below = np.nextafter(gate, 0.0)
    count, got_ids, got_d2 = pool.gated_targets(t, z, gate, 3000)
    assert same((count, got_ids, got_d2), brute_pool(name, pool, cls, Q, R, t, z, gate, 3000))
    c_below, ids_below, _ = pool.gated_targets(t, z, below, 3000)
    assert same(pool.gated_targets(t, z, below, 3000), brute_pool(name, pool, cls, Q, R, t, z, below, 3000))
    for j in range(8):
        target = full[1][j, at[j]]
        hit = np.nonzero(got_ids[j, :count[j]] == target)[0]
        assert hit.size == 1 and got_d2[j, hit[0]] == gate[j]                           # d2 == gate: inside
        assert target not in ids_below[j, :c_below[j]] and c_below[j] < count[j]         # one ulp less: outside
    pool.close()


def test_class_without_a_factor_is_never_a_candidate():
    import target_estimation_b200 as te
    name = "uniform_acceleration"
    Q, R, P0 = dense_classes(name, 2, 8)
    R[1, 0, 0] = -10.0                                        # R_pp of class 1 is indefinite: S00 < 0, S has no factor
    pool = te.TargetPool(name)
    for c in range(2):
        assert pool.register_class(Q[c], R[c], P0[c]) == c
    n = 4000
    ids = np.arange(n, dtype=np.uint32) + 1
    cls = (np.arange(n) // 5) % 2
    fall = Falling(n, seed=3)
    pool.add(ids, fall.meas(0.0), cls=cls)
    for _ in range(10):
        pool.predict_all(DT)                                   # no update: R never enters the filters
    z = pool.read_estimates(ids[:6])["pose"][:, :3]
    good = int((cls == 0).sum())
    for when in (None, 10 * DT + 0.02):
        count, got_ids, got_d2 = pool.gated_targets(when, z, np.inf, n)
        assert np.all(count == good)
        assert not np.isin(got_ids, ids[cls == 1]).any()
        assert same((count, got_ids, got_d2), brute_pool(name, pool, cls, Q, R, when, z, np.inf, n))
    pool.close()


# ---- 6. read-only ---------------------------------------------------------------------------------------------------------------
def test_query_leaves_the_filters_alone():
    name = "angular_rates"
    pool, ids, cls, Q, R, fall, t = dense_pool(name, 5000, 40)
    want = ("x", "P", "t", "n_meas")
    before = pool.read_state(ids, want=want)
    rng = np.random.default_rng(12)
    z = near(pool, ids, t, 40, rng)
    for when in (t + 0.01 * (np.arange(40) % 4), None):
        for gate in (CHI2, np.inf):
            pool.gated_targets(when, z, gate, 700)
    after = pool.read_state(ids, want=want)
    for key in want:
        assert np.array_equal(_bits(before[key]), _bits(after[key])), key
    pool.close()


# ---- 7. mixed-model managers (C++) -----------------------------------------------------------------------------------------------
def test_cpp_gated_on_mixed_model_managers(tmp_path):
    lib = os.path.join(ROOT, "target_estimation_b200", "lib")
    exe = str(tmp_path / "gate_test")
    subprocess.check_call(["g++", "-O1", "-ffp-contract=off", "-std=c++17", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "gate_test.cpp"), "-o", exe, "-L", lib, "-ltarget_c", "-lte_pool",
                           "-Wl,-rpath," + lib])
    for G in ("1", "3"):
        r = subprocess.run([exe, os.path.join(ROOT, "models"), G], capture_output=True, text=True, timeout=600)
        print(r.stdout[-3000:], r.stderr[-2000:])
        assert r.returncode == 0 and r.stdout.strip().splitlines()[-1].startswith("ok:")


# ---- 8. scale: every target is a candidate ----------------------------------------------------------------------------------------
def test_one_mi_targets_sixteen_queries_gate_inf():
    name = "uniform_acceleration"
    n = 1 << 20
    pool, ids, cls, Q, R, fall, t = dense_pool(name, n, 30, seed=31)
    z = near(pool, ids, t, 16, np.random.default_rng(5), sigma=2.0)
    ref = brute_pool(name, pool, cls, Q, R, t + 0.05, z, np.inf, 10000)
    assert np.all(ref[0] == n)
    assert same(pool.gated_targets(t + 0.05, z, np.inf, 10000), ref)
    pool.close()
