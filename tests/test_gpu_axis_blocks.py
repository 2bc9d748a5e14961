"""-m gpu: the axis-blocked UV / UA step (te_kin_sym.cuh AXIS).  A pool whose classes never couple the x / y / z axes moves only the
per-axis covariance blocks; its twin holds the same classes plus one unused, bitwise-symmetric coupled class, so it runs the packed
direct kernel on the whole upper triangle.  After every phase both pools hold the same x, P, t and n_meas (np.array_equal: +0 and -0
count as equal), and every cross-axis entry of P reads back as 0."""
import ctypes as C

import numpy as np
import pytest

from tests import orc, synth

pytestmark = pytest.mark.gpu
DT = 1.0 / 250.0
MODELS = ["uniform_velocity", "uniform_acceleration"]


def _cross(N):
    a = np.arange(N) % 3
    return a[:, None] != a[None, :]


def _sym(A):
    return np.triu(A) + np.triu(A, 1).T   # bitwise symmetric


def _decoupled_class(N, M, rng):
    """random SPD blocks on each axis (indices r, r + 3, ...), zeros between axes, diagonal R"""
    Q, P0 = np.zeros((N, N)), np.zeros((N, N))
    for r in range(3):
        idx = np.ix_(np.arange(r, N, 3), np.arange(r, N, 3))
        for A, s in ((Q, 1e-3), (P0, 1.0)):
            B = rng.normal(size=(N // 3, N // 3))
            A[idx] = s * (B @ B.T + N // 3 * np.eye(N // 3))
    return _sym(Q), np.diag(rng.uniform(1e-4, 1e-2, M)), _sym(P0)


def _coupled_class(N, M, rng):
    B = rng.normal(size=(N, N))
    Q = _sym(1e-3 * (B @ B.T + N * np.eye(N)))
    B = rng.normal(size=(M, M))
    R = _sym(1e-3 * (B @ B.T + M * np.eye(M)))
    B = rng.normal(size=(N, N))
    return Q, R, _sym(B @ B.T + N * np.eye(N))


def _twins(te, mtype, classes, coupled):
    """(blocked pool, twin on the full path): the same classes in the same order, the twin with the coupled class behind them"""
    pools = []
    for extra in ((), (coupled,)):
        p = te.TargetPool(mtype)
        for c in tuple(classes) + extra:
            p.register_class(*c)
        pools.append(p)
    return pools


def _check(blk, ref, ids, N, what):
    want = ("x", "P", "t", "n_meas")
    a, b = blk.read_state(ids, want=want), ref.read_state(ids, want=want)
    for key in want:
        assert np.array_equal(a[key], b[key]), (what, key)
    assert np.all(a["P"][:, _cross(N)] == 0.0), what
    assert np.all(np.isfinite(a["P"])), what


def _setup(model, n, ticks, seed):
    import target_estimation_b200 as te
    mtype, _, Q, R, P0 = te.load_model(model)
    N, M = te.model_dims(mtype)
    assert np.all(Q[_cross(N)] == 0) and np.all(P0[_cross(N)] == 0) and np.array_equal(R, np.diag(np.diag(R)))   # shipped: decoupled
    rng = np.random.default_rng(seed)
    meas, action, scale = synth.make_streams(n, ticks, DT, accel=model == "uniform_acceleration", angular=False, seed=seed)
    action[1:, ::13] = 0                                   # ACT_NONE lanes next to the 5 % predict-only ones
    return te, mtype, N, M, (Q, R, P0), _coupled_class(N, M, rng), rng, meas, action, scale


@pytest.mark.parametrize("model", MODELS)
def test_blocked_equals_full_path(model):
    """dense ticks (strides 7 and 3), sparse ticks by id with per-row dt, predict_all, replay, a live launch and the host-tick pipeline"""
    import torch
    n, ticks = 3000 + 17, 12
    te, mtype, N, M, cls, coupled, rng, meas, action, scale = _setup(model, n, ticks, 71)
    blk, ref = _twins(te, mtype, [cls], coupled)
    ids = np.arange(n, dtype=np.uint32) * 3 + 1
    t0 = rng.uniform(0.0, 1.0, n)
    for p in (blk, ref):
        p.add(ids, meas[0], t0=t0, p0_scale=scale)
    _check(blk, ref, ids, N, "add")
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    for k in range(4):
        stride = 7 if k < 2 else 3
        for p in (blk, ref):
            p.step_dense(DT, dev(meas[k][:, :stride]), stride, dev(action[k]))
        _check(blk, ref, ids, N, ("dense", k, stride))
    # sparse ticks by id: a shuffled subset, per-row dt, mixed actions; then a predict of everybody
    for k in range(2):
        sel = rng.permutation(n)[: n // 3]
        dts = rng.uniform(0.5, 2.0, sel.size) * DT
        act = rng.choice(np.array([te.ACT_PREDICT, te.ACT_UPDATE], dtype=np.uint8), size=sel.size, p=[0.1, 0.9])
        for p in (blk, ref):
            assert p.step_ids(ids[sel], dts, meas[4 + k][sel], act) == sel.size
        _check(blk, ref, ids, N, ("ids", k))
    for p in (blk, ref):
        p.predict_all(0.5 * DT)
    _check(blk, ref, ids, N, "predict_all")
    # replay: four ticks in one launch
    for stride in (7, 3):
        m = dev(meas[6:10, :, :stride])
        a = dev(action[6:10])
        for p in (blk, ref):
            p.step_dense_ticks(4, DT, m, stride, a)
        _check(blk, ref, ids, N, ("replay", stride))
    # one short live launch per pool (nothing may synchronise the device while a launch is resident)
    for p in (blk, ref):
        d_meas = torch.zeros((3, n, 7), dtype=torch.float64, device="cuda")
        d_act = torch.zeros((3, n), dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        p.live_begin(3, DT, d_meas, 7, d_act, te.ACT_UPDATE, None)
        for k in range(3):
            assert p.live_push(np.ascontiguousarray(meas[9 + k]), action[9 + k]) == k + 1
        assert p.live_wait(3) >= 3
        assert p.live_end() == 3
    _check(blk, ref, ids, N, "live")
    # the host-tick pipeline: synchronous, then two ticks in flight
    outs = {}
    for name, p in (("blk", blk), ("ref", ref)):
        outs[name] = [np.zeros((n, 3)) for _ in range(3)]
        for k in range(3):
            ms = np.ascontiguousarray(meas[k][:, :3])
            fn = te.lib.te_pool_tick_host if k == 0 else te.lib.te_pool_tick_host_async
            assert fn(p._h, DT, ms.ctypes.data_as(C.c_void_p), 3, action[k].ctypes.data_as(C.c_void_p), te.ACT_UPDATE,
                      outs[name][k].ctypes.data_as(C.c_void_p)) == 0
            if k:
                assert te.lib.te_pool_tick_host_wait(p._h, 1) == 0
        assert te.lib.te_pool_tick_host_wait(p._h, 0) == 0
    for k in range(3):
        assert np.array_equal(outs["blk"][k], outs["ref"][k]), k
    _check(blk, ref, ids, N, "tick_host")
    for p in (blk, ref):
        p.close()


def _dirty_device_memory(te, mtype, coupled, n):
    """a pool of dense covariances, stepped and destroyed: the allocations that follow are likely to reuse its memory"""
    p = te.TargetPool(mtype)
    p.register_class(*coupled)
    p.add(np.arange(n, dtype=np.uint32), np.tile([1.0, 2.0, 3.0, 0, 0, 0, 1.0], (n, 1)))
    p.predict_all(DT)
    p.sync()
    p.close()


@pytest.mark.parametrize("model", MODELS)
def test_blocked_equals_full_path_compacting(model):
    """fused step + expiry (the step writes the survivors into the compacted slots of the second buffer) and mailbox ticks with churn"""
    import torch
    n0, ticks = 3000 + 13, 16
    te, mtype, N, M, cls, coupled, rng, meas_all, action_all, scale = _setup(model, n0 + 40 * ticks, ticks, 72)
    _dirty_device_memory(te, mtype, coupled, 200000)
    blk, ref = _twins(te, mtype, [cls], coupled)
    for p in (blk, ref):
        p.add(np.arange(n0, dtype=np.uint32), meas_all[0, :n0], p0_scale=scale[:n0])
    silent = np.zeros(n0 + 40 * ticks, dtype=bool)
    next_id, total = n0, 0
    for k in range(ticks):
        ids = blk.ids()
        assert np.array_equal(ids, ref.ids())
        silent[rng.choice(ids, size=max(1, ids.size // (5 if k in (2, 9) else 50)), replace=False)] = True
        act = np.where(silent[ids], te.ACT_PREDICT, action_all[k, ids]).astype(np.uint8)
        act[silent[ids] & (rng.random(ids.size) < 0.1)] = te.ACT_NONE
        m = torch.from_numpy(np.ascontiguousarray(meas_all[k, ids])).cuda()
        a = torch.from_numpy(act).cuda()
        ns = 1000 * 10**9 + k * 4000000
        er = [p.step_dense_expire(DT, m, 7, a, te.ACT_UPDATE, (ns // 10**9, ns % 10**9), (ns // 10**9, ns % 10**9), 3 * DT) for p in (blk, ref)]
        assert np.array_equal(er[0], er[1]), k
        total += er[0].size
        _check(blk, ref, blk.ids(), N, ("expire", k))
        fresh = np.arange(next_id, next_id + 40, dtype=np.uint32)
        next_id += 40
        for p in (blk, ref):
            p.add(fresh, meas_all[k, fresh], t0=np.full(40, k * DT), p0_scale=scale[fresh])
    assert total > n0 // 4
    for p in (blk, ref):
        p.close()
    # mailbox ticks: survivors stepped into their merged slots, new targets initialised and updated in a sparse follow-up launch
    _dirty_device_memory(te, mtype, coupled, 200000)
    blk, ref = _twins(te, mtype, [cls], coupled)
    universe = rng.choice(100000, size=3000, replace=False).astype(np.uint32)
    live, nxt, n_er = list(range(900)), 900, 0
    for k in range(ticks):
        now = 1000 * 10**9 + k * 4_000_000
        gone = set(j for j in live if rng.random() < 0.03)
        live = [j for j in live if j not in gone] + list(range(nxt, nxt + 40))
        nxt += 40
        speak = np.array([j for j in live if rng.random() < 0.95])
        st = np.tile([now // 10**9, now % 10**9], (speak.size, 1)).astype(np.uint32)
        out = []
        for p in (blk, ref):
            p.mailbox_ingest(universe[speak], st[:, 0].copy(), st[:, 1].copy(), meas_all[k, speak])
            out.append(p.mailbox_tick(DT, k * DT, (now // 10**9, now % 10**9), 6 * DT, want_added=True))
        for x, y in zip(out[0], out[1]):
            assert np.array_equal(x, y), k
        n_er += out[0][0].size
        assert np.array_equal(blk.ids(), ref.ids())
        _check(blk, ref, blk.ids(), N, ("mailbox", k))
    assert n_er > 50
    for p in (blk, ref):
        p.close()


@pytest.mark.parametrize("model", MODELS)
def test_eight_decoupled_classes(model):
    """8 random decoupled classes in every warp: equal to the twin, and to the oracle at the 1e-9 bar"""
    import torch
    n, ticks = 2000 + 5, 20
    te, mtype, N, M, _, coupled, rng, meas, action, scale = _setup(model, n, ticks, 73)
    classes = [_decoupled_class(N, M, rng) for _ in range(8)]
    blk, ref = _twins(te, mtype, classes, coupled)
    ids = np.arange(n, dtype=np.uint32) + 11
    cls = (np.arange(n) % 8).astype(np.uint16)
    for p in (blk, ref):
        p.add(ids, meas[0], cls=cls, p0_scale=scale)
    mgr = orc.ShardedManager()
    for c in range(8):
        s = cls == c
        mgr.init_batch(mtype, ids[s], DT, *classes[c], meas[0][s], scale[s])
    for k in range(ticks):
        for p in (blk, ref):
            p.step_dense(DT, torch.from_numpy(np.ascontiguousarray(meas[k])).cuda(), 7, torch.from_numpy(action[k]).cuda())
        if k % 5 == 4:
            _check(blk, ref, ids, N, ("dense", k))
    mgr.step_ticks(ids, DT, meas, action)
    want, got = mgr.states(ids, N), blk.read_state(ids)
    assert synth.compare_h2(got["x"], want["x"]) <= 1.0 and synth.compare_h2(got["P"], want["P"]) <= 1.0
    assert np.array_equal(got["n_meas"], want["n_meas"])
    for p in (blk, ref):
        p.close()
    mgr.close()


@pytest.mark.parametrize("model", MODELS)
def test_coupled_class_mid_stream(model):
    """a coupled class registered after some blocked ticks: the pool switches to the full path and stays equal to a twin that was
    on it from the start, its new coupled targets included"""
    import torch
    n, ticks = 2000 + 9, 10
    te, mtype, N, M, cls, coupled, rng, meas, action, scale = _setup(model, n + 300, ticks, 74)
    blk, ref = _twins(te, mtype, [cls], coupled)
    ids = np.arange(n, dtype=np.uint32)
    for p in (blk, ref):
        p.add(ids, meas[0, :n], p0_scale=scale[:n])
    step = lambda p, k, sel: p.step_dense(DT, torch.from_numpy(np.ascontiguousarray(meas[k, sel])).cuda(), 7,
                                          torch.from_numpy(np.ascontiguousarray(action[k, sel])).cuda())
    for k in range(4):
        for p in (blk, ref):
            step(p, k, slice(0, n))
    _check(blk, ref, ids, N, "blocked")
    assert blk.register_class(*coupled) == 1
    new = np.arange(n, n + 300, dtype=np.uint32)
    for p in (blk, ref):
        p.add(new, meas[4, n:n + 300], cls=np.ones(300, dtype=np.uint16), p0_scale=scale[n:n + 300])
    all_ids = np.concatenate([ids, new])
    for k in range(4, ticks):
        for p in (blk, ref):
            step(p, k, slice(0, n + 300))
    want = ("x", "P", "t", "n_meas")
    a, b = blk.read_state(all_ids, want=want), ref.read_state(all_ids, want=want)
    for key in want:
        assert np.array_equal(a[key], b[key]), key
    assert np.all(a["P"][:n][:, _cross(N)] == 0.0)       # the decoupled targets keep their zeros on the full path
    assert np.any(a["P"][n:][:, _cross(N)] != 0.0)
    for p in (blk, ref):
        p.close()
