"""not gpu: target_manager_nearest and te_pool_nearest_targets reject invalid arguments with -1 and a message, and q = 0 or a
manager without targets return 0 without device work (a plain manager makes no device call until it holds targets)."""
import ctypes as C
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def mgr():
    from target_estimation_b200.manager import TargetManagerC
    m = TargetManagerC(os.path.join(ROOT, "models", "model_uniform_velocity_params.yaml"))
    yield m
    m.close()


def _err():
    from target_estimation_b200.manager import clib
    return clib.target_manager_last_error().decode()


def test_bad_arguments(mgr):
    from target_estimation_b200.manager import _ptr, clib
    t1, p, r = np.zeros(2), np.zeros((2, 3)), np.ones(2)
    ids, d, c = np.zeros((2, 4), dtype=np.uint32), np.zeros((2, 4)), np.zeros(2, dtype=np.int64)
    args = [_ptr(t1), _ptr(p), _ptr(r), 4, _ptr(ids), _ptr(d), _ptr(c)]
    assert clib.target_manager_nearest(None, 2, *args) == -1 and "null manager" in _err()
    assert clib.target_manager_nearest(mgr.h, -1, *args) == -1 and "q must be" in _err()
    for k in (-1, 65537):
        assert clib.target_manager_nearest(mgr.h, 2, _ptr(t1), _ptr(p), _ptr(r), k, _ptr(ids), _ptr(d), _ptr(c)) == -1
        assert "k must be" in _err()
    for i in (1, 2, 4, 5, 6):   # point, radius, ids_out, dist_out, count_out (t1 may be NULL)
        a = list(args)
        a[i] = None
        assert clib.target_manager_nearest(mgr.h, 2, *a) == -1 and "required" in _err()
    for bad in (-1.0, -1e-300, np.nan):
        rb = np.array([1.0, bad])
        assert clib.target_manager_nearest(mgr.h, 2, _ptr(t1), _ptr(p), _ptr(rb), 4, _ptr(ids), _ptr(d), _ptr(c)) == -1
        assert "radius must be" in _err() and "query 1" in _err()
    with pytest.raises(RuntimeError, match="k must be"):
        mgr.nearest(0.0, p, 1.0, 70000)
    with pytest.raises(RuntimeError, match="radius must be"):
        mgr.nearest(None, p, -0.5, 3)


def test_zero_queries_counts_only_and_empty_manager(mgr):
    from target_estimation_b200.manager import _ptr, clib
    assert clib.target_manager_nearest(mgr.h, 0, None, None, None, 5, None, None, None) == 0
    c = np.full(3, 7, dtype=np.int64)
    p, r = np.zeros((3, 3)), np.array([1.0, 0.0, np.inf])   # 0 and +inf are valid radii
    assert clib.target_manager_nearest(mgr.h, 3, None, _ptr(p), _ptr(r), 0, None, None, _ptr(c)) == 0   # counts only
    assert not c.any()
    count, ids, dist = mgr.nearest([0.0, 0.1, 0.2], p, np.inf, 5)
    assert count.shape == (3,) and ids.shape == (3, 5) and dist.shape == (3, 5)
    assert not count.any() and np.all(ids == 0xFFFFFFFF) and np.all(dist == -1.0)
    count, ids, dist = mgr.nearest(None, p, 2.0, 0)
    assert ids.shape == (3, 0) and not count.any()


def test_pool_entry_rejects_a_null_pool():
    from target_estimation_b200._lib import last_error, lib
    h = np.zeros(1, dtype=np.int64)
    p = h.ctypes.data_as(C.c_void_p)
    assert lib.te_pool_nearest_targets(None, 1, p, p, p, 1, p, p, p) == -1 and "null pool" in last_error()
