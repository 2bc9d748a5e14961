"""not gpu: target_manager_gated and te_pool_gated_targets reject invalid arguments with -1 and a message, q = 0 or a manager
without targets return 0 without device work, and the nearest query's messages are unchanged by the argument rules the two
queries share."""
import ctypes as C
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def mgr():
    from target_estimation_b200.manager import TargetManagerC
    m = TargetManagerC(os.path.join(ROOT, "models", "model_uniform_acceleration_params.yaml"))
    yield m
    m.close()


def _err():
    from target_estimation_b200.manager import clib
    return clib.target_manager_last_error().decode()


def test_bad_arguments(mgr):
    from target_estimation_b200.manager import _ptr, clib
    t1, z, g = np.zeros(2), np.zeros((2, 3)), np.full(2, 11.34)
    ids, d2, c = np.zeros((2, 4), dtype=np.uint32), np.zeros((2, 4)), np.zeros(2, dtype=np.int64)
    args = [_ptr(t1), _ptr(z), _ptr(g), 4, _ptr(ids), _ptr(d2), _ptr(c)]
    assert clib.target_manager_gated(None, 2, *args) == -1 and _err() == "null manager"
    assert clib.target_manager_gated(mgr.h, -1, *args) == -1 and _err() == "q must be >= 0"
    for k in (-1, 65537):
        assert clib.target_manager_gated(mgr.h, 2, _ptr(t1), _ptr(z), _ptr(g), k, _ptr(ids), _ptr(d2), _ptr(c)) == -1
        assert _err() == "k must be in [0, 65536]"
    for i in (1, 2, 6):   # z, gate, count_out (t1 may be NULL)
        a = list(args)
        a[i] = None
        assert clib.target_manager_gated(mgr.h, 2, *a) == -1 and _err() == "z, gate and count_out are required"
    for i in (4, 5):      # ids_out, d2_out
        a = list(args)
        a[i] = None
        assert clib.target_manager_gated(mgr.h, 2, *a) == -1 and _err() == "ids_out and d2_out are required when k > 0"
    for bad in (-1.0, -1e-300, np.nan, -np.inf):
        gb = np.array([1.0, bad])
        assert clib.target_manager_gated(mgr.h, 2, _ptr(t1), _ptr(z), _ptr(gb), 4, _ptr(ids), _ptr(d2), _ptr(c)) == -1
        assert _err() == "gate must be >= 0 and not NaN (query 1)"
    with pytest.raises(RuntimeError, match="k must be"):
        mgr.gated(0.0, z, 11.34, 70000)
    with pytest.raises(RuntimeError, match="gate must be"):
        mgr.gated(None, z, -0.5, 3)


def test_nearest_messages_unchanged(mgr):
    """the nearest query words its errors as it always has: point / radius / dist_out"""
    from target_estimation_b200.manager import _ptr, clib
    p, r = np.zeros((2, 3)), np.ones(2)
    ids, d, c = np.zeros((2, 4), dtype=np.uint32), np.zeros((2, 4)), np.zeros(2, dtype=np.int64)
    assert clib.target_manager_nearest(mgr.h, 2, None, None, _ptr(r), 4, _ptr(ids), _ptr(d), _ptr(c)) == -1
    assert _err() == "point, radius and count_out are required"
    assert clib.target_manager_nearest(mgr.h, 2, None, _ptr(p), _ptr(r), 4, _ptr(ids), None, _ptr(c)) == -1
    assert _err() == "ids_out and dist_out are required when k > 0"
    rb = np.array([np.nan, 1.0])
    assert clib.target_manager_nearest(mgr.h, 2, None, _ptr(p), _ptr(rb), 4, _ptr(ids), _ptr(d), _ptr(c)) == -1
    assert _err() == "radius must be >= 0 and not NaN (query 0)"


def test_zero_queries_counts_only_and_empty_manager(mgr):
    from target_estimation_b200.manager import _ptr, clib
    assert clib.target_manager_gated(mgr.h, 0, None, None, None, 5, None, None, None) == 0
    c = np.full(3, 7, dtype=np.int64)
    z, g = np.zeros((3, 3)), np.array([11.34, 0.0, np.inf])   # 0 and +inf are valid gates
    assert clib.target_manager_gated(mgr.h, 3, None, _ptr(z), _ptr(g), 0, None, None, _ptr(c)) == 0   # counts only
    assert not c.any()
    count, ids, d2 = mgr.gated([0.0, 0.1, 0.2], z, np.inf, 5)
    assert count.shape == (3,) and ids.shape == (3, 5) and d2.shape == (3, 5)
    assert not count.any() and np.all(ids == 0xFFFFFFFF) and np.all(d2 == -1.0)
    count, ids, d2 = mgr.gated(None, z, 11.34, 0)
    assert ids.shape == (3, 0) and not count.any()


def test_pool_entry_rejects_a_null_pool():
    from target_estimation_b200._lib import last_error, lib
    h = np.zeros(1, dtype=np.int64)
    p = h.ctypes.data_as(C.c_void_p)
    assert lib.te_pool_gated_targets(None, 1, p, p, p, 1, p, p, p) == -1 and "null pool" in last_error()
