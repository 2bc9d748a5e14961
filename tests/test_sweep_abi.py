"""not gpu: target_isolver_earliest and te_pool_earliest_intersections reject invalid arguments with -1 and a message, and q = 0 or a
manager without targets return 0 without device work (a plain manager makes no device call until it holds targets)."""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def solver():
    from target_estimation_b200.manager import IntersectionSolverC, TargetManagerC
    m = TargetManagerC(os.path.join(ROOT, "models", "model_uniform_acceleration_params.yaml"))
    s = IntersectionSolverC(m, n_streams=1, filters_length=10)
    yield s
    s.close()
    m.close()


def _err():
    from target_estimation_b200.manager import clib
    return clib.target_manager_last_error().decode()


def test_bad_arguments(solver):
    from target_estimation_b200.manager import _ptr, clib
    t1, o, r = np.zeros(2), np.zeros((2, 3)), np.ones(2)
    ids, d, h = np.zeros((2, 4), dtype=np.uint32), np.zeros((2, 4)), np.zeros(2, dtype=np.int64)
    args = [_ptr(t1), _ptr(o), _ptr(r), 4, _ptr(ids), _ptr(d), _ptr(h)]
    assert clib.target_isolver_earliest(None, 2, *args) == -1 and "null solver" in _err()
    assert clib.target_isolver_earliest(solver.h, -1, *args) == -1 and "q must be" in _err()
    for k in (-1, 65537):
        assert clib.target_isolver_earliest(solver.h, 2, _ptr(t1), _ptr(o), _ptr(r), k, _ptr(ids), _ptr(d), _ptr(h)) == -1
        assert "k must be" in _err()
    for i in range(3):   # t1, origin, radius
        a = list(args)
        a[i] = None
        assert clib.target_isolver_earliest(solver.h, 2, *a) == -1 and "required" in _err()
    for i in (4, 5, 6):   # ids_out, delta_out, hits_out
        a = list(args)
        a[i] = None
        assert clib.target_isolver_earliest(solver.h, 2, *a) == -1 and "required" in _err()
    with pytest.raises(RuntimeError, match="k must be"):
        solver.earliest(0.0, o, 1.0, 70000)


def test_zero_spheres_and_empty_manager(solver):
    from target_estimation_b200.manager import _ptr, clib
    assert clib.target_isolver_earliest(solver.h, 0, None, None, None, 5, None, None, None) == 0
    h = np.full(3, 7, dtype=np.int64)
    o = np.zeros((3, 3))
    t1, r = np.zeros(3), np.ones(3)
    assert clib.target_isolver_earliest(solver.h, 3, _ptr(t1), _ptr(o), _ptr(r), 0, None, None, _ptr(h)) == 0   # counts only
    assert not h.any()
    hits, ids, delta = solver.earliest([0.0, 0.1, 0.2], o, 1.0, 5)
    assert hits.shape == (3,) and ids.shape == (3, 5) and delta.shape == (3, 5)
    assert not hits.any() and np.all(ids == 0xFFFFFFFF) and np.all(delta == -1.0)


def test_pool_entry_rejects_a_null_pool():
    import ctypes as C
    from target_estimation_b200._lib import last_error, lib
    h = np.zeros(1, dtype=np.int64)
    p = h.ctypes.data_as(C.c_void_p)
    assert lib.te_pool_earliest_intersections(None, 1, p, p, p, 1, p, p, p) == -1 and "null pool" in last_error()
