"""not gpu: target_isolver_* rejects invalid arguments with NULL / -1 / false and a message, before any device work (a plain manager
makes no device call until it holds targets)."""
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


def test_new_rejects_bad_arguments(mgr):
    from target_estimation_b200.manager import IntersectionSolverC, clib
    assert clib.target_isolver_new(None, 1, 250) is None and "null manager" in _err()
    assert clib.target_isolver_new(mgr.h, 0, 250) is None and "n_streams" in _err()
    assert clib.target_isolver_new(mgr.h, 4, 0) is None and "filters_length" in _err()
    with pytest.raises(RuntimeError, match="n_streams"):
        IntersectionSolverC(mgr, n_streams=-3)


def test_calls_reject_bad_arguments(mgr):
    from target_estimation_b200.manager import IntersectionSolverC, _ptr, clib
    s = IntersectionSolverC(mgr, n_streams=4, filters_length=10)
    origin = np.zeros(3)
    assert clib.target_isolver_get_time(None, 1, 0.0, _ptr(origin), 1.0) == -1.0 and "null solver" in _err()
    assert clib.target_isolver_query_batch(None, 1, None, None, None, None, None, None, None, None, None, None) == -1
    pose = np.zeros(7)
    assert not clib.target_isolver_get_pose(s.h, 1, 0.0, -0.1, 0.1, _ptr(origin), 1.0, _ptr(pose)) and ">= 0" in _err()
    assert not clib.target_isolver_get_pose(s.h, 1, 0.0, 0.1, 0.1, None, 1.0, _ptr(pose)) and "origin" in _err()
    with pytest.raises(RuntimeError, match="bad stream index"):
        s.query_batch([1, 2], 0.0, origin, 1.0, 0.1, 0.1, stream=[0, 4])
    with pytest.raises(RuntimeError, match="bad stream index"):
        s.query_batch([1], 0.0, origin, 1.0, 0.1, 0.1, stream=[-1])
    with pytest.raises(RuntimeError, match="more queries than solver streams"):
        s.query_batch(np.arange(5), 0.0, origin, 1.0, 0.1, 0.1)
    with pytest.raises(RuntimeError, match="bad stream index"):
        s.query_batch([1], 0.0, origin, 1.0, stream=[9], with_pose=False)
    with pytest.raises(RuntimeError, match=">= 0"):
        s.query_batch([1], -1.0, origin, 1.0, 0.1, 0.1)
    with pytest.raises(RuntimeError, match="thresholds are required"):
        s.query_batch([1], 0.0, origin, 1.0)
    ids = np.array([1], dtype=np.uint32)
    assert clib.target_isolver_query_batch(s.h, 1, _ptr(ids), None, None, None, None, None, None, None, None, None) == -1
    assert "required" in _err()
    assert clib.target_isolver_query_batch(s.h, -1, None, None, None, None, None, None, None, None, None, None) == -1
    assert clib.target_isolver_query_batch(s.h, 0, None, None, None, None, None, None, None, None, None, None) == 0
    assert clib.target_isolver_last_timing(s.h, None) == -1
    ms = np.zeros(4)
    assert clib.target_isolver_last_timing(s.h, ms.ctypes.data_as(C.c_void_p)) == 0 and not ms.any()
    s.close()
