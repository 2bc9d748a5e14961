"""not gpu: target_manager_associate and the pool entries of the association reject every argument error of the contract with -1
and a message and apply nothing; q = 0 and a manager without targets return 0 without device work."""
import ctypes as C
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NO_ID = 0xFFFFFFFF


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
    det = np.zeros((2, 7))
    ids, d2, c = np.full(2, 5, dtype=np.uint32), np.full(2, 5.0), np.full(2, 5, dtype=np.int64)

    def call(h=mgr.h, t1=0.0, q=2, d=_ptr(det), gate=11.34, K=4, apply=1, i=_ptr(ids), o=_ptr(d2), cnt=_ptr(c)):
        return clib.target_manager_associate(h, t1, q, d, gate, K, apply, i, o, cnt)
    assert call(h=None) == -1 and _err() == "null manager"
    for t1 in (np.nan, np.inf, -np.inf):
        assert call(t1=t1) == -1 and _err() == "t1 must be finite"
    for gate in (-1.0, -1e-300, np.nan, np.inf, -np.inf):
        assert call(gate=gate) == -1 and _err() == "gate must be >= 0 and finite"
    for K in (0, -1, 33, 1 << 20):
        assert call(K=K) == -1 and _err() == "K must be in [1, 32]"
    assert call(q=-1) == -1 and _err() == "q must be >= 0"
    for kw in ({"d": None}, {"i": None}, {"o": None}):
        assert call(**kw) == -1 and _err() == "det, id_out and d2_out are required"
    # nothing was written
    assert np.all(ids == 5) and np.all(d2 == 5.0) and np.all(c == 5)
    with pytest.raises(RuntimeError, match="K must be"):
        mgr.associate(0.0, det, 11.34, 0)
    with pytest.raises(RuntimeError, match="gate must be"):
        mgr.associate(0.0, det, np.inf, 4, apply=True)


def test_zero_detections_and_empty_manager(mgr):
    from target_estimation_b200.manager import _ptr, clib
    assert clib.target_manager_associate(mgr.h, 0.0, 0, None, 11.34, 4, 1, None, None, None) == 0
    det = np.zeros((3, 7))
    ids, d2, count = mgr.associate(1.0, det, 0.0, 32, apply=True)   # 0 is a valid gate
    assert np.all(ids == NO_ID) and np.all(d2 == -1.0) and not count.any()
    ids, d2 = np.zeros(3, dtype=np.uint32), np.zeros(3)
    assert clib.target_manager_associate(mgr.h, 1.0, 3, _ptr(det), 1.0, 1, 0, _ptr(ids), _ptr(d2), None) == 0   # count_out may be NULL
    assert np.all(ids == NO_ID)


def test_pool_entries_reject_a_null_pool_and_bad_rows():
    from target_estimation_b200._lib import last_error, lib
    h = np.zeros(64, dtype=np.float64)
    p = h.ctypes.data_as(C.c_void_p)
    assert lib.te_pool_associate(None, 0.0, 1, p, 1.0, 4, 0, p, p, p) == -1 and "null pool" in last_error()
    assert lib.te_pool_gated_candidates(None, 0.0, 1, p, 1.0, 4, p, p, p) == -1 and "null pool" in last_error()
    assert lib.te_assign_greedy(None, 1, 4, p, p, p, p) == -1 and "null pool" in last_error()
    assert lib.te_pool_update_at(None, 1, p, 0.0, p) == -1 and "null pool" in last_error()
