"""not gpu: the oracle's target models against the REFERENCE's own src/types/*.cpp + src/target_interface.cpp + src/kalman.cpp
(with geometry.hpp / utils.hpp), compiled unmodified from /root/reference into oracle/_ref/libref_models.so (oracle/Makefile;
Eigen itself is absent from the image, so the files are compiled against the stand-in oracle/eigen_standin/Eigen/Dense).
Reference objects (TargetUniformVelocity / ...Acceleration / AngularRates / AngularVelocities) and the oracle's TargetManager
receive the same constructor arguments and the same addMeasurement / update calls; filter state, covariance, time, measurement
count and the derived outputs (getEstimatedPose / Twist / Acceleration, current and extrapolated to t1) are compared after
every tick.  Pins rows a7-a12 of SURVEY.md section 8 -- A(dt), measurement conversion (quaternion -> rpy -> unwrap), EKF f / h /
Jacobians, updateTargetState, the extrapolating getters, bookkeeping -- to the reference source; Eigen's own rounding is not
pinned (DESIGN.md section 3).  Skipped where neither /root/reference nor a prebuilt oracle/_ref exists."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests import orc, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "oracle", "_ref", "libref_models.so")
DT = 1.0 / 250.0


def _lib():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s"])
    if not os.path.exists(LIB):
        pytest.skip("needs oracle/_ref/libref_models.so, which `make -C oracle REF=<checkout of the original target_estimation project>` "
                    "builds from the original's own sources; they are not part of this repository, and this comparison has no stored form")
    L = C.CDLL(LIB)
    p, i, d, u = C.c_void_p, C.c_int, C.c_double, C.c_uint
    L.ref_target_new.restype = p; L.ref_target_new.argtypes = [i, u, d, d, p, i, p, i, p, p, p, p]
    L.ref_target_delete.argtypes = [p]
    L.ref_target_add_measurement.argtypes = [p, d, p]
    L.ref_target_update.argtypes = [p, d]
    L.ref_target_state.restype = i; L.ref_target_state.argtypes = [p, p, p, p, p]
    L.ref_target_estimates.argtypes = [p, i, d, p, p, p]
    return L


def _rel(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / max(1e-300, np.abs(np.asarray(b)).max()))


def _qrel(a, b):   # quaternions up to sign
    return min(_rel(a, b), _rel(-np.asarray(a), b))


@pytest.mark.parametrize("name", ["uniform_velocity", "uniform_acceleration", "angular_rates", "angular_velocities"])
def test_oracle_models_match_reference_sources(name):
    L = _lib()
    y_ = orc.load_yaml(os.path.join(ROOT, "models", "model_%s_params.yaml" % name))
    mtype, Q, R, P0 = y_["type"], y_["Q"], y_["R"], y_["P"]
    N, M = Q.shape[0], R.shape[0]
    n, ticks = 6, 400
    meas, action, scale = synth.make_streams(n, ticks, DT, accel=name in ("uniform_acceleration", "angular_rates"), angular=M == 6, seed=91)
    rng = np.random.default_rng(5)
    mgr = orc.Manager()
    worst = {"x": 0.0, "P": 0.0, "pose": 0.0, "twist": 0.0, "acc": 0.0, "pose_t1": 0.0, "twist_t1": 0.0}
    for k in range(n):
        v0 = rng.normal(0, 0.1, 6) if k % 2 else None      # the full constructor honours v0 / a0
        a0 = rng.normal(0, 0.1, 6) if k % 3 == 0 else None
        t0 = 0.25 * k
        Pk = scale[k] * P0
        mgr.init_full(mtype, k, DT, t0, Q, R, Pk, meas[0, k], v0, a0)
        Qc, Rc, Pc = orc.colmajor(Q), orc.colmajor(R), orc.colmajor(Pk)
        p0 = np.ascontiguousarray(meas[0, k])
        h = L.ref_target_new(mtype, k, DT, t0, Qc.ctypes.data, N, Rc.ctypes.data, M, Pc.ctypes.data, p0.ctypes.data,
                             None if v0 is None else np.ascontiguousarray(v0).ctypes.data, None if a0 is None else np.ascontiguousarray(a0).ctypes.data)
        assert h
        xr, Pr = np.zeros(N), np.zeros((N, N), order="F")
        tr, nr = C.c_double(), C.c_longlong()
        pose, twist, acc = np.zeros(7), np.zeros(6), np.zeros(6)
        for t in range(ticks + 1):
            if t > 0:
                act = int(action[t - 1, k])
                if act == 2:
                    m = np.ascontiguousarray(meas[t - 1, k])
                    mgr.update_meas(k, DT, m); L.ref_target_add_measurement(h, DT, m.ctypes.data)
                elif act == 1:
                    mgr.update(k, DT); L.ref_target_update(h, DT)
                else:
                    continue
            so = mgr.state(k, N)
            L.ref_target_state(h, xr.ctypes.data, Pr.ctypes.data, C.byref(tr), C.byref(nr))
            worst["x"] = max(worst["x"], _rel(xr, so["x"])); worst["P"] = max(worst["P"], _rel(np.asarray(Pr), so["P"]))
            assert tr.value == so["t"] and nr.value == so["n_meas"], (name, k, t)
            L.ref_target_estimates(h, 0, 0.0, pose.ctypes.data, twist.ctypes.data, acc.ctypes.data)
            worst["pose"] = max(worst["pose"], _rel(pose[:3], mgr.pose(k)[1][:3]), _qrel(pose[3:], mgr.pose(k)[1][3:]))
            worst["twist"] = max(worst["twist"], _rel(twist, mgr.twist(k)[1]))
            if np.abs(acc).max() > 0 or np.abs(mgr.acc(k)[1]).max() > 0:
                worst["acc"] = max(worst["acc"], _rel(acc, mgr.acc(k)[1]))
            if t % 7 == 0:
                t1 = so["t"] + 0.13
                L.ref_target_estimates(h, 1, t1, pose.ctypes.data, twist.ctypes.data, acc.ctypes.data)
                worst["pose_t1"] = max(worst["pose_t1"], _rel(pose[:3], mgr.pose_at(k, t1)[1][:3]), _qrel(pose[3:], mgr.pose_at(k, t1)[1][3:]))
                worst["twist_t1"] = max(worst["twist_t1"], _rel(twist, mgr.twist_at(k, t1)[1]))
        L.ref_target_delete(h)
    print("worst relative deviation oracle vs reference sources (%s): %s" % (name, {k_: "%.2g" % v for k_, v in worst.items()}))
    # same operand order and the same stand-in rules as the oracle assumes of Eigen: agreement at rounding level
    assert max(worst.values()) <= 1e-12, worst
