"""not gpu: the oracle's Kalman-filter restatement against the REFERENCE's own src/kalman.cpp, compiled unmodified from
/root/reference into oracle/_ref/libref_kalman.so (oracle/Makefile; Eigen itself is absent from the image, so the file is
compiled against the stand-in oracle/eigen_standin/Eigen/Dense, which supplies the dozen MatrixXd / VectorXd operations it
uses with the evaluation rules the oracle assumes of Eigen).  The reference classes are driven exactly as src/types/*.cpp
drive them -- update(y, A(dt)) / update(A(dt)), EKF with f, h and the Jacobian at the previous posterior -- on the same seeded
streams as the oracle's TargetManager path, and state + covariance are compared after every tick.  This pins the
restatement's control flow, operand order and update formulas to the reference source; Eigen's own rounding is not pinned
(DESIGN.md section 3).  Skipped where neither /root/reference nor a prebuilt oracle/_ref exists."""
import ctypes as C
import importlib.util
import os
import subprocess

import numpy as np
import pytest

from tests import orc, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "oracle", "_ref", "libref_kalman.so")
DT = 1.0 / 250.0
VECFN = C.CFUNCTYPE(None, C.POINTER(C.c_double), C.c_int, C.POINTER(C.c_double), C.c_int, C.c_void_p)


def _golden():
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(ROOT, "tests", "golden", "make_golden.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _lib():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s"])
    if not os.path.exists(LIB):
        pytest.skip("needs oracle/_ref/libref_kalman.so, which `make -C oracle REF=<checkout of the original target_estimation project>` "
                    "builds from the original's own sources; they are not part of this repository, and this comparison has no stored form")
    L = C.CDLL(LIB)
    p, i = C.c_void_p, C.c_int
    L.ref_lkf_new.restype = p; L.ref_lkf_new.argtypes = [p, p, p, p, p, i, i]
    L.ref_ekf_new.restype = p; L.ref_ekf_new.argtypes = [VECFN, VECFN, p, p, p, p, p, p, i, i]
    L.ref_kf_delete.argtypes = [p]
    L.ref_kf_init.argtypes = [p, p]
    L.ref_kf_update_meas.restype = i; L.ref_kf_update_meas.argtypes = [p, p, p]
    L.ref_kf_update.restype = i; L.ref_kf_update.argtypes = [p, p]
    L.ref_kf_get.argtypes = [p, p, p]
    return L


def _cm(a):   # column-major copy, as Eigen::MatrixXd stores
    return np.asfortranarray(a, dtype=np.float64)


@pytest.mark.parametrize("name", ["uniform_velocity", "uniform_acceleration", "angular_rates", "angular_velocities"])
def test_oracle_filter_matches_reference_kalman_source(name):
    L, g = _lib(), _golden()
    y_ = orc.load_yaml(os.path.join(ROOT, "models", "model_%s_params.yaml" % name))
    mtype, Q, R, P0 = y_["type"], y_["Q"], y_["R"], y_["P"]
    N, M = Q.shape[0], R.shape[0]
    n, ticks = 6, 250
    meas, action, scale = synth.make_streams(n, ticks, DT, accel=name in ("uniform_acceleration", "angular_rates"), angular=M == 6, seed=77)
    Cm = np.hstack([np.eye(M), np.zeros((M, N - M))])
    mgr = orc.Manager()
    worst = 0.0
    for k in range(n):
        mgr.init_full(mtype, k, DT, 0.0, Q, R, scale[k] * P0, meas[0, k])
        s0 = mgr.state(k, N)
        # the model's A(dt), f, h exactly as the numpy restatement of tests/golden builds them (src/types/*.cpp updateA / f / h)
        filt = g.Filter(name, Q, R, scale[k] * P0, meas[0, k])
        filt.x = s0["x"].copy()
        keep = []
        if name == "angular_velocities":
            def f_cb(xp, nn, outp, no, ctx, filt=filt):
                x = np.ctypeslib.as_array(xp, shape=(nn,)).copy()
                saved = filt.x
                filt.x = x
                out = filt.f(DT)
                filt.x = saved
                for i in range(no):
                    outp[i] = out[i]

            def h_cb(xp, nn, outp, no, ctx):
                for i in range(no):
                    outp[i] = xp[i]
            f_c, h_c = VECFN(f_cb), VECFN(h_cb)
            keep += [f_c, h_c]
            A0 = _cm(filt.A(DT)); C0 = _cm(Cm); Q0 = _cm(Q); R0 = _cm(R); Pp = _cm(scale[k] * P0)
            h = L.ref_ekf_new(f_c, h_c, None, A0.ctypes.data, C0.ctypes.data, Q0.ctypes.data, R0.ctypes.data, Pp.ctypes.data, N, M)
        else:
            A0 = _cm(filt.A(DT)); C0 = _cm(Cm); Q0 = _cm(Q); R0 = _cm(R); Pp = _cm(scale[k] * P0)
            h = L.ref_lkf_new(A0.ctypes.data, C0.ctypes.data, Q0.ctypes.data, R0.ctypes.data, Pp.ctypes.data, N, M)
        x0 = np.ascontiguousarray(s0["x"])
        L.ref_kf_init(h, x0.ctypes.data)
        xr, Pr = np.zeros(N), np.zeros((N, N), order="F")
        for t in range(ticks):
            act = int(action[t, k])
            if act == 0:
                continue
            L.ref_kf_get(h, xr.ctypes.data, Pr.ctypes.data)
            filt.x = xr.copy()                      # A (and f) are evaluated at the previous posterior (angular_velocities.cpp:84,108)
            A = _cm(filt.A(DT))
            if act == 2:
                mgr.update_meas(k, DT, meas[t, k])
                so = mgr.state(k, N)
                y = np.ascontiguousarray(np.concatenate([meas[t, k, :3], so["prev_rpy"]]) if M == 6 else meas[t, k, :3].copy())
                assert L.ref_kf_update_meas(h, y.ctypes.data, A.ctypes.data) == 0
            else:
                mgr.update(k, DT)
                so = mgr.state(k, N)
                assert L.ref_kf_update(h, A.ctypes.data) == 0
            L.ref_kf_get(h, xr.ctypes.data, Pr.ctypes.data)
            ex = np.abs(xr - so["x"]).max() / max(1e-300, np.abs(so["x"]).max())
            eP = np.abs(np.asarray(Pr) - so["P"]).max() / np.abs(so["P"]).max()
            worst = max(worst, ex, eP)
        L.ref_kf_delete(h)
    # same operand order, same LU inverse: agreement at rounding level (the AV Jacobian comes from numpy's trig, a few ulp)
    print("worst relative deviation oracle vs reference kalman.cpp (%s): %.3g" % (name, worst))
    assert worst <= 1e-12, worst
