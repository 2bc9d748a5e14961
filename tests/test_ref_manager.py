"""not gpu: the oracle's TargetManager, IntersectionSolver, moving-average filters, frame-name parsing and C-ABI semantics
against the REFERENCE's own src/target_manager.cpp, src/intersection_solver.cpp, utils.hpp and src/target_manager_c.cpp,
compiled unmodified from /root/reference into oracle/_ref/libref_manager.so (oracle/Makefile; stand-ins for the absent Eigen,
yaml-cpp and ROS headers under oracle/eigen_standin -- the polynomial root finder behind the intersection solver is the
oracle's own restatement in BOTH arms, so that part pins the control flow around it, not the roots).  Skipped where neither
/root/reference nor a prebuilt oracle/_ref exists."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests import orc, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "oracle", "_ref", "libref_manager.so")
DT = 1.0 / 250.0


def _lib():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s"])
    if not os.path.exists(LIB):
        pytest.skip("needs oracle/_ref/libref_manager.so, which `make -C oracle REF=<checkout of the original target_estimation project>` "
                    "builds from the original's own sources; they are not part of this repository, and this comparison has no stored form")
    orc.lib()   # libte_oracle.so first: the stand-in polynomial solver resolves orc_poly_roots from it
    L = C.CDLL(LIB, mode=C.RTLD_GLOBAL)
    p, i, d, u, ll = C.c_void_p, C.c_int, C.c_double, C.c_uint, C.c_longlong
    L.refm_new.restype = p; L.refm_new.argtypes = [C.c_char_p]
    L.refm_delete.argtypes = [p]
    L.refm_init_full.argtypes = [p, i, u, d, d, p, i, p, i, p, p, p, p]
    L.refm_init_default.restype = i; L.refm_init_default.argtypes = [p, u, d, d, p]
    L.refm_update_meas.restype = i; L.refm_update_meas.argtypes = [p, u, d, p]
    L.refm_update.restype = i; L.refm_update.argtypes = [p, u, d]
    L.refm_update_all.argtypes = [p, d]
    L.refm_erase.restype = i; L.refm_erase.argtypes = [p, u]
    L.refm_ids.restype = i; L.refm_ids.argtypes = [p, p, i]
    L.refm_state.restype = i; L.refm_state.argtypes = [p, u, p, p, p, p]
    for f in ("refm_pose", "refm_twist", "refm_acc"):
        getattr(L, f).restype = i; getattr(L, f).argtypes = [p, u, p]
    L.refm_n_meas.restype = ll; L.refm_n_meas.argtypes = [p, u]
    L.refs_new.restype = p; L.refs_new.argtypes = [p, u]
    L.refs_delete.argtypes = [p]
    L.refs_time.restype = d; L.refs_time.argtypes = [p, u, d, p, d]
    L.refs_pose.restype = i; L.refs_pose.argtypes = [p, u, d, d, d, p, d, p]
    L.refu_mavg_new.restype = p; L.refu_mavg_new.argtypes = [u]
    L.refu_mavg_update.restype = d; L.refu_mavg_update.argtypes = [p, d]
    L.refu_mavg_variance.restype = d; L.refu_mavg_variance.argtypes = [p]
    L.refu_mavg_delete.argtypes = [p]
    L.refu_avg_new.restype = p; L.refu_avg_new.argtypes = [u]
    L.refu_avg_update.restype = d; L.refu_avg_update.argtypes = [p, d]
    L.refu_avg_delete.argtypes = [p]
    L.refu_get_id.restype = i; L.refu_get_id.argtypes = [C.c_char_p, p]
    L.refu_to_sec.restype = d; L.refu_to_sec.argtypes = [u, u]
    # the reference's own C-ABI (include/target_estimation/target_manager_c.h:28-37)
    L.target_manager_new.restype = p; L.target_manager_new.argtypes = [C.c_char_p]
    L.target_manager_init.argtypes = [p, u, d, p, d]
    L.target_manager_update_meas.argtypes = [p, u, d, p]
    L.target_manager_update.argtypes = [p, u, d]
    for f in ("target_manager_get_est_pose", "target_manager_get_est_twist", "target_manager_get_est_acceleration"):
        getattr(L, f).restype = C.c_bool; getattr(L, f).argtypes = [p, u, p]
    L.target_manager_get_n_measurements.restype = i; L.target_manager_get_n_measurements.argtypes = [p, u]
    L.target_manager_delete.argtypes = [p]
    return L


def _same(a, b):
    return np.array_equal(np.asarray(a), np.asarray(b))


def test_manager_registry_and_models_match_reference_source():
    """init (incl. the no-op on an existing id), update on a missing id, predict-all, erase, ascending ids, getters on unknown
    ids, measurement counts -- mixed model types in one manager, as the reference allows"""
    L = _lib()
    ref = L.refm_new(None); mgr = orc.Manager()
    rng = np.random.default_rng(12)
    names = ["angular_rates", "angular_velocities", "uniform_acceleration", "uniform_velocity"]
    models = {}
    for nm in names:
        y = orc.load_yaml(os.path.join(ROOT, "models", "model_%s_params.yaml" % nm))
        models[y["type"]] = y
    ids = [17, 3, 250, 8, 99, 4, 1000, 56]
    streams, _, _ = synth.make_streams(len(ids), 120, DT, accel=True, angular=True, seed=31)
    for j, id_ in enumerate(ids):
        y = models[j % 4]
        Q, R, P = y["Q"], y["R"], y["P"]
        for target in (ref, mgr):
            for rep in range(2):   # the second init of the same id must be a no-op
                p0 = streams[0, j] if rep == 0 else streams[5, j]
                if target is ref:
                    Qc, Rc, Pc = orc.colmajor(Q), orc.colmajor(R), orc.colmajor(P)
                    p0c = np.ascontiguousarray(p0)
                    L.refm_init_full(ref, j % 4, id_, DT, 0.5 * j, Qc.ctypes.data, Q.shape[0], Rc.ctypes.data, R.shape[0], Pc.ctypes.data, p0c.ctypes.data, None, None)
                else:
                    mgr.init_full(j % 4, id_, DT, 0.5 * j, Q, R, P, p0)
    out = np.zeros(64, dtype=np.uint32)
    assert L.refm_ids(ref, out.ctypes.data, 64) == len(ids) and _same(out[:len(ids)], mgr.ids()) and _same(mgr.ids(), sorted(ids))
    for t in range(1, 120):
        for j, id_ in enumerate(ids + [7777]):                      # 7777 never exists
            m = np.ascontiguousarray(streams[t, j % len(ids)])
            r = rng.random()
            if r < 0.75:
                assert bool(L.refm_update_meas(ref, id_, DT, m.ctypes.data)) == mgr.update_meas(id_, DT, m)
            elif r < 0.9:
                assert bool(L.refm_update(ref, id_, DT)) == mgr.update(id_, DT)
        if t % 25 == 0:
            L.refm_update_all(ref, DT); mgr.update_all(DT)
        if t == 60:
            for id_ in (8, 4242):
                assert bool(L.refm_erase(ref, id_)) == mgr.erase(id_)
            ids.remove(8)
        if t % 10 == 0:
            assert L.refm_ids(ref, out.ctypes.data, 64) == len(ids) and _same(out[:len(ids)], mgr.ids())
            for id_ in ids + [7777]:
                n = models[ids.index(id_) % 4]["Q"].shape[0] if id_ in ids else 18
                x, P = np.zeros(18), np.zeros(18 * 18)
                tt, nm = C.c_double(), C.c_longlong()
                nn = L.refm_state(ref, id_, x.ctypes.data, P.ctypes.data, C.byref(tt), C.byref(nm))
                if id_ not in ids:
                    assert nn == 0
                    continue
                so = mgr.state(id_, nn)
                assert _same(x[:nn], so["x"]) and _same(P[:nn * nn].reshape(nn, nn).T, so["P"]) and tt.value == so["t"] and nm.value == so["n_meas"]
                assert L.refm_n_meas(ref, id_) == so["n_meas"]
                for fn, og, k in ((L.refm_pose, mgr.pose, 7), (L.refm_twist, mgr.twist, 6), (L.refm_acc, mgr.acc, 6)):
                    o = np.zeros(k)
                    ok = fn(ref, id_, o.ctypes.data)
                    ok2, o2 = og(id_)
                    assert bool(ok) == ok2 and _same(o, o2), (fn, id_)
            assert L.refm_n_meas(ref, 7777) == mgr.L.orc_get_n_measurements(mgr.h, 7777) == 0
    L.refm_delete(ref)


def test_intersection_solver_matches_reference_source():
    L = _lib()
    ref = L.refm_new(None); mgr = orc.Manager()
    y = orc.load_yaml(os.path.join(ROOT, "models", "model_uniform_acceleration_params.yaml"))
    ya = orc.load_yaml(os.path.join(ROOT, "models", "model_angular_rates_params.yaml"))
    yv = orc.load_yaml(os.path.join(ROOT, "models", "model_uniform_velocity_params.yaml"))
    n, ticks = 6, 80
    streams, action, _ = synth.make_streams(n, ticks, DT, accel=True, angular=True, seed=2)
    for k in range(n):
        yy = (y, ya, yv)[k % 3]
        Qc, Rc, Pc = orc.colmajor(yy["Q"]), orc.colmajor(yy["R"]), orc.colmajor(yy["P"])
        p0 = np.ascontiguousarray(streams[0, k])
        L.refm_init_full(ref, yy["type"], k, DT, 0.0, Qc.ctypes.data, yy["Q"].shape[0], Rc.ctypes.data, yy["R"].shape[0], Pc.ctypes.data, p0.ctypes.data, None, None)
        mgr.init_full(yy["type"], k, DT, 0.0, yy["Q"], yy["R"], yy["P"], p0)
    rs = L.refs_new(ref, 7); os_ = orc.lib().orc_isolver_new(mgr.h, 7)
    rng = np.random.default_rng(3)
    found = conv = 0
    for t in range(1, ticks):
        for k in range(n):
            m = np.ascontiguousarray(streams[t, k])
            L.refm_update_meas(ref, k, DT, m.ctypes.data); mgr.update_meas(k, DT, m)
        for k in list(range(n)) + [99]:                 # one solver object shared by all ids (its filters too), plus an unknown id
            ok, p = mgr.pose_at(k, t * DT + 0.3) if k < n else (False, np.zeros(7))
            origin = np.ascontiguousarray(p[:3] + rng.normal(0, 0.05, 3)); radius = float(rng.uniform(0.1, 0.5)); t1 = t * DT
            d_ref = L.refs_time(rs, k, t1, origin.ctypes.data, radius)
            d_orc = orc.lib().orc_isolver_time(os_, k, t1, orc.ptr(origin), radius)
            assert d_ref == d_orc, (t, k, d_ref, d_orc)
            pr, po = np.zeros(7), np.zeros(7)
            c_ref = L.refs_pose(rs, k, t1, 0.05, 0.1, origin.ctypes.data, radius, pr.ctypes.data)
            c_orc = orc.lib().orc_isolver_pose(os_, k, t1, 0.05, 0.1, orc.ptr(origin), radius, orc.ptr(po))
            assert c_ref == c_orc and _same(pr, po), (t, k)
            found += d_ref >= 0; conv += c_ref
    assert found > 50          # the accelerating models do intercept; the uniform-velocity ones never do (t^4 coefficient 0)
    L.refs_delete(rs); orc.lib().orc_isolver_delete(os_); L.refm_delete(ref)


def test_utils_filters_ids_stamps_match_reference_source():
    L = _lib(); O = orc.lib()
    rng = np.random.default_rng(4)
    for n in (1, 5, 250):
        a, b = L.refu_mavg_new(n), O.orc_mavg_new(n)
        c, d = L.refu_avg_new(n), O.orc_avg_new(n)
        for v in rng.normal(5, 1, 3 * n + 7):
            assert L.refu_mavg_update(a, float(v)) == O.orc_mavg_update(b, float(v))
            assert L.refu_mavg_variance(a) == O.orc_mavg_variance(b)
            assert L.refu_avg_update(c, float(v)) == O.orc_avg_update(d, float(v))
        L.refu_mavg_delete(a); O.orc_mavg_delete(b); L.refu_avg_delete(c); O.orc_avg_delete(d)
    for s in ("target_7", "target_007", "target_", "target", "target_filt_3", "a_b_c", "x_-4", "x_12abc", "obj_4294967295", "obj_99999999999", "_5", "t_ 6"):
        i1, i2 = C.c_uint(0), C.c_uint(0)
        assert L.refu_get_id(s.encode(), C.byref(i1)) == O.orc_get_id(s.encode(), C.byref(i2)) and i1.value == i2.value, s
    for sec, nsec in ((0, 0), (1000, 4000000), (1639654196, 354783181), (4294967295, 999999999)):
        assert L.refu_to_sec(sec, nsec) == O.orc_to_sec(sec, nsec)


def test_reference_c_abi_matches_oracle_c_abi_semantics():
    """the reference's own extern "C" wrapper (src/target_manager_c.cpp): defaults from the YAML file, stale scratch on unknown
    ids, n_measurements truncated to int"""
    L = _lib()
    path = os.path.join(ROOT, "models", "model_uniform_acceleration_params.yaml")
    ref = L.target_manager_new(path.encode())
    mgr = orc.Manager(path)
    streams, _, _ = synth.make_streams(3, 40, DT, accel=True, angular=False, seed=6)
    for k in range(3):
        p0 = np.ascontiguousarray(streams[0, k])
        L.target_manager_init(ref, 10 + k, DT, p0.ctypes.data, 0.0)
        assert mgr.L.orc_init_default(mgr.h, 10 + k, DT, orc.ptr(p0), 0.0)
    last = {}
    for t in range(1, 40):
        for k in range(3):
            m = np.ascontiguousarray(streams[t, k])
            if (t + k) % 5:
                L.target_manager_update_meas(ref, 10 + k, DT, m.ctypes.data); mgr.update_meas(10 + k, DT, m)
            else:
                L.target_manager_update(ref, 10 + k, DT); mgr.update(10 + k, DT)
        for id_ in (10, 11, 12):
            for fn, og, kk in ((L.target_manager_get_est_pose, mgr.pose, 7), (L.target_manager_get_est_twist, mgr.twist, 6),
                               (L.target_manager_get_est_acceleration, mgr.acc, 6)):
                o = np.zeros(kk)
                assert fn(ref, id_, o.ctypes.data) and _same(o, og(id_)[1])
                last[fn.__name__] = o.copy()
            assert L.target_manager_get_n_measurements(ref, id_) == mgr.state(id_, 9)["n_meas"]
        # unknown id: false, and the output receives the previous value of the file-static scratch (src/target_manager_c.cpp:8-9,39-42)
        o = np.full(7, -1.0)
        assert not L.target_manager_get_est_pose(ref, 555, o.ctypes.data)
        assert _same(o, last["target_manager_get_est_pose"])
        assert L.target_manager_get_n_measurements(ref, 555) == 0
    L.target_manager_delete(ref)


@pytest.mark.parametrize("name", ["uniform_velocity", "uniform_acceleration", "angular_rates", "angular_velocities"])
def test_cpu_baseline_loops_agree(name):
    """bench.py's two CPU arms (orc_bench_steps on the port, refm_bench_steps on the reference's own sources) run the same
    workload: the checksum over every target's final estimated position must be bit-identical, for 1 and 3 threads"""
    L = _lib(); O = orc.lib()
    y = orc.load_yaml(os.path.join(ROOT, "models", "model_%s_params.yaml" % name))
    L.refm_bench_steps.restype = C.c_double; L.refm_bench_steps.argtypes = O.orc_bench_steps.argtypes
    n_t = 60
    rng = np.random.default_rng(5)
    meas = np.zeros((n_t, 7)); meas[:, :3] = rng.uniform(-5, 5, (n_t, 3)); meas[:, 6] = 1.0
    Qc, Rc, Pc = orc.colmajor(y["Q"]), orc.colmajor(y["R"]), orc.colmajor(y["P"])
    for threads in (1, 3):
        c1, c2 = C.c_double(), C.c_double()
        a = (y["type"], orc.ptr(Qc), y["Q"].shape[0], orc.ptr(Rc), y["R"].shape[0], orc.ptr(Pc), n_t, 25, threads, DT, orc.ptr(meas), 0.05)
        assert L.refm_bench_steps(*a, C.byref(c1)) > 0 and O.orc_bench_steps(*a, C.byref(c2)) > 0
        assert c1.value == c2.value and np.isfinite(c1.value)


def test_write_txt_file_matches_reference_source(tmp_path):
    """target_write_txt_file (host library; what TargetManager::writeLog uses) against the reference's own writeTxtFile
    (utils.hpp:78-120, both overloads) byte for byte -- default ostream formatting of awkward values included.  No GPU: the
    host library loads and this entry point does not touch CUDA."""
    L = _lib()
    so = os.path.join(ROOT, "target_estimation_b200", "lib", "libtarget_c.so")
    if not os.path.exists(so):
        pytest.skip("libtarget_c.so not built")
    H = C.CDLL(so)
    H.target_write_txt_file.restype = C.c_int
    H.target_write_txt_file.argtypes = [C.c_char_p, C.c_void_p, C.c_longlong, C.c_longlong]
    L.refu_write_txt_vec.argtypes = [C.c_char_p, C.c_void_p, C.c_int]
    L.refu_write_txt_mat.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_int]
    rng = np.random.default_rng(6)
    vals = np.concatenate([rng.normal(0, 1, 40), rng.normal(0, 1e-7, 10), rng.normal(0, 1e9, 10),
                           [0.0, -0.0, 1.0, 1e-5, 123456.7, 1234567.8, 0.1 + 0.2, 1.0 / 3.0, np.inf, -np.inf, np.nan, 5e-324]])
    a, b = str(tmp_path / "a"), str(tmp_path / "b")
    L.refu_write_txt_vec(a.encode(), vals.ctypes.data, vals.size)
    assert H.target_write_txt_file(b.encode(), vals.ctypes.data, vals.size, 1) == 1
    assert open(a, "rb").read() == open(b, "rb").read() and os.path.getsize(a) > 300
    m = np.ascontiguousarray(vals.reshape(12, 6))
    L.refu_write_txt_mat(a.encode(), m.ctypes.data, 12, 6)
    assert H.target_write_txt_file(b.encode(), m.ctypes.data, 12, 6) == 1
    assert open(a, "rb").read() == open(b, "rb").read()
    assert open(b).read().splitlines()[0].endswith(" ")        # "value " per column, then the newline
    assert H.target_write_txt_file(str(tmp_path / "no" / "dir").encode(), m.ctypes.data, 2, 6) == 0
