#!/usr/bin/env python3
"""The k earliest sphere intercepts over every target (IntersectionSolverC.earliest / target_isolver_earliest) against the brute-force
path a caller has without it: a times-only target_isolver_query_batch over every id for every sphere, then np.lexsort on the host.

Workloads: 1 Mi and 4 Mi uniform-acceleration targets and 1 Mi angular-rates targets, falling from 15-25 m as in
tools/bench_isolver_handles.py, here thrown sideways and measured for 50 ticks, so that every target has settled on its acceleration;
spheres of 1 m on the future paths of random targets, so that a fraction of a percent to a few percent of the targets reach each.  q in {1, 16, 64} spheres per call, k in {100, 10 000}, on a plain handle and on 8 shards on
cuda:0.  One JSON line per (workload, handle, q, k): host clock around the synchronous call after warm-up, (target x sphere) pairs per
second, and the brute-force path of the same q measured in the same run on the plain handle (with whether both give the same rows).

  python tools/bench_sphere_sweep.py [--calls K] [--warmup W] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
DT = 1.0 / 250.0
TICKS = 50


def stats(v):
    v = 1e3 * np.asarray(v)
    return {"mean": float(v.mean()), "median": float(np.median(v)), "worst": float(v.max())}


def falling(p0, v, t):
    p = p0 + v * t
    p[:, 2] -= 0.5 * 9.81 * t * t
    return p


def setup(mgr, n, seed):
    """targets thrown sideways from 15-25 m and falling; returns ids, start positions and velocities"""
    rng = np.random.default_rng(seed)
    ids = np.arange(n, dtype=np.uint32)
    p0 = rng.uniform(-5, 5, (n, 3)); p0[:, 2] += 20.0
    v = rng.uniform(-2, 2, (n, 3)); v[:, 2] = 0.0
    m = np.zeros((n, 7)); m[:, 6] = 1.0
    m[:, :3] = p0
    assert mgr.init_batch(ids, DT, m) == n
    for k in range(1, TICKS + 1):                           # falling measurements: every target has settled on its acceleration
        m[:, :3] = falling(p0, v, k * DT)
        assert mgr.update_batch(ids, DT, m) == n
    return ids, p0, v


def spheres(p0, v, q, seed):
    """q spheres of radius 1 m on the paths of random targets, 0.3 s ahead: the targets that pass within 1 m of those points reach
    them.  (The lateral motion matters: the reference takes the smallest real root, and the parabola of a target falling straight
    down crosses a sphere below it at a negative time too, which makes the answer -1.)"""
    rng = np.random.default_rng(seed)
    rows = rng.choice(p0.shape[0], q, replace=False)
    return falling(p0[rows], v[rows], TICKS * DT + 0.3) + rng.normal(0, 0.1, (q, 3)), np.full(q, 1.0)


def brute(solver, ids, t1, origin, radius, k):
    hits, out = np.zeros(origin.shape[0], dtype=np.int64), []
    for j in range(origin.shape[0]):
        _, d, _, _ = solver.query_batch(ids, t1, origin[j], radius[j], with_pose=False)
        hit = d >= 0
        hits[j] = int(hit.sum())
        ii, dd = ids[hit], d[hit]
        order = np.lexsort((ii, dd))[:k]
        out.append((ii[order], dd[order]))
    return hits, out


def matches(got, ref):
    hits, ids, delta = got
    if not np.array_equal(hits, ref[0]):
        return False
    for j, (ri, rd) in enumerate(ref[1]):
        m = ri.size
        if not (np.array_equal(ids[j, :m], ri) and np.array_equal(delta[j, :m].view(np.uint64), rd.view(np.uint64))):
            return False
    return True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from target_estimation_b200.manager import IntersectionSolverC, ShardedManagerC, TargetManagerC
    n_gpu = torch.cuda.device_count()
    if n_gpu == 0:
        raise SystemExit("no CUDA device: this measurement needs a GPU")
    gpu = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                               timeout=30).stdout.split("\n")[0].strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    out = open(a.out, "a") if a.out else None
    t1 = TICKS * DT
    for model, n in (("uniform_acceleration", 1 << 20), ("uniform_acceleration", 4 << 20), ("angular_rates", 1 << 20)):
        yaml = os.path.join(ROOT, "models", "model_%s_params.yaml" % model)
        brute_ms = {}
        for handle in ("plain", "8 shards on cuda:0"):
            mgr = TargetManagerC(yaml, device=0) if handle == "plain" else ShardedManagerC(yaml, 8, [0] * 8)
            ids, p0, v = setup(mgr, n, 7)
            s = IntersectionSolverC(mgr, 1, 10)
            for q in (1, 16, 64):
                origin, radius = spheres(p0, v, q, q)
                ref = None
                if handle == "plain":
                    ta = time.perf_counter()
                    ref = brute(s, ids, t1, origin, radius, 10000)
                    brute_ms[q] = 1e3 * (time.perf_counter() - ta)
                for k in (100, 10000):
                    ms = []
                    for c in range(a.warmup + a.calls):
                        ta = time.perf_counter()
                        got = s.earliest(t1, origin, radius, k)
                        tb = time.perf_counter()
                        if c >= a.warmup:
                            ms.append(tb - ta)
                    line = {"bench": "sphere_sweep", "gpu": gpu, "power_limit": power, "visible_gpus": n_gpu, "model": model, "targets": n,
                            "handle": handle, "spheres": q, "k": k, "calls": a.calls, "ms_call": stats(ms),
                            "pairs_per_s": n * q / float(np.median(ms)), "hits_total": int(got[0].sum()),
                            "hits_per_sphere_mean": float(got[0].mean()), "falling_ticks": TICKS,
                            "brute_force_ms_plain": brute_ms[q], "speedup_vs_brute_force": brute_ms[q] / (1e3 * float(np.median(ms))),
                            "note": "host clock around the synchronous call after warm-up, pageable caller arrays; brute force = times-only "
                                    "query_batch over every id per sphere + np.lexsort, measured once on the plain handle in this run"}
                    if ref is not None:
                        line["matches_brute_force"] = matches(got, (ref[0], [(i[:k], d[:k]) for i, d in ref[1]]))
                    print(json.dumps(line), flush=True)
                    if out:
                        out.write(json.dumps(line) + "\n"); out.flush()
            s.close(); mgr.close()


if __name__ == "__main__":
    main()
