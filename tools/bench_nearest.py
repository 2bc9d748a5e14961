#!/usr/bin/env python3
"""The k nearest targets inside a sphere at a given time (TargetManagerC.nearest / target_manager_nearest) against the brute-force
path a caller has without it: the id list, get_estimates_batch over every id, the distance in numpy and np.lexsort on the host.

Workloads: 1 Mi targets of each of the four models, falling from 15-25 m and thrown sideways as in tools/bench_sphere_sweep.py,
measured for 50 ticks; 16 query points near random targets, all at t1 = now + 50 ms ("what is in reach in 50 ms"), with a radius of
1 m (a few thousand targets inside each) and of +inf (every target is a candidate: plain k nearest); k in {100, 10 000}; plain handle
on cuda:0.  One JSON line per (model, radius, k): host clock around the synchronous call after warm-up, (target x query) pairs per
second, and the brute-force path for the same 16 queries timed in the same run with the same warm-up and calls (one read-back per
distinct t1, so one here), with whether both give the same rows.

  python tools/bench_nearest.py [--calls K] [--warmup W] [--out FILE]
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
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_sphere_sweep import DT, TICKS, falling, setup, stats  # noqa: E402

MODELS = ("uniform_acceleration", "angular_rates", "uniform_velocity", "angular_velocities")
Q = 16


def brute(mgr, t1, point, radius, k):
    """what a caller does without the query: every id, every estimate at t1, distances and a sort on the host"""
    ids = mgr.ids()
    pos = mgr.get_estimates_batch(ids, t1)[0][:, :3]
    count, out = np.zeros(point.shape[0], dtype=np.int64), []
    for j in range(point.shape[0]):
        d = pos - point[j]
        dist = np.sqrt((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2])
        inside = dist <= radius
        count[j] = int(inside.sum())
        ii, dd = ids[inside], dist[inside]
        order = np.lexsort((ii, dd))[:k]
        out.append((ii[order], dd[order]))
    return count, out


def matches(got, ref, k):
    count, ids, dist = got
    if not np.array_equal(count, ref[0]):
        return False
    for j, (ri, rd) in enumerate(ref[1]):
        ri, rd = ri[:k], rd[:k]
        m = ri.size
        if not (np.array_equal(ids[j, :m], ri) and np.array_equal(dist[j, :m].view(np.uint64), rd.view(np.uint64))
                and np.all(ids[j, m:] == 0xFFFFFFFF) and np.all(dist[j, m:] == -1.0)):
            return False
    return True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from target_estimation_b200.manager import TargetManagerC
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
    n = 1 << 20
    t1 = TICKS * DT + 0.05
    for model in MODELS:
        mgr = TargetManagerC(os.path.join(ROOT, "models", "model_%s_params.yaml" % model), device=0)
        _, p0, v = setup(mgr, n, 7)
        rng = np.random.default_rng(3)
        rows = rng.choice(n, Q, replace=False)
        point = falling(p0[rows], v[rows], t1) + rng.normal(0, 0.1, (Q, 3))
        for radius in (1.0, float("inf")):
            brute_s = []
            for c in range(a.warmup + a.calls):   # the same warm-up and calls as the query
                ta = time.perf_counter()
                ref = brute(mgr, t1, point, radius, 10000)
                tb = time.perf_counter()
                if c >= a.warmup:
                    brute_s.append(tb - ta)
            brute_ms = 1e3 * float(np.median(brute_s))
            for k in (100, 10000):
                ms = []
                for c in range(a.warmup + a.calls):
                    ta = time.perf_counter()
                    got = mgr.nearest(t1, point, radius, k)
                    tb = time.perf_counter()
                    if c >= a.warmup:
                        ms.append(tb - ta)
                line = {"bench": "nearest", "gpu": gpu, "power_limit": power, "visible_gpus": n_gpu, "model": model, "targets": n,
                        "handle": "plain", "queries": Q, "k": k, "radius": radius if np.isfinite(radius) else "inf", "calls": a.calls,
                        "ms_call": stats(ms), "pairs_per_s": n * Q / float(np.median(ms)), "count_total": int(got[0].sum()),
                        "count_per_query_mean": float(got[0].mean()), "falling_ticks": TICKS, "t1": "now + 50 ms",
                        "brute_force_ms": stats(brute_s), "speedup_vs_brute_force": brute_ms / (1e3 * float(np.median(ms))),
                        "matches_brute_force": matches(got, ref, k),
                        "note": "host clock around the synchronous call after warm-up, pageable caller arrays; brute force = id list + "
                                "get_estimates_batch over every id (one read-back: all queries share t1) + numpy distance + np.lexsort "
                                "per query, timed in this run with the same warm-up and calls; speed-up = ratio of the medians"}
                print(json.dumps(line), flush=True)
                if out:
                    out.write(json.dumps(line) + "\n"); out.flush()
        mgr.close()


if __name__ == "__main__":
    main()
