#!/usr/bin/env python3
"""Gating: the k targets with the smallest Mahalanobis distance to a measured position (TargetPool.gated_targets /
te_pool_gated_targets, the call every manager handle runs per pool) against the brute-force path a caller has without it: every
covariance and time read back in one batched call (te_pool_read_state -- a manager offers only target_manager_get_state, one id
and one device sync at a time, so this is the cheapest brute force there is), every position at t1 (read_estimates), the
contract's C, S, Cholesky factor and d^2 in numpy, and np.lexsort on the host.

Workloads: 1 Mi targets of each of the four models over 8 dense random SPD classes (interleaved: every warp holds all 8), falling
from 15-25 m and thrown sideways as in tools/bench_sphere_sweep.py, measured for 50 ticks; 16 measured positions a few millimetres
from random targets, all at t1 = now + 50 ms; gates of 11.34 (the 99 % chi-square quantile for 3 degrees of freedom: a handful of
targets inside each) and +inf (every target with a factor is a candidate); k in {100, 10 000}; cuda:0.  One JSON line per (model,
gate, k): host clock around the synchronous call after warm-up, (target x query) pairs per second, and the brute force for the
same 16 queries timed in the same run (1 warm-up, 3 calls: it reads back up to 2.7 GB per call), with whether both give the same
rows bit for bit.

  python tools/bench_gate.py [--calls K] [--warmup W] [--out FILE]
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
from bench_sphere_sweep import DT, TICKS, falling, stats  # noqa: E402
from tests.test_gpu_gate import CHI2, brute_pool, dense_classes, same  # noqa: E402

MODELS = ("uniform_acceleration", "angular_rates", "uniform_velocity", "angular_velocities")
Q = 16
N_CLS = 8


def setup(name, n, seed):
    """a pool of n falling targets over N_CLS dense classes after TICKS measured ticks"""
    import target_estimation_b200 as te
    Qc, Rc, P0c = dense_classes(name, N_CLS, seed)
    pool = te.TargetPool(name, device=0)
    for c in range(N_CLS):
        pool.register_class(Qc[c], Rc[c], P0c[c])
    rng = np.random.default_rng(seed)
    ids = np.arange(n, dtype=np.uint32)
    cls = np.arange(n) % N_CLS
    p0 = rng.uniform(-5, 5, (n, 3)); p0[:, 2] += 20.0
    v = rng.uniform(-2, 2, (n, 3)); v[:, 2] = 0.0
    m = np.zeros((n, 7)); m[:, 6] = 1.0
    m[:, :3] = p0
    pool.add(ids, m, cls=cls)
    for k in range(1, TICKS + 1):
        m[:, :3] = falling(p0, v, k * DT) + rng.normal(0, 0.002, (n, 3))
        pool.step_ids(ids, DT, m)
    return pool, ids, cls, Qc, Rc, p0, v


def timed(f, warmup, calls):
    s, out = [], None
    for c in range(warmup + calls):
        ta = time.perf_counter()
        out = f()
        tb = time.perf_counter()
        if c >= warmup:
            s.append(tb - ta)
    return s, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
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
        pool, ids, cls, Qc, Rc, p0, v = setup(model, n, 7)
        rng = np.random.default_rng(3)
        rows = rng.choice(n, Q, replace=False)
        z = pool.read_estimates(ids[rows], t1)["pose"][:, :3] + rng.normal(0, 0.003, (Q, 3))
        for gate in (CHI2, float("inf")):
            brute_s, ref = timed(lambda: brute_pool(model, pool, cls, Qc, Rc, t1, z, gate, 10000), 1, 3)
            brute_ms = 1e3 * float(np.median(brute_s))
            for k in (100, 10000):
                ms, got = timed(lambda: pool.gated_targets(t1, z, gate, k), a.warmup, a.calls)
                line = {"bench": "gate", "gpu": gpu, "power_limit": power, "visible_gpus": n_gpu, "model": model, "targets": n,
                        "classes": N_CLS, "handle": "pool", "queries": Q, "k": k, "gate": gate if np.isfinite(gate) else "inf",
                        "calls": a.calls, "ms_call": stats(ms), "pairs_per_s": n * Q / float(np.median(ms)),
                        "count_total": int(got[0].sum()), "count_per_query_mean": float(got[0].mean()), "falling_ticks": TICKS,
                        "t1": "now + 50 ms", "brute_force_ms": stats(brute_s),
                        "speedup_vs_brute_force": brute_ms / (1e3 * float(np.median(ms))),
                        "matches_brute_force": same(got, (ref[0], ref[1][:, :k], ref[2][:, :k])),
                        "note": "host clock around the synchronous call after warm-up, pageable caller arrays; brute force = one "
                                "batched read_state of every P and t + read_estimates at t1 + the contract in numpy + np.lexsort per "
                                "query, timed in this run (1 warm-up, 3 calls); speed-up = ratio of the medians"}
                print(json.dumps(line), flush=True)
                if out:
                    out.write(json.dumps(line) + "\n"); out.flush()
        pool.close()


if __name__ == "__main__":
    main()
