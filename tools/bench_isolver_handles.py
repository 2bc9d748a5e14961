#!/usr/bin/env python3
"""IntersectionSolver on the manager handles (target_isolver_* of libtarget_c.so): 1 Mi uniform-acceleration targets, one pose query
per target per call (target_isolver_query_batch), stream = target index, on G = 1 shard, 8 shards on cuda:0 and one shard per visible
GPU.

For each G it prints one JSON line: ms per batched call on the sharded handle, split into its phases (routing by owner, moves of
stream state between shards, the shards' device queries -- uploads, kernels, read-backs, all shards at once -- and the results put
back in call order); the same call on a plain handle on cuda:0; a call in which every stream changes shard (the ids of the streams
rotate by one between calls, the worst case: in steady state a stream stays with its target's owner and nothing moves); and the
latency of the per-id calls (target_isolver_get_time / _get_pose) on both handles.

  python tools/bench_isolver_handles.py [--targets N] [--calls K] [--warmup W] [--filters-length L] [--out FILE]
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


def stats(v):
    v = 1e3 * np.asarray(v)
    return {"mean": float(v.mean()), "median": float(np.median(v)), "worst": float(v.max())}


def setup(mgr, n, rng):
    ids = np.arange(n, dtype=np.uint32)
    p = np.zeros((n, 7)); p[:, :3] = rng.uniform(-5, 5, (n, 3)); p[:, 2] += 20.0; p[:, 6] = 1.0
    assert mgr.init_batch(ids, DT, p) == n
    for k in range(1, 6):                                   # a few falling measurements: every target has an acceleration
        m = p.copy(); m[:, 2] -= 0.5 * 9.81 * (k * DT) ** 2
        assert mgr.update_batch(ids, DT, m) == n
    return ids, p


def time_calls(solver, ids, t1, origin, radius, stream, calls, warmup, rotate=False):
    out = []
    n = ids.size
    shifted = (ids, np.roll(ids, 1))
    phases = []
    for k in range(warmup + calls):
        q = shifted[k % 2] if rotate else ids
        ta = time.perf_counter()
        found, _, _, _ = solver.query_batch(q, t1, origin, radius, 0.5, 0.5, stream=stream)
        tb = time.perf_counter()
        assert found == n
        if k >= warmup:
            out.append(tb - ta)
            phases.append(solver.last_timing())
    return out, {key: float(np.mean([p[key] for p in phases])) for key in phases[0]}


def per_id(solver, n, origin, reps=200):
    rng = np.random.default_rng(3)
    pick = rng.integers(0, n, reps)
    ta = time.perf_counter()
    for i in pick:
        solver.time(int(i), 0.05, origin[i], 1.0)
    tb = time.perf_counter()
    for i in pick:
        solver.pose(int(i), 0.05, 0.5, 0.5, origin[i], 1.0)
    tc = time.perf_counter()
    return 1e6 * (tb - ta) / reps, 1e6 * (tc - tb) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--targets", type=int, default=1 << 20)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--filters-length", type=int, default=250)
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
    yaml = os.path.join(ROOT, "models", "model_uniform_acceleration_params.yaml")
    n, L = a.targets, a.filters_length
    rng = np.random.default_rng(1)
    configs = [[0], [0] * 8]
    if n_gpu > 1:
        configs.append(list(range(n_gpu)))
    plain = TargetManagerC(yaml, device=0)
    ids, p = setup(plain, n, np.random.default_rng(7))
    t1 = np.full(n, 5 * DT)
    origin = p[:, :3] - np.array([0.0, 0.0, 3.0]) + rng.normal(0, 0.1, (n, 3))   # below every target: an interception exists
    radius = np.full(n, 1.0)
    stream = np.arange(n, dtype=np.int32)
    s_plain = IntersectionSolverC(plain, n, L)
    ms_plain, ph_plain = time_calls(s_plain, ids, t1, origin, radius, stream, a.calls, a.warmup)
    us_plain = per_id(s_plain, n, origin)
    s_plain.close(); plain.close()
    out = open(a.out, "a") if a.out else None
    for devices in configs:
        G = len(devices)
        mgr = ShardedManagerC(yaml, G, devices)
        setup(mgr, n, np.random.default_rng(7))
        s = IntersectionSolverC(mgr, n, L)
        ms, ph = time_calls(s, ids, t1, origin, radius, stream, a.calls, a.warmup)
        ms_mv, ph_mv = time_calls(s, ids, t1, origin, radius, stream, max(4, a.calls // 4), 1, rotate=True)
        us = per_id(s, n, origin)
        s.close(); mgr.close()
        line = {"bench": "isolver_handles", "gpu": gpu, "power_limit": power, "visible_gpus": n_gpu, "shards": G, "devices": devices,
                "targets": n, "queries_per_call": n, "filters_length": L, "calls": a.calls,
                "ms_call_sharded": stats(ms), "ms_phases_sharded": ph,
                "ms_call_plain": stats(ms_plain), "ms_phases_plain": ph_plain,
                "ms_call_every_stream_moves": stats(ms_mv), "ms_phases_every_stream_moves": ph_mv,
                "us_per_id_time_sharded": us[0], "us_per_id_pose_sharded": us[1],
                "us_per_id_time_plain": us_plain[0], "us_per_id_pose_plain": us_plain[1],
                "note": "host clock around target_isolver_query_batch (ends in a device synchronise), pageable caller arrays; phases "
                        "= target_isolver_last_timing (route, move, device incl. uploads and read-backs, writeback); the plain handle "
                        "is on cuda:0; every_stream_moves rotates the ids of the streams by one between calls"}
        print(json.dumps(line), flush=True)
        if out:
            out.write(json.dumps(line) + "\n"); out.flush()


if __name__ == "__main__":
    main()
