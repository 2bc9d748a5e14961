#!/usr/bin/env python3
"""Association of one frame of unlabelled detections (TargetPool.associate / te_pool_associate, the call a manager handle whose
targets live in one pool runs) against the path a caller has without it: gatedTargets(k = 8) for every detection, the greedy on the
host, and te_pool_step_ids with dt = t1 - t per row (the pool form of updateBatch with per-row dt).

Workload: 1 Mi targets of each of the four models over 8 dense random SPD classes (interleaved: every warp holds all 8), falling as
in tools/bench_sphere_sweep.py and measured for 50 ticks; at t1 = now + 50 ms, q detections drawn from q distinct targets'
predicted S (position p + L n, n standard normal), plus 10 % clutter uniform over the scene, shuffled; gate 11.34 (the 99 %
chi-square quantile for 3 degrees of freedom), K = 8; q in {4 096, 65 536, 1 Mi}; cuda:0.  One JSON line per (model, q): host clock
around the synchronous call after warm-up with apply = 0 and with apply = 1, candidates per detection, grid levels that held
targets, matching rounds, the share of target detections assigned to their own target, and at q = 4 096 the alternative timed in
the same run with whether it gives the same assignment.

  python tools/bench_associate.py [--calls K] [--warmup W] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_gate import MODELS, N_CLS, setup, timed  # noqa: E402
from bench_sphere_sweep import DT, TICKS, stats  # noqa: E402
from tests.test_gpu_associate import greedy, same_assignment  # noqa: E402
from tests.test_gpu_gate import CHI2, pos_cov  # noqa: E402

K = 8


def draw(name, pool, ids, cls, Qc, Rc, rows, t1, rng):
    """one detection per listed target, drawn from its predicted position covariance S (in chunks: AR's P is 2.6 KB a target)"""
    if rows.size > 65536:
        return np.concatenate([draw(name, pool, ids, cls, Qc, Rc, rows[i:i + 65536], t1, rng) for i in range(0, rows.size, 65536)])
    st = pool.read_state(ids[rows], want=("P", "t"))
    C = pos_cov(name, st["P"], st["t"], cls[rows], Qc, t1)
    S = np.zeros((rows.size, 3, 3))
    for (a, b), v in C.items():
        S[:, a, b] = S[:, b, a] = v + Rc[cls[rows], b, a]
    L = np.linalg.cholesky(S)
    p = pool.read_estimates(ids[rows], t1)["pose"][:, :3]
    return p + np.einsum("nij,nj->ni", L, rng.normal(size=(rows.size, 3)))


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
        pos = pool.read_estimates(ids, t1)["pose"][:, :3]
        lo, hi = pos.min(axis=0), pos.max(axis=0)
        for q in (4096, 65536, n):
            rows = rng.choice(n, q, replace=False)
            z = np.concatenate([draw(model, pool, ids, cls, Qc, Rc, rows, t1, rng), rng.uniform(lo, hi, (q // 10, 3))])
            src = np.concatenate([ids[rows], np.full(q // 10, 0xFFFFFFFF, dtype=np.uint32)])
            perm = rng.permutation(z.shape[0])
            det = np.zeros((z.shape[0], 7)); det[:, 6] = 1.0
            det[:, :3] = z[perm]
            src = src[perm]
            ms0, got = timed(lambda: pool.associate(t1, det, CHI2, K), a.warmup, a.calls)
            st0 = pool.assoc_stats()
            line = {"bench": "associate", "gpu": gpu, "power_limit": power, "visible_gpus": n_gpu, "model": model, "targets": n,
                    "classes": N_CLS, "handle": "pool", "detections": int(det.shape[0]), "from_targets": q, "clutter": q // 10,
                    "gate": CHI2, "K": K, "calls": a.calls, "ms_apply0": stats(ms0), "assigned": int((got[0] != 0xFFFFFFFF).sum()),
                    "candidates_per_detection": float(got[2].mean()), "levels": st0["levels"], "everywhere": st0["everywhere"],
                    "rounds": st0["rounds"],
                    "own_target_rate": float((got[0][src != 0xFFFFFFFF] == src[src != 0xFFFFFFFF]).mean())}
            if q == 4096:
                same_alt = same_assignment(greedy(*pool.gated_targets(t1, det[:, :3], CHI2, K)[1:]), got[:2])

                def alternative():
                    cnt, cid, cd2 = pool.gated_targets(t1, det[:, :3], CHI2, K)
                    gid, gd2 = greedy(cid, cd2)
                    hit = gid != 0xFFFFFFFF
                    t_now = pool.read_state(gid[hit], want=("t",))["t"]
                    pool.step_ids(gid[hit], t1 - t_now, det[hit])
                    return gid, gd2
                alt_s, alt = timed(alternative, 1, 3)
                line.update({"alternative_ms": stats(alt_s), "alternative_same_assignment": same_alt,
                             "alternative": "gated_targets(k=8) + host greedy + read_state(t) + step_ids(dt = t1 - t); timed after "
                                            "the associate calls, on the same pool"})
            ms1, got1 = timed(lambda: pool.associate(t1, det, CHI2, K, apply=True), a.warmup, a.calls)
            line.update({"ms_apply1": stats(ms1), "rounds_apply1": pool.assoc_stats()["rounds"],
                         "note": "host clock around the synchronous call after warm-up, pageable caller arrays; apply = 1 calls run "
                                 "one after the other on the same pool (targets already at t1 get dt = 0)"})
            print(json.dumps(line), flush=True)
            if out:
                out.write(json.dumps(line) + "\n"); out.flush()
        pool.close()


if __name__ == "__main__":
    main()
