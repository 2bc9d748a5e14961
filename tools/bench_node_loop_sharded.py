#!/usr/bin/env python3
"""The node loop over several GPUs (target_tick_manager_new_sharded): the C3 churn of tools/bench_configs.py::c3_tick_manager --
1 Mi angular-rates targets, every tick 1 % of the speaking ids fall silent (they expire 8 ticks later by the reference's predicate)
and as many fresh ids appear -- with the /tf messages in page-locked host arrays, on G = 1 / 2 / 4 / 8 shards over the visible GPUs.

For every G and both routes of a message (`device`: te_group_route_records; `host`: the router threads, forced through
TE_SHARD_HOST_ROUTE) it prints one JSON line: mean / median / worst ms per tick of the callback (target_tick_manager_callback_ids),
of the tick without the broadcast (publish off) and of the tick with it (publish on, a second run of the same churn); `publish` is
the difference of the two tick means.  --same-device puts all G shards on cuda:0 (host and routing overheads without the scaling).

  python tools/bench_node_loop_sharded.py [--targets N] [--ticks K] [--shards 1,2,4,8] [--same-device] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
DT = 1.0 / 250.0


def clock(tk):
    ns_ = 1000 * 10 ** 9 + tk * 4000000
    return ns_ // 10 ** 9, ns_ % 10 ** 9


def make_messages(n, ticks, lib):
    """the churn of c3_tick_manager, every array page-locked (te_host_register) so that the G uploads of a message run at once"""
    rng = np.random.default_rng(2)
    ids = np.arange(n, dtype=np.int64); silent_at = np.full(n, 1 << 30, dtype=np.int64); next_id = n
    poses = np.zeros((int(n * 1.1), 7)); poses[:, :3] = rng.uniform(-5, 5, (poses.shape[0], 3)); poses[:, 6] = 1.0
    keep = [poses]
    msgs = []
    for k in range(ticks + 1):
        if k > 0:
            old = np.nonzero(silent_at > k)[0]
            quit_ = rng.choice(old, size=max(1, old.size // 100), replace=False)
            silent_at[quit_] = k
            fresh = np.arange(next_id, next_id + quit_.size, dtype=np.int64); next_id += quit_.size
            ids = np.concatenate([ids, fresh]); silent_at = np.concatenate([silent_at, np.full(fresh.size, 1 << 30, dtype=np.int64)])
        sec, nsec = clock(k)
        r = np.ascontiguousarray(ids[silent_at > k].astype(np.uint32))
        s_ = np.full(r.size, sec, dtype=np.uint32); ns_ = np.full(r.size, nsec, dtype=np.uint32)
        keep += [r, s_, ns_]
        msgs.append((r, s_, ns_, poses[:r.size]))
    for a in keep:
        if lib.te_host_register(a.ctypes.data_as(C.c_void_p), a.nbytes) != 0:
            raise RuntimeError("te_host_register failed")
    return msgs, keep


def stats(v):
    v = 1e3 * np.asarray(v)
    return {"mean": float(v.mean()), "median": float(np.median(v)), "worst": float(v.max())}


def run(msgs, G, devices, route, publish, yaml):
    from target_estimation_b200.manager import ShardedTickManagerC
    if route == "host":
        os.environ["TE_SHARD_HOST_ROUTE"] = "1"
    else:
        os.environ.pop("TE_SHARD_HOST_ROUTE", None)
    mgr = ShardedTickManagerC(yaml, G, devices)
    os.environ.pop("TE_SHARD_HOST_ROUTE", None)
    mgr.set_expiration(8 * DT); mgr.set_publish(publish)
    r, s_, ns_, p_ = msgs[0]
    mgr.callback_ids(r, s_, ns_, p_); mgr.tick(DT, *clock(0))          # first sight of every id (untimed)
    cb, tk = [], []
    n_erased = 0
    for k in range(1, len(msgs)):
        r, s_, ns_, p_ = msgs[k]
        ta = time.perf_counter()
        mgr.callback_ids(r, s_, ns_, p_)
        tb = time.perf_counter()
        n_erased += mgr.tick(DT, *clock(k), cap=1 << 16).size
        tc = time.perf_counter()
        cb.append(tb - ta); tk.append(tc - tb)
    n_live = mgr.ids().size
    n_pub = mgr.published()[0].size if publish else 0
    mgr.close()
    return cb, tk, n_erased, n_live, n_pub


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--targets", type=int, default=1 << 20)
    ap.add_argument("--ticks", type=int, default=40)
    ap.add_argument("--shards", default="1,2,4,8")
    ap.add_argument("--same-device", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import target_estimation_b200 as te
    n_gpu = torch.cuda.device_count()
    if n_gpu == 0:
        raise SystemExit("no CUDA device: this measurement needs a GPU")
    gpu = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                               timeout=30).stdout.split("\n")[0].strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    yaml = os.path.join(ROOT, "models", "model_angular_rates_params.yaml")
    msgs, keep = make_messages(a.targets, a.ticks, te.lib)
    out = open(a.out, "a") if a.out else None
    for G in (int(x) for x in a.shards.split(",")):
        if not a.same_device and G > n_gpu:
            continue
        devices = [0] * G if a.same_device else list(range(G))
        for route in ("device", "host"):
            cb, tk_off, n_er, n_live, _ = run(msgs, G, devices, route, False, yaml)
            cb_on, tk_on, n_er2, n_live2, n_pub = run(msgs, G, devices, route, True, yaml)
            assert (n_er, n_live) == (n_er2, n_live2) and n_pub == n_live
            line = {"bench": "node_loop_sharded", "gpu": gpu, "power_limit": power, "visible_gpus": n_gpu, "shards": G,
                    "devices": devices, "route": route, "targets": a.targets, "ticks": a.ticks, "erased": int(n_er), "live_at_end": int(n_live),
                    "ms_callback": stats(cb + cb_on), "ms_tick_no_publish": stats(tk_off), "ms_tick_with_publish": stats(tk_on),
                    "ms_publish_mean": 1e3 * (float(np.mean(tk_on)) - float(np.mean(tk_off))),
                    "ms_per_tick_with_publish": stats(np.asarray(cb_on) + np.asarray(tk_on)),
                    "note": "host clock around target_tick_manager_callback_ids / target_tick_manager_update (both end in a device "
                            "synchronise); page-locked message arrays; publish = mean tick with the broadcast - mean tick without it"}
            print(json.dumps(line), flush=True)
            if out:
                out.write(json.dumps(line) + "\n"); out.flush()
    for arr in keep:
        te.lib.te_host_unregister(arr.ctypes.data_as(C.c_void_p))


if __name__ == "__main__":
    main()
