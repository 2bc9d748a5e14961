#!/usr/bin/env python3
"""The axis-blocked UV / UA step against the full packed step, on the flagship workload: 4 Mi targets of one shipped model on cuda:0,
one dense tick per step (95 % update, 5 % predict-only), [n][7] pose measurements in device memory.

Two pools of the same targets: `blocked` holds the shipped class only (its Q, R and P0 never couple the x / y / z axes, so the pool
steps the per-axis covariance blocks); `full` holds the same class plus one unused, bitwise-symmetric class that couples the axes,
so it runs the packed direct kernel on the whole upper triangle.  `blocked` is also timed at the other launch shapes of its large-pool
kernel (TE_AXIS_SHAPE = WARPSxCTAS).  The forms alternate in one process, ROUNDS times, each in a window of at least --window s of
device time (CUDA events around back-to-back ticks on the pool's stream, after a warm-up).  One JSON line per (model, form):
ms per tick (median and spread over the rounds), target-steps/s, the bytes an update step moves from the field lists of the two
forms, and GB/s against MEASURED_PEAKS.json (bench.py's fallback without it).

  python tools/bench_axis_blocks.py [--targets N] [--window S] [--rounds R] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import peaks  # noqa: E402

DT = 1.0 / 250.0
SHAPES = ("4x3", "8x1", "8x2", "4x4")
DEFAULT_SHAPE = {"uniform_acceleration": "4x3", "uniform_velocity": "8x2"}   # te_step.cu launch_kin


def fields_moved(N, blocked):
    """fields a packed update step reads and writes: x, the upper triangle (blocked: its in-axis entries only), t, n_meas"""
    P = sum(1 for i in range(N) for j in range(i, N) if not blocked or i % 3 == j % 3)
    return N + P + 2


def step_bytes(N, blocked, update):
    # state in and out, xyz of the measurement (update steps), action byte, class index
    return 16 * fields_moved(N, blocked) + (24 if update else 0) + 1 + 2


def coupled_class(N, M, rng):
    sym = lambda A: np.triu(A) + np.triu(A, 1).T
    B = rng.normal(size=(N, N)); Q = sym(1e-3 * (B @ B.T + N * np.eye(N)))
    B = rng.normal(size=(M, M)); R = sym(1e-3 * (B @ B.T + M * np.eye(M)))
    B = rng.normal(size=(N, N)); P0 = sym(B @ B.T + N * np.eye(N))
    return Q, R, P0


def query_gpu():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.split("\n")[0].strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--targets", type=int, default=4 << 20)
    ap.add_argument("--window", type=float, default=1.0, help="seconds of device time per timed window")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--models", default="uniform_acceleration,uniform_velocity")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import target_estimation_b200 as te
    if torch.cuda.device_count() == 0:
        raise SystemExit("no CUDA device: this measurement needs a GPU")
    gpu = query_gpu()
    peak, peak_src = peaks()
    out = open(a.out, "a") if a.out else None
    n = a.targets
    for model in a.models.split(","):
        mtype, _, Q, R, P0 = te.load_model(model)
        N, M = te.model_dims(mtype)
        rng = np.random.default_rng(5)
        meas = np.zeros((n, 7)); meas[:, :3] = rng.uniform(-5, 5, (n, 3)); meas[:, 6] = 1.0
        action = np.where(rng.uniform(size=n) < 0.05, te.ACT_PREDICT, te.ACT_UPDATE).astype(np.uint8)
        n_upd = int((action == te.ACT_UPDATE).sum())
        d_meas = torch.from_numpy(meas).cuda()
        d_act = torch.from_numpy(action).cuda()
        ids = np.arange(n, dtype=np.uint32)
        torch.cuda.synchronize()
        stream = torch.cuda.Stream()
        pools = {}
        for name in ("blocked", "full"):
            p = te.TargetPool(mtype, device=0)
            p.set_stream(stream.cuda_stream)   # the timing events and the ticks on one stream
            p.register_class(Q, R, P0)
            if name == "full":
                p.register_class(*coupled_class(N, M, rng))
            p.add(ids, meas, p0_scale=rng.uniform(0.5, 2.0, n))
            pools[name] = p
        forms = [("full", None)] + [("blocked", s) for s in SHAPES]

        def run(form, ticks):
            name, shape = form
            if shape:
                os.environ["TE_AXIS_SHAPE"] = shape
            else:
                os.environ.pop("TE_AXIS_SHAPE", None)
            p = pools[name]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(ticks):
                p.step_dense(DT, d_meas, 7, d_act, te.ACT_UPDATE)
            e1.record(stream)
            e1.synchronize()
            return e0.elapsed_time(e1) / ticks

        ticks = {}
        for form in forms:
            run(form, 20)                                   # warm-up: module load, first-touch of both buffers
            ticks[form] = max(50, int(a.window / (run(form, 50) * 1e-3)) + 1)
        times = {form: [] for form in forms}
        for r in range(a.rounds):
            for form in forms:
                times[form].append(run(form, ticks[form]))
                print("%s %s round %d: %d ticks, %.4f ms per tick" % (model, form, r, ticks[form], times[form][-1]), file=sys.stderr, flush=True)
        os.environ.pop("TE_AXIS_SHAPE", None)
        for form in forms:
            name, shape = form
            blocked = name == "blocked"
            ms = float(np.median(times[form]))
            moved = n_upd * step_bytes(N, blocked, True) + (n - n_upd) * step_bytes(N, blocked, False)
            line = {"bench": "axis_blocks", "gpu": gpu, "model": model, "targets": n, "form": name,
                    "launch_shape": shape if blocked else ("8x1" if model == "uniform_acceleration" else "4x3"),
                    "default_shape": (shape == DEFAULT_SHAPE[model]) if blocked else True,
                    "ticks_per_window": ticks[form], "rounds": a.rounds, "ms_per_tick": ms, "ms_per_tick_rounds": times[form],
                    "spread": (max(times[form]) - min(times[form])) / ms, "target_steps_per_s": n / (ms * 1e-3),
                    "fields_moved": fields_moved(N, blocked), "bytes_per_update_step": step_bytes(N, blocked, True),
                    "bytes_per_predict_step": step_bytes(N, blocked, False), "bytes_per_tick": moved, "gbs": moved / (ms * 1e-3) / 1e9,
                    "peak_gbs": peak, "peak_source": peak_src, "frac_of_peak": moved / (ms * 1e-3) / 1e9 / peak,
                    "note": "CUDA events around back-to-back dense ticks (95 % update), windows alternated in one process; bytes from "
                            "the field lists of the form (state in and out, xyz of the measurement, action, class)"}
            print(json.dumps(line), flush=True)
            if out:
                out.write(json.dumps(line) + "\n"); out.flush()
        for p in pools.values():
            p.close()
        del d_meas, d_act
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
