#!/usr/bin/env python3
"""bench.py -- KF predict+update target-steps/sec on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (oracle port) on host cores
    python bench.py ... --dump-outputs DIR                   # + state after the last timed step, seeded sample of targets, DIR/*.npy

One "step" = one tick of the hot path over every target of the pool: TargetManager::update(id, dt, meas) for
each target (predict + update + t / n_meas bookkeeping; a Philox-free 5 % of the targets miss their measurement
each tick and take the predict-only path, SURVEY.md 8(d) anti-cohort rule).  Workload: BASELINE.json configs[1]'s
model and arithmetic (uniform-acceleration, FP64 predict+update per measurement tick on 1 B200) at a target count
whose state (720 B/target) is far larger than the 126 MB L2, so every tick streams from HBM; the literal 10k-target
case is L2-resident and launch-bound (SURVEY.md H8) and is reported beside it under "c2_10k".

value    : targets x steps / device time, inputs (measurements, action masks) resident in HBM.
e2e      : same ticks through te_pool_tick_host (HOST pinned buffers -> H2D inside the timed region, the tick, and a
           D2H read of every target's estimated position, pipelined in chunks over three streams).
roofline : achieved = algorithmic bytes per launch (SURVEY.md 8(d): UA 1496 B per update step, 1456 B per
           predict-only step) / average kernel duration (CUDA events on the pool's stream); peak = MEASURED_PEAKS.json.
cpu_baseline : the oracle port (oracle/, Eigen-free restatement of the reference TargetManager path) and the reference's own
               sources on a stand-in Eigen (oracle/_ref) on host cores; the faster one is the value, both are listed.
"""
import argparse
import json
import os
import sys

import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

DT = 1.0 / 250.0
METRIC = "kf_predict_update_target_steps_per_sec"
UNIT = "target-steps/s"
# dominant kernel per model with the default variant (te_pool.cu launch_step)
KERNEL_NAME = {"uniform_velocity": "te::kf_step_kin_direct_kernel", "uniform_acceleration": "te::kf_step_kin_direct_kernel",
               "angular_velocities": "te::kf_step_av_stream_kernel", "angular_rates": "te::kf_step_split_kernel"}
MODEL_SHORT = {"uniform_velocity": "UV", "uniform_acceleration": "UA", "angular_velocities": "AV", "angular_rates": "AR"}
MODEL_DIMS = {"uniform_velocity": (6, 3), "uniform_acceleration": (9, 3), "angular_velocities": (12, 6), "angular_rates": (18, 6)}   # (n, m)


def model_yaml(model):
    return os.path.join(ROOT, "models", "model_%s_params.yaml" % model)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="uniform_acceleration", choices=list(MODEL_SHORT))
    ap.add_argument("--targets", type=int, default=0, help="targets per GPU (default: 4Mi for UV/UA, 1Mi for AV/AR)")
    ap.add_argument("--variant", type=int, default=-1)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-ref-abi", action="store_true", help="skip the e2e figure through libtarget_c.so")
    ap.add_argument("--no-node-loop", action="store_true", help="skip the secondary node-loop (mailbox churn) figure")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the sampled oracle check of the benchmarked pool")
    ap.add_argument("--no-small", action="store_true")
    ap.add_argument("--allgather", action="store_true", help="(default at N>1; kept for compatibility)")
    ap.add_argument("--no-allgather", action="store_true", help="skip the all-gather of estimate records at N>1")
    ap.add_argument("--no-c5", action="store_true", help="skip BASELINE configs[4] (mixed models sharded by id, all-gather at N>1)")
    ap.add_argument("--c5-targets", type=int, default=8 << 20, help="C5 targets per GPU (64 Mi over 8 GPUs)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the state of a fixed, seeded sample of the benchmarked targets as DIR/<name>.npy "
                         "(with --gpus N > 1: a sample of rank 0's shard)")
    return ap.parse_args()


def ncu_traffic(model, n):
    """per-launch DRAM bytes of the dominant kernel from the committed ncu capture of this configuration"""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            e = json.load(f).get("%s@%d" % (model, n))
        if e:
            return e["traffic_bytes"], e["source"]
    return None, None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class stdout_to_stderr:
    """NCCL prints its version banner to the process's stdout (file descriptor 1) when the communicator is created: point
    fd 1 at stderr for that moment, so that stdout carries nothing but the one JSON line."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


class ClockSampler(threading.Thread):
    """nvidia-smi style clock/throttle sampling through NVML during the timed region."""

    def __init__(self, index, uuid=None):
        super().__init__(daemon=True)
        self.index = index
        self.uuid = uuid      # NVML indices ignore CUDA_VISIBLE_DEVICES: address the device by UUID when torch knows it
        self.stop_flag = False
        self.sm = []
        self.reasons = set()
        self.sm_max = None
        self.power = []

    def run(self):
        if os.environ.get("TE_NO_SAMPLER"):   # debugging switch
            self.reasons.add("sampler_disabled")
            return
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = None
            if self.uuid:
                try:
                    h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + self.uuid).encode())
                except Exception:
                    h = None
            if h is None:
                h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
            }
            while not self.stop_flag:
                self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
                except Exception:
                    pass
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.02)
        except Exception as e:  # NVML missing: report that instead of inventing clocks
            self.reasons.add("nvml_unavailable:%s" % type(e).__name__)

    def result(self):
        self.stop_flag = True
        self.join(timeout=2.0)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max,
                "power_w_max": max(self.power) if self.power else None, "samples": len(self.sm), "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port and the reference's own sources (oracle/_ref) on host cores
# ------------------------------------------------------------------------------------------------------
REF_LIB = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle", "_ref", "libref_manager.so")


def _cpu_bench_fn(kind):
    """kind 'port': orc_bench_steps of oracle/libte_oracle.so (the Eigen-free restatement); kind 'reference':
    refm_bench_steps of oracle/_ref/libref_manager.so = the reference's own src/*.cpp (TargetManager, the model types,
    kalman.cpp) compiled unmodified against the stand-in Eigen of oracle/eigen_standin.  Same workload, same arguments;
    None when the library is absent."""
    import ctypes as C
    from tests import orc
    L = orc.lib()
    if kind == "port":
        return L.orc_bench_steps
    if not os.path.exists(REF_LIB):
        return None
    R = C.CDLL(REF_LIB, mode=C.RTLD_GLOBAL)
    if not hasattr(R, "refm_bench_steps"):
        return None
    R.refm_bench_steps.restype = C.c_double
    R.refm_bench_steps.argtypes = L.orc_bench_steps.argtypes
    return R.refm_bench_steps


_TICK_RATE = {}   # (kind, model, threads) -> ticks per second of the last timed run: later runs skip the probe


def cpu_run(model_name, threads, seconds, n_targets=10000, kind="port"):
    import ctypes as C
    from tests import orc
    y = orc.load_yaml(model_yaml(model_name))   # the oracle's own reader: the CPU arms never load the CUDA library
    mtype, Q, R, P0 = y["type"], y["Q"], y["R"], y["P"]
    fn = _cpu_bench_fn(kind)
    if fn is None:
        return None
    rng = np.random.default_rng(7)
    meas = np.zeros((n_targets, 7))
    meas[:, :3] = rng.uniform(-5, 5, (n_targets, 3))
    meas[:, 6] = 1.0
    Qc, Rc, Pc = orc.colmajor(Q), orc.colmajor(R), orc.colmajor(P0)
    n, m = Q.shape[0], R.shape[0]
    chk = C.c_double()

    def run(ticks):
        return fn(mtype, orc.ptr(Qc), n, orc.ptr(Rc), m, orc.ptr(Pc), n_targets, ticks, threads, DT, orc.ptr(meas), 0.05, C.byref(chk))
    key = (kind, model_name, threads)
    if key not in _TICK_RATE:
        _TICK_RATE[key] = 2.0 / max(run(2), 1e-9)
    ticks = max(2, int(seconds * _TICK_RATE[key]))
    t = run(ticks)
    _TICK_RATE[key] = ticks / max(t, 1e-9)
    return {"value": n_targets * ticks / t, "ticks": ticks, "targets": n_targets, "seconds": t, "threads": threads, "kind": kind}


def cpu_best(model_name, threads, seconds):
    """both CPU implementations on the same bounded sample (half the time each); the FASTER one is the reported baseline (the
    stand-in Eigen under the reference's sources is heap-backed and unvectorised, so the port usually wins), both are listed"""
    ref = cpu_run(model_name, threads, seconds / 2, kind="reference")
    port = cpu_run(model_name, threads, seconds / 2 if ref else seconds, kind="port")
    best = ref if (ref and ref["value"] > port["value"]) else port
    return best, {"port": port["value"], "reference_sources_on_standin_eigen": ref["value"] if ref else None}


def default_targets(model):
    return (4 << 20) if MODEL_SHORT[model] in ("UV", "UA") else (1 << 20)


def make_config(model, n, world, variant, n_sets=4, stride=7):
    N, M = MODEL_DIMS[model]
    short = MODEL_SHORT[model]
    return {"workload": "BASELINE configs[1] (%s, FP64 predict+update per measurement tick) at %d targets per GPU" % (short, n),
            "motion_model": model, "targets_per_gpu": n, "targets_total": n * world, "dt": DT, "missed_measurement_prob": 0.05,
            "measurement_layout": "[n][7] pose, device resident, %d rotating sets" % n_sets,
            "l2": "inputs larger than L2: state %.0f MB + %.0f MB of measurements per tick vs 126 MB L2" % (
                n * (N + N * N + 2) * 8 / 1e6, n * stride * 8 / 1e6),
            "sharding": "owner(id) = id mod n_gpus, no data-path collective", "kernel_variant": variant}


def reference_arm(args, rank):
    if rank != 0:
        return
    from tests import orc
    cores = orc.lib().orc_hardware_threads()
    K = max(1, args.steps)
    per_step = min(5.0, 100.0 / (K + args.warmup))   # bounded sample: the whole run stays within a few minutes
    for _ in range(args.warmup):
        cpu_best(args.model, cores, per_step / 4)
    vals, secs, kinds = [], 0.0, []
    sample = both = None
    for _ in range(K):
        r, both = cpu_best(args.model, cores, per_step)
        vals.append(r["value"]); secs += r["seconds"]; kinds.append(r["kind"])
        sample = "%d %s targets x %d ticks per step, one TargetManager per thread sharded by id %% %d; value = the faster of the oracle port and " \
                 "the reference's own src/*.cpp on the stand-in Eigen (oracle/_ref), last step: %s" % (
                     r["targets"], MODEL_SHORT[args.model], r["ticks"], cores, json.dumps(both))
    v = float(np.mean(vals))
    kind = "reference" if all(k == "reference" for k in kinds) else "port"
    out = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": args.warmup,
           "ms_per_step": 1e3 * secs / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
           "data": "synthetic", "config": dict(make_config(args.model, args.targets or default_targets(args.model), args.gpus, args.variant),
                                               reference_arm="the reference as a whole cannot be built here (Eigen / yaml-cpp absent, no network): its TargetManager "
                                               "path runs (a) as the Eigen-free oracle port and (b) from its own sources on a stand-in Eigen (oracle/_ref, "
                                               "bit-identical results), -O2 -ffp-contract=off, all host threads, bounded sample: " + sample),
           "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "both": both},
           "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------------
# the CUDA arm
# ------------------------------------------------------------------------------------------------------
def make_pool(te, torch, model_name, n, rank, world, stream, variant):
    mtype, _, Q, R, P0 = te.load_model(model_name)
    pool = te.TargetPool(mtype, device=torch.cuda.current_device(), stream=stream.cuda_stream)
    if variant >= 0:
        pool.set_variant(variant)
    pool.register_class(Q, R, P0)
    pool.reserve(n)
    rng = np.random.default_rng(0x7A26E7 + rank)
    chunk = 1 << 20
    p0_all, scale_all = [], []
    for s in range(0, n, chunk):
        k = min(chunk, n - s)
        ids = (np.arange(s, s + k, dtype=np.int64) * world + rank).astype(np.uint32)   # owner(id) = id mod G
        p0 = np.zeros((k, 7))
        p0[:, :3] = rng.uniform(-5, 5, (k, 3))
        ang = rng.uniform(-1, 1, (k, 3)) * np.array([3.0, 1.0, 3.0])
        from tests.synth import rpy_to_quat
        p0[:, 3:7] = rpy_to_quat(ang)
        scale = rng.uniform(0.5, 2.0, k)                                                # anti-cohort P0 scale (H6)
        pool.add(ids, p0, p0_scale=scale)
        p0_all.append(p0)
        scale_all.append(scale)
    return pool, mtype, np.concatenate(p0_all), np.concatenate(scale_all)


def make_inputs(torch, p0, n_sets, stride, miss_prob, seed):
    """n_sets rotating device-resident measurement blocks [n][stride] + action masks [n] (uint8)."""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    base = torch.from_numpy(p0).cuda()
    meas, act = [], []
    for k in range(n_sets):
        m = base[:, :stride].clone()
        m[:, :3] += 0.01 * torch.randn((base.shape[0], 3), dtype=torch.float64, device="cuda", generator=g) + 0.004 * (k + 1)
        meas.append(m.contiguous())
        u = torch.rand((base.shape[0],), device="cuda", generator=g)
        act.append(torch.where(u < miss_prob, 1, 2).to(torch.uint8).contiguous())
    return meas, act


DUMP_BYTES = 48 << 20   # float64 payload of --dump-outputs whatever the model: small enough to keep beside a result and compare


DUMP_FIELDS = ("x", "P", "t", "n_meas")


def dump_ids(n, world, rank, N):
    """ids of the targets --dump-outputs writes: a fixed, seeded sample of this process's n targets (owner(id) = id mod world),
    ascending.  It depends on the model, the target count and the number of GPUs only, so two builds run with the same arguments
    are compared target for target.  With --gpus N > 1 only rank 0 writes, so the sample comes from rank 0's shard."""
    k = min(n, DUMP_BYTES // ((N + N * N + 3) * 8))
    sample = np.sort(np.random.default_rng(20261020).choice(n, k, replace=False))
    return (sample.astype(np.int64) * world + rank).astype(np.uint32)


def write_outputs(out_dir, ids, state):
    """What a caller of the timed path reads back after its last step (te_pool_read_state: x, P, t, n_meas) for the targets
    `ids`, as float64 DIR/<name>.npy files."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in [("ids", ids)] + [(f, state[f]) for f in DUMP_FIELDS]:
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist
    import target_estimation_b200 as te   # raises if the CUDA library is missing: no fallback

    torch.cuda.set_device(local_rank)
    if world > 1:
        with stdout_to_stderr():
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
    model = args.model
    short = MODEL_SHORT[model]
    n = args.targets or default_targets(model)
    K, W = args.steps, max(args.warmup, 3)
    stream = torch.cuda.Stream()
    pool, mtype, p0, p0_scale = make_pool(te, torch, model, n, rank, world, stream, args.variant)
    N, M = te.model_dims(mtype)
    stride = 7
    n_sets = 4
    meas, act = make_inputs(torch, p0, n_sets, stride, 0.05, 1234 + rank)
    n_upd = [int((a == 2).sum().item()) for a in act]
    B_upd = te.bytes_per_step(mtype)
    B_pred = B_upd - 8 * (7 if M == 6 else 3) - 16          # no measurement read, n_meas untouched
    d_ids = dump_ids(n, world, rank, N) if args.dump_outputs and rank == 0 else None
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    history = []   # measurement / action set of every tick the pool has seen, in order (replayed by the oracle in parity_check)

    def tick(k):
        pool.step_dense(DT, meas[k % n_sets], stride, act[k % n_sets])
        history.append(k % n_sets)

    # ---- resident-input throughput -----------------------------------------------------------------
    for k in range(W):
        tick(k)
    barrier()
    try:
        dev_uuid = str(torch.cuda.get_device_properties(local_rank).uuid)
    except Exception:
        dev_uuid = None
    sampler = ClockSampler(local_rank, dev_uuid)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for k in range(K):
        tick(k)
    ev1.record(stream)
    barrier()
    burst_note = None
    dumped = None
    if not sampler.sm:
        if d_ids is not None:
            dumped = pool.read_state(d_ids, want=DUMP_FIELDS)   # the burst below moves the state on
        # the timed region was shorter than NVML start-up + one 20 ms sample: keep sampling under an untimed burst of the same ticks
        t_end = time.perf_counter() + 0.5
        while time.perf_counter() < t_end:
            for k in range(16):
                tick(k)
            torch.cuda.synchronize()
        burst_note = "timed region shorter than one NVML sample: clocks sampled under an untimed burst of the same ticks right after it"
    clocks = sampler.result()
    if burst_note:
        clocks["note"] = burst_note
    if d_ids is not None:   # written after the clock sampling; the burst decision above is taken before any read
        write_outputs(args.dump_outputs, d_ids, dumped if dumped is not None else pool.read_state(d_ids, want=DUMP_FIELDS))
    ms = ev0.elapsed_time(ev1)
    t_ms = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max = float(t_ms.item())
    value = n * world * K / (ms_max * 1e-3)
    alg_bytes = sum(n_upd[k % n_sets] * B_upd + (n - n_upd[k % n_sets]) * B_pred for k in range(K)) / K
    peak, peak_src = peaks()
    achieved = alg_bytes / (ms / K * 1e-3) / 1e9
    traffic, traffic_src = ncu_traffic(model, n)
    # bytes the default kernel actually has to move: UV / UA / AV keep the covariance packed (upper triangle only is read
    # and written, SURVEY.md 8(d) "symmetric-packed" clause), AR moves the full matrix
    npv = 3 if M == 6 else 0
    if model != "angular_rates" and args.variant in (-1, 0):
        fields = N + N * (N + 1) // 2 + 2 + npv
        L_upd = 2 * fields * 8 + 8 * (7 if M == 6 else 3) + 3
        L_pred = 2 * fields * 8 + 3
        layout_note = "packed covariance: state + upper triangle + t + n_meas%s in and out, measurement, action + class bytes" % (" + prev_rpy" if npv else "")
    else:
        L_upd, L_pred = B_upd, B_pred
        layout_note = "full covariance (the SURVEY.md 8(d) figure)"
    layout_bytes = sum(n_upd[k % n_sets] * L_upd + (n - n_upd[k % n_sets]) * L_pred for k in range(K)) / K
    achieved_layout = layout_bytes / (ms / K * 1e-3) / 1e9

    # ---- e2e: host buffers through the C-ABI ---------------------------------------------------------
    # Headline form: the pipelined host tick (te_pool_tick_host_async + te_pool_tick_host_wait(2): the copies of tick k + 1 run under
    # the kernels of tick k and the read-back of tick k - 1) with the measurement block the model reads -- [n][3] positions for the linear models
    # (UV / UA use x y z of the pose only), [n][7] poses for the angular ones.  Every step moves its inputs from pinned host memory
    # and every target's estimated position back to pinned host memory inside the timed region.  The synchronous call and the
    # 56-byte pose form of the same tick are reported beside it.
    e2e = None
    if not args.no_e2e:
        h_act = [a.cpu().pin_memory() for a in act[:2]]
        h_out = [torch.empty((n, 3), dtype=torch.float64).pin_memory() for _ in range(3)]
        Ke = max(5, min(K, 40))

        def run_e2e(h_in, st, pipelined):
            def one(k):
                fn = te.lib.te_pool_tick_host_async if pipelined else te.lib.te_pool_tick_host
                if fn(pool._h, DT, h_in[k % 2].data_ptr(), st, h_act[k % 2].data_ptr(), 2, h_out[k % 3].data_ptr()) < 0:
                    raise RuntimeError(te._lib.last_error())
                if pipelined and te.lib.te_pool_tick_host_wait(pool._h, 2) < 0:      # results of tick k - 2 are in h_out[(k - 2) % 3] now
                    raise RuntimeError(te._lib.last_error())
                history.append(k % 2)
            for k in range(4):
                one(k)
            te.lib.te_pool_tick_host_wait(pool._h, 0)
            barrier()
            t0 = time.perf_counter()
            for k in range(Ke):
                one(k)
            if te.lib.te_pool_tick_host_wait(pool._h, 0) < 0:
                raise RuntimeError(te._lib.last_error())
            wall = (time.perf_counter() - t0) * 1e3          # host-synchronous end: the wall clock covers every copy
            barrier()
            t_e = torch.tensor([wall], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
            w = float(t_e.item())
            return {"value": n * world * Ke / (w * 1e-3), "unit": UNIT, "h2d_bytes_per_step": n * (st * 8 + 1), "d2h_bytes_per_step": n * 24,
                    "steps": Ke, "ms_per_step": w / Ke}

        h7 = [m.cpu().pin_memory() for m in meas[:2]]
        h3 = [m[:, :3].contiguous().cpu().pin_memory() for m in meas[:2]] if M == 3 else None
        if M == 3:
            e2e = run_e2e(h3, 3, True)
            e2e["api"] = "te_pool_tick_host_async + te_pool_tick_host_wait(2): pinned host meas[n][3] (x y z: all the linear models read of a pose) + action[n] in, est. position [n][3] out, three ticks in flight"
            e2e["pose7_pipelined"] = dict(run_e2e(h7, 7, True), api="the same with the reference's 56-byte pose measurements meas[n][7]")
            e2e["xyz_sync"] = dict(run_e2e(h3, 3, False), api="te_pool_tick_host (one tick at a time, returns when est_pos_out is complete), meas[n][3]")
            e2e["pose7_sync"] = dict(run_e2e(h7, 7, False), api="te_pool_tick_host, meas[n][7] (the round-1 headline form)")
        else:
            e2e = run_e2e(h7, 7, True)
            e2e["api"] = "te_pool_tick_host_async + te_pool_tick_host_wait(2): pinned host meas[n][7] + action[n] in, est. position [n][3] out, three ticks in flight"
            e2e["pose7_sync"] = dict(run_e2e(h7, 7, False), api="te_pool_tick_host (one tick at a time), meas[n][7]")
        h_meas = h7

        # the same tick through the REFERENCE-FACING C-ABI (include/target_manager_c.h, libtarget_c.so): a TargetManager built from the
        # model file, one target_manager_update_batch(ids, dt, meas, action) per step from pinned host arrays and one
        # target_manager_get_est_pose read-back (a sync point); rank 0 only, a few steps (the manager keeps a host registry per id)
        if rank == 0 and not args.no_ref_abi and stride == 7:
            try:
                from target_estimation_b200.manager import TargetManagerC, clib
                import ctypes as C
                mpath = os.path.join(os.path.dirname(os.path.abspath(__file__)), "models", "model_%s_params.yaml" % model)
                mg = TargetManagerC(mpath, device=torch.cuda.current_device())
                r_ids = torch.from_numpy(np.arange(n, dtype=np.int32)).pin_memory()
                ids_np = r_ids.numpy().view(np.uint32)
                p0_abi = h_meas[0].numpy()
                chunk = 1 << 20
                for c0 in range(0, n, chunk):
                    mg.init_batch(ids_np[c0:c0 + chunk], DT, p0_abi[c0:c0 + chunk])
                pose = np.zeros(7)

                def tick_abi(k):
                    rc = clib.target_manager_update_batch(mg.h, n, ids_np.ctypes.data_as(C.c_void_p), DT, C.c_void_p(h_meas[k % 2].data_ptr()),
                                                          C.c_void_p(h_act[k % 2].data_ptr()))
                    if rc != n:
                        raise RuntimeError("target_manager_update_batch applied %d of %d" % (rc, n))
                    mg.get_est_pose(int(ids_np[k % n]), pose)
                for k in range(2):
                    tick_abi(k)
                Ka = 5
                t0 = time.perf_counter()
                for k in range(Ka):
                    tick_abi(k)
                ta = (time.perf_counter() - t0) * 1e3
                # the dense tick of the same library: records in target_manager_get_dense_ids order, no ids travel, every target's estimated
                # position comes back (target_manager_update_dense_async / _wait: three ticks in flight, as the headline form)
                h_in_abi = h3 if M == 3 else h7
                st_abi = 3 if M == 3 else 7

                def tick_dense(k):
                    rc = clib.target_manager_update_dense_async(mg.h, DT, C.c_void_p(h_in_abi[k % 2].data_ptr()), st_abi, C.c_void_p(h_act[k % 2].data_ptr()),
                                                                C.c_void_p(h_out[k % 3].data_ptr()))
                    if rc != n or clib.target_manager_update_dense_wait(mg.h, 2) < 0:
                        raise RuntimeError("target_manager_update_dense_async: %s" % clib.target_manager_last_error().decode())
                for k in range(4):
                    tick_dense(k)
                clib.target_manager_update_dense_wait(mg.h, 0)
                Kd = 20
                t0 = time.perf_counter()
                for k in range(Kd):
                    tick_dense(k)
                clib.target_manager_update_dense_wait(mg.h, 0)
                td = (time.perf_counter() - t0) * 1e3
                e2e["reference_abi_dense"] = {"value": n * Kd / (td * 1e-3), "unit": UNIT, "h2d_bytes_per_step": n * (st_abi * 8 + 1), "d2h_bytes_per_step": n * 24,
                                              "ms_per_step": td / Kd, "n_gpus": 1,
                                              "api": "libtarget_c.so: target_manager_update_dense_async(dt, meas[n][%d], action[n], est_pos_out[n][3]) + "
                                                     "target_manager_update_dense_wait(2), pinned host arrays in target_manager_get_dense_ids order" % st_abi}
                e2e["reference_abi"] = {"value": n * Ka / (ta * 1e-3), "unit": UNIT, "h2d_bytes_per_step": n * (4 + 7 * 8 + 1), "d2h_bytes_per_step": 56,
                                        "ms_per_step": ta / Ka, "n_gpus": 1,
                                        "api": "libtarget_c.so: target_manager_update_batch(n, ids, dt, meas[n][7], action[n]) + target_manager_get_est_pose(id), "
                                               "pinned host arrays, one sparse-by-id launch per step (ids are looked up on the device)"}
                mg.close()
            except Exception as e:   # report, do not fail the headline
                e2e["reference_abi"] = {"error": str(e)[:300]}

    # ---- optional all-gather of estimate records (off the hot path) -----------------------------------
    allgather = None
    if world > 1 and not args.no_allgather:
        rec = torch.empty((n, 13), dtype=torch.float64, device="cuda")
        out = torch.empty((world * n, 13), dtype=torch.float64, device="cuda")
        with torch.cuda.stream(stream):
            for _ in range(2):
                pool.estimates_dev(rec)
                dist.all_gather_into_tensor(out, rec)
            barrier()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(stream)
            for _ in range(5):
                pool.estimates_dev(rec)
                dist.all_gather_into_tensor(out, rec)
            a1.record(stream)
        barrier()
        ag = torch.tensor([a0.elapsed_time(a1) / 5], dtype=torch.float64, device="cuda")
        dist.all_reduce(ag, op=dist.ReduceOp.MAX)
        allgather = {"ms": float(ag.item()), "bytes_per_rank": n * 104, "records": "pose7|twist6 per target",
                     "bus_gbs": (world - 1) * n * 104 / (float(ag.item()) * 1e-3) / 1e9}

    # ---- BASELINE configs[4]: mixed models sharded by id (+ the NCCL all-gather of [pose7 | twist6] records at N > 1), every rank ----
    c5 = None
    if not args.no_c5:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_mixed
            c5 = bench_mixed.run_c5(rank, world, local_rank, stream, args.c5_targets, 16, 3, barrier=barrier)
        except Exception as e:   # a collective inside may leave the other ranks waiting: report and let the watchdog decide
            c5 = {"error": ("%s: %s" % (type(e).__name__, e))[:300]}
        torch.cuda.synchronize()

    # ---- BASELINE configs[1] literally: 10k targets, L2-resident, launch-bound (reported, not the headline) ----
    small = None
    if rank == 0 and not args.no_small:
        ns = 10000
        sp, _, p0s, _ = make_pool(te, torch, model, ns, 0, 1, stream, args.variant)
        ms_, as_ = make_inputs(torch, p0s, 2, stride, 0.05, 99)
        for k in range(20):
            sp.step_dense(DT, ms_[k % 2], stride, as_[k % 2])
        torch.cuda.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        Ks = 1000
        s0.record(stream)
        for k in range(Ks):
            sp.step_dense(DT, ms_[k % 2], stride, as_[k % 2])
        s1.record(stream)
        torch.cuda.synchronize()
        sms = s0.elapsed_time(s1)
        small = {"targets": ns, "ticks": Ks, "us_per_tick": 1e3 * sms / Ks, "value": ns * Ks / (sms * 1e-3), "unit": UNIT,
                 "note": "state 7.2 MB is L2-resident; back-to-back launches on one stream"}
        # the same 10k targets in replay launches: 64 buffered ticks per launch, tiles stay on chip across ticks
        T = 64
        mt = torch.stack([ms_[k % 2] for k in range(T)]).contiguous()
        at = torch.stack([as_[k % 2] for k in range(T)]).contiguous()
        for _ in range(3):
            sp.step_dense_ticks(T, DT, mt, stride, at)
        torch.cuda.synchronize()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        Kr = 50
        r0.record(stream)
        for _ in range(Kr):
            sp.step_dense_ticks(T, DT, mt, stride, at)
        r1.record(stream)
        torch.cuda.synchronize()
        rms = r0.elapsed_time(r1)
        small["replay64"] = {"ticks_per_launch": T, "launches": Kr, "us_per_tick": 1e3 * rms / (Kr * T), "value": ns * Kr * T / (rms * 1e-3),
                             "unit": UNIT, "note": "te_pool_step_dense_ticks: 64 buffered ticks per launch (batched ingestion / catch-up)"}
        # live launch (te_pool_live_*): the same 10k targets held in registers by ONE resident launch, ticks released one by one.
        # (a) closed loop through the host: release tick k (a 4-byte write on the copy stream), spin until the launch reports it
        # applied, release the next -- the round trip a 250 Hz loop sees; (b) ticks released as fast as the host can write the
        # gate, waited for at the end -- the rate at which the launch drains ticks that arrive faster than it can apply them
        try:
            Tl = 512
            ml = torch.stack([ms_[k % 2][:, :3] for k in range(Tl)]).contiguous()
            al = torch.stack([as_[k % 2] for k in range(Tl)]).contiguous()
            pl = torch.zeros((Tl, ns, 3), dtype=torch.float64, device="cuda")
            torch.cuda.synchronize()
            L_ = te.lib
            sp.live_begin(Tl, DT, ml, 3, al, 2, pl)
            for k in range(32):
                sp.live_release(k + 1); sp.live_wait(k + 1)
            t0 = time.perf_counter()
            for k in range(32, 32 + 200):
                L_.te_pool_live_release(sp._h, k + 1)
                L_.te_pool_live_wait(sp._h, k + 1)
            closed = (time.perf_counter() - t0) / 200
            t0 = time.perf_counter()
            L_.te_pool_live_release(sp._h, Tl)           # every remaining tick at once: the rate at which the launch drains its ring
            L_.te_pool_live_wait(sp._h, Tl)
            burst = (time.perf_counter() - t0) / (Tl - 232)
            done = sp.live_end()
            # the same closed loop with one launch per tick: launch, wait for it, launch the next
            for k in range(20):
                sp.step_dense(DT, ms_[k % 2], stride, as_[k % 2]); sp.sync()
            t0 = time.perf_counter()
            for k in range(200):
                sp.step_dense(DT, ms_[k % 2], stride, as_[k % 2]); sp.sync()
            launch_loop = (time.perf_counter() - t0) / 200
            small["live"] = {"ticks": done, "closed_loop_us_per_tick": 1e6 * closed, "closed_loop_value": ns / closed,
                             "closed_loop_one_launch_per_tick_us": 1e6 * launch_loop,
                             "drain_us_per_tick": 1e6 * burst, "drain_value": ns / burst, "unit": UNIT,
                             "note": "te_pool_live_*: one resident launch, every target in registers between ticks, ticks released by a store to a "
                                     "page-locked word (no CUDA call per tick); closed loop = the host releases a tick, spins until the launch reports "
                                     "it applied, releases the next (closed_loop_one_launch_per_tick_us: te_pool_step_dense + te_pool_sync per tick, "
                                     "same Python loop); drain = all remaining ticks released at once: the launch's own rate per tick (gate, "
                                     "measurement block, tick, positions, completion count)"}
        except Exception as e:   # secondary figure: report, do not fail the bench
            small["live"] = {"error": ("%s: %s" % (type(e).__name__, e))[:300]}
            try:
                sp.live_end()
            except Exception:
                pass
        # the per-tick launches again, captured once into a CUDA graph (100 ticks) and replayed: the host's launch cost per
        # tick (Python + ctypes + cudaLaunchKernel, what the loop above is bound by) leaves the measurement
        try:
            g = torch.cuda.CUDAGraph()
            Tg = 100
            with torch.cuda.graph(g, stream=stream):
                for k in range(Tg):
                    sp.step_dense(DT, ms_[k % 2], stride, as_[k % 2])
            for _ in range(3):
                g.replay()
            torch.cuda.synchronize()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            Kg = 20
            with torch.cuda.stream(stream):
                g0.record(stream)
                for _ in range(Kg):
                    g.replay()
                g1.record(stream)
            torch.cuda.synchronize()
            gms = g0.elapsed_time(g1)
            small["cuda_graph"] = {"ticks_per_graph": Tg, "replays": Kg, "us_per_tick": 1e3 * gms / (Kg * Tg), "value": ns * Kg * Tg / (gms * 1e-3),
                                   "unit": UNIT, "note": "same one-launch-per-tick kernels, 100 ticks captured in a CUDA graph"}
        except Exception as e:   # capture unsupported in this environment: report, do not fail the bench
            small["cuda_graph"] = {"error": str(e)[:200]}
        sp.close()

    # ---- parity_check: sampled targets of THIS pool after everything above, against the oracle replaying the same history ----
    parity = None
    if rank == 0 and not args.no_parity:
        from tests import orc, synth
        rng = np.random.default_rng(5)
        ns = min(n, 1024)
        sample = np.unique(np.concatenate([np.arange(min(n, 32)), np.arange(max(0, n - 40), n), rng.choice(n, ns, replace=False)]))
        ids_s = (sample.astype(np.int64) * world + rank).astype(np.uint32)
        st = torch.from_numpy(sample).cuda()
        meas_s = [m[st].cpu().numpy() for m in meas]
        act_s = [a_[st].cpu().numpy() for a_ in act]
        full = np.zeros((len(history), sample.size, 7))
        full[:, :, 6] = 1.0
        acts = np.zeros((len(history), sample.size), dtype=np.uint8)
        for j, h in enumerate(history):
            full[j, :, :stride] = meas_s[h]
            acts[j] = act_s[h]
        _, _, Qm, Rm, P0m = te.load_model(model)
        ref = orc.ShardedManager()
        ref.init_batch(mtype, ids_s, DT, Qm, Rm, P0m, p0[sample], p0_scale[sample])
        ref.step_ticks(ids_s, DT, full, acts)
        want = ref.states(ids_s, N)
        got = pool.read_state(ids_s)
        rx, rx6 = synth.compare_both(got["x"], want["x"])
        rP, rP6 = synth.compare_both(got["P"], want["P"])
        exact = bool(np.array_equal(got["n_meas"], want["n_meas"]) and np.array_equal(got["t"], want["t"]))
        parity = {"n": int(sample.size), "ticks_replayed": len(history), "max_ratio": max(rx, rP), "max_ratio_x": rx, "max_ratio_P": rP,
                  "max_ratio_floor1e-6": max(rx6, rP6), "t_and_n_meas_exact": exact, "pass": bool(max(rx, rP) <= 1.0 and exact),
                  "bar": "|d| <= 1e-9 * max(|ref_ij|, 1e-4 * max|ref|) per state vector / covariance matrix (tests/synth.py compare_h2); "
                         "max_ratio = worst |d| / bound over the sampled targets of the %d-target pool after every tick of this run "
                         "(resident-input ticks, clock burst, e2e ticks), oracle = oracle/ port replaying the copied-back inputs" % n}
        ref.close()

    cpu = None
    if rank == 0 and not args.no_cpu:
        from tests import orc
        cores = orc.lib().orc_hardware_threads()
        r1 = cpu_run(model, 1, args.cpu_seconds * 0.3)
        rN, both = cpu_best(model, cores, args.cpu_seconds * 0.7)
        cpu = {"value": rN["value"], "unit": UNIT, "cores": cores, "kind": rN["kind"],
               "sample": "%d %s targets x %d ticks, one TargetManager per thread (id %% %d), the faster of the oracle port and the reference's own "
                         "sources on the stand-in Eigen (oracle/_ref); 1-thread port figure: %.4g %s over %d ticks"
               % (rN["targets"], short, rN["ticks"], cores, r1["value"], UNIT, r1["ticks"]),
               "single_thread_value": r1["value"], "both": both}

    if rank == 0:
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_max / K,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
               "config": make_config(model, n, world, args.variant, n_sets, stride),
               "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                            "peak_source": peak_src, "kernel": KERNEL_NAME.get(model, "te::kf_step_kernel") + "<%s>" % short, "alg_bytes_per_launch": alg_bytes,
                            "alg_bytes_per_update_step": B_upd, "alg_bytes_per_predict_step": B_pred, "kernel_ms": ms / K,
                            "layout": {"bytes_per_update_step": L_upd, "bytes_per_predict_step": L_pred, "bytes_per_launch": layout_bytes,
                                       "achieved": achieved_layout, "frac": achieved_layout / peak, "note": layout_note +
                                       "; `frac` above uses the contract's full-matrix bytes and can therefore exceed 1, this one is the HBM utilisation"}},
               "clocks": clocks, "gpu_launches": K, "e2e": e2e, "cpu_baseline": cpu, "parity_check": parity, "c2_10k": small}
        if allgather:
            out["allgather"] = allgather
        if c5 is not None:
            out["c5"] = c5
        if world == 1 and not args.no_node_loop:
            # Secondary figures (NOT the headline), all in ONE process of their own -- whatever happens there cannot take the headline
            # line with it (tools/bench_configs.py benchline):
            #   c3         BASELINE configs[2]: 1 Mi ANGULAR-RATES targets through the reference's node loop -- /tf records from pinned host
            #              memory into the device-resident mailboxes, first-sight init, sticky update / predict, expiry, 1 % id churn per tick
            #   node_loop  the same loop for the benchmarked motion model
            #   c4_*       BASELINE configs[3]: 1 Mi uniform-velocity targets + one IntersectionSolver query per target per tick (reference
            #              semantics: c4 == 0, every query returns -1) and the same on 1 Mi uniform-acceleration targets (quartic path)
            try:
                import subprocess
                tool = os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools", "bench_configs.py")
                env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(local_rank)))
                pr = subprocess.run([sys.executable, tool, "benchline", model], capture_output=True, text=True, timeout=420, env=env)
                r = json.loads(pr.stdout.strip().splitlines()[-1])
                keep = ("model", "targets", "ticks", "erased", "added", "records_per_tick", "h2d_bytes_per_tick", "records_in", "ms_per_tick", "target_steps_per_s",
                        "ms_per_tick_median", "ms_per_tick_worst", "ms_per_tick_parts", "note", "error")
                for key in ("c3", "node_loop", "c3_sync", "node_loop_sync"):
                    if key in r:
                        out[key] = {k_: r[key][k_] for k_ in keep if k_ in r[key]}
                if "node_loop" not in out and "c3" in out:
                    out["node_loop"] = out["c3"]
                out["c4"] = {"uniform_velocity": r.get("c4_uniform_velocity"), "uniform_acceleration": r.get("c4_uniform_acceleration"),
                             "note": "1 Mi targets, one query per target per tick, queries and results device resident; UV returns -1 for every query by "
                                     "reference semantics (src/intersection_solver.cpp:72: c4 == 0), UA exercises the quartic path"}
            except Exception as e:   # secondary figures: report, never fail the headline
                out["c3"] = {"error": ("%s: %s" % (type(e).__name__, e))[:300]}
        print(json.dumps(out), flush=True)
    pool.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
