#!/usr/bin/env python
"""Benchmark of the registration hot path (BASELINE.json metric: registrations/sec on 20480-point
KITTI-shaped batches; SURVEY.md 8d defines the inputs and the byte accounting).

    python bench.py --gpus 1 --steps 5 --warmup 3                     # our arm (CUDA)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...                              # CPU arm (oracle port of the Ceres path)
    python bench.py ... --dump-outputs DIR                            # + the last timed step's results as DIR/*.npy

A "step" is one pass of the hot path over one batch: S_local clouds x 20480 points -> on-device
initial guess + front filter + 60 perturbed inits -> batched LM solves -> arg-min pose per cloud
(+ the pose all-gather when N > 1).  Weak scaling: S_local = 512 clouds per GPU, so N = 8 is
BASELINE config 4 (4096 x 20480 x 60) exactly.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BYTES_PER_POINT = 13          # x,y,z float32 + int8 label (SURVEY.md 8d)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="multistart60", choices=["multistart60", "single_init"])
    ap.add_argument("--samples-per-gpu", type=int, default=None)
    ap.add_argument("--points", type=int, default=20480)
    ap.add_argument("--inits", type=int, default=None)
    ap.add_argument("--is-3d", action="store_true")
    ap.add_argument("--cpu-samples", type=int, default=3, help="registrations timed on the host cores")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-repeats", type=int, default=2, help="repetitions of the CPU sample (its run-to-run spread is reported)")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE sub-config records (configs[0..2], 6-DoF)")
    ap.add_argument("--config2-samples", type=int, default=4096)
    ap.add_argument("--ops", action="store_true", help="also time index_max / ball_query (config 3)")
    ap.add_argument("--ops-only", action="store_true", help="only time index_max / ball_query and print that JSON")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step's register_batch returned (rank 0) as DIR/<name>.npy, so that "
                         "two builds can be compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.ops_only):
        ap.error("--dump-outputs dumps the CUDA registration path: it takes neither --impl reference nor --ops-only")
    return args


def workload_shape(args):
    if args.workload == "multistart60":
        return (args.samples_per_gpu or 512), (args.inits or 60)
    return (args.samples_per_gpu or 4096), (args.inits or 1)


def load_measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic(S_local, n_inits, is_2d):
    """DRAM bytes (read + write) of ONE launch of the dominant kernel, from the committed ncu --set full capture
    (profiles/r01_traffic.json, written by scripts/ncu_traffic.py) -- only if it was taken on this workload."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    try:
        with open(p) as f:
            t = json.load(f)
        if t["samples_per_gpu"] == S_local and t["inits"] == n_inits and bool(t["is_2d"]) == bool(is_2d):
            return t["dram_bytes_read"] + t["dram_bytes_write"]
    except Exception:  # noqa: BLE001
        pass
    return None


def load_ncu_fractions(S_local, n_inits, is_2d):
    """What the committed ncu --set full capture of the dominant kernel says about its limiter (SURVEY 8d asks for the
    FP64-ALU fraction next to the bandwidth fraction; VERDICT r1 for l2 / issue / dram as well); None when the capture
    is of another workload."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    try:
        with open(p) as f:
            t = json.load(f)
        if t["samples_per_gpu"] == S_local and t["inits"] == n_inits and bool(t["is_2d"]) == bool(is_2d):
            secs = t["gpu_time_ns"] * 1e-9
            l2_bytes = t.get("lts_t_bytes") or ((t.get("l2_read_sectors_from_l1") or 0) * 32.0)
            return {"issue_frac": (t.get("issue_active_pct") or 0) / 100.0, "fp64_frac": (t.get("fp64_pipe_active_pct") or 0) / 100.0,
                    "dram_frac": (t.get("dram_throughput_pct") or 0) / 100.0,
                    "l2_to_l1_GBps": l2_bytes / secs / 1e9 if secs > 0 else None,
                    "warps_active_frac": (t.get("warps_active_pct") or 0) / 100.0,
                    "lts_t_bytes": t.get("lts_t_bytes"), "dram_bytes": t["dram_bytes_read"] + t["dram_bytes_write"],
                    "source": "profiles/r02_traffic.json (%s)" % t.get("source")}
    except Exception:  # noqa: BLE001
        pass
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region.  nvidia-smi needs a few hundred ms to
    start emitting, so the sampler is started before the warm-up and the samples are filtered to the timed
    window by their timestamps (if fewer than 3 fall inside it, all samples taken under load are used)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def parse(rows):
            sm, mx, reasons = [], [], set()
            for _, ln in rows:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 8:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for n, v in zip(names, f[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            return sm, mx, reasons

        inside = [r for r in self.lines if self.t0 is not None and self.t1 is not None and self.t0 <= r[0] <= self.t1 + 0.05]
        window = "timed region"
        if len(inside) < 3:
            inside, window = self.lines, "warm-up + timed region"
        sm, mx, reasons = parse(inside)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "window": window, "reasons": sorted(reasons)}


def make_host_batch(first_id, S, n_points):
    """Seeded KITTI-shaped clouds (seed = global sample id) in the layout the plugin takes:
    xyz float32 [S,3,Ns], pred int8 [S,Ns]."""
    from deepi2p_b200 import synthetic as syn
    Ns = (n_points + 15) // 16 * 16
    xyz = np.zeros((S, 3, Ns), dtype=np.float32)
    pred = np.full((S, Ns), -1, dtype=np.int8)
    meta = None
    for s in range(S):
        smp = syn.make_sample(first_id + s, n_points)
        xyz[s, :, :n_points] = smp["points"]
        pred[s, :n_points] = smp["pred"]
        meta = smp
    return xyz, pred, meta


def cpu_registrations(first_id, count, n_points, n_inits, is_2d, threads):
    """`count` registrations on the host with the oracle port of the Ceres path: all count x n_inits solves
    are spread over `threads` worker threads (the C++ oracle releases the GIL), then the arg-min per sample.
    Mirrors the reference driver's process-per-solve fan-out (registration_lsq.py:142-186) with every core busy."""
    import oracle
    from concurrent.futures import ThreadPoolExecutor
    from deepi2p_b200 import synthetic as syn
    jobs, per = [], []
    for c in range(count):
        smp = syn.make_sample(first_id + c, n_points)
        iy, pf, lf, _ = oracle.initial_guess(smp["points"], smp["pred"])
        ry, t = syn.make_inits(first_id + c, iy, n_inits)
        per.append((smp, pf, lf, ry, t))
        jobs += [(c, i) for i in range(n_inits)]

    def one(job):
        c, i = job
        smp, pf, lf, ry, t = per[c]
        return oracle.solve(pf, lf, smp["K"], ry[i], t[i], smp["H"], smp["W"], syn.T_LB, syn.T_UB, 500, is_2d,
                            want_residuals=False)

    t0 = time.perf_counter()
    with ThreadPoolExecutor(max(1, threads)) as ex:
        outs = list(ex.map(one, jobs))
    dt = time.perf_counter() - t0
    res = []
    for c in range(count):
        o = outs[c * n_inits:(c + 1) * n_inits]
        costs = np.array([x[1] for x in o])
        best = int(np.argmin(costs))
        res.append(dict(sample=per[c][0], pf=per[c][1], lf=per[c][2], ry=per[c][3], t=per[c][4], P=o[best][0],
                        cost=float(costs[best]), evals=sum(x[3]["unique_evals"] for x in o),
                        params=np.stack([x[4] for x in o]), costs=costs))
    return res, dt


def cpu_batch_size(cores, n_inits):
    """Registrations per CPU step so that every core has ~2 solves to chew on."""
    return max(1, int(math.ceil(2.0 * cores / max(n_inits, 1))))


def run_reference(args):
    """CPU arm: the oracle restatement of solvePGivenK + the 60-init driver on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle  # noqa: F401  (builds the C++ oracle if needed)
    S_local, n_inits = workload_shape(args)
    cores = os.cpu_count() or 1
    is_2d = not args.is_3d
    R = cpu_batch_size(cores, n_inits)
    for w in range(args.warmup):
        cpu_registrations(10_000 + w * R, 1, args.points, min(n_inits, cores), is_2d, cores)
    total_dt, evals = 0.0, 0
    for k in range(args.steps):
        res, dt = cpu_registrations(20_000 + k * R, R, args.points, n_inits, is_2d, cores)
        total_dt += dt
        evals += sum(r["evals"] for r in res)
    value = args.steps * R / total_dt
    line = {
        "impl": "reference", "metric": "registrations/sec", "value": value, "unit": "registrations/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "%s: %d-pt KITTI-shaped clouds x %d inits, max_iter 500, %s" % (
            args.workload, args.points, n_inits, "4-DoF" if is_2d else "6-DoF"),
            "note": "each step = %d registrations (bounded sample of the GPU arm's batch), all %d x %d solves spread "
                    "over %d threads" % (R, R, n_inits, cores)},
        "cpu_baseline": {"value": value, "unit": "registrations/s", "cores": cores, "kind": "port",
                         "sample": "%d steps x %d registrations x %d inits, oracle port of the Ceres path (Ceres itself is "
                                   "not installable offline), %d threads" % (args.steps, R, n_inits, cores)},
        "e2e": {"value": value, "unit": "registrations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "mean_cloud_passes_per_solve": evals / float(args.steps * R * n_inits),
    }
    emit(line)


def make_host_batch_threads(first_id, S, n_points, threads=16):
    """make_host_batch over a thread pool (numpy releases the GIL in the heavy parts); used for the 4096-cloud config."""
    from concurrent.futures import ThreadPoolExecutor
    from deepi2p_b200 import synthetic as syn
    Ns = (n_points + 15) // 16 * 16
    xyz = np.zeros((S, 3, Ns), dtype=np.float32)
    pred = np.full((S, Ns), -1, dtype=np.int8)

    def one(s):
        smp = syn.make_sample(first_id + s, n_points)
        xyz[s, :, :n_points] = smp["points"]
        pred[s, :n_points] = smp["pred"]

    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(one, range(S)))
    return xyz, pred


class SolveTimer:
    """CUDA events recorded by the library right before / after the solver kernel of every launch of this thread
    (dib_profile_solve_events): the dominant kernel is timed INSIDE the timed steps, so kernel_ms <= ms_per_step."""

    def __init__(self, torch, lib):
        self.torch, self.lib = torch, lib
        self.e0 = torch.cuda.Event(enable_timing=True)
        self.e1 = torch.cuda.Event(enable_timing=True)
        self.e0.record(); self.e1.record()                      # creates the underlying cudaEvent_t handles
        torch.cuda.synchronize()

    def __enter__(self):
        self.lib.dib_profile_solve_events(self.e0.cuda_event, self.e1.cuda_event)
        return self

    def __exit__(self, *exc):
        self.lib.dib_profile_solve_events(None, None)

    def ms(self):
        self.e1.synchronize()
        return self.e0.elapsed_time(self.e1)


def run_registration_config(torch, frustum, lib, dev, xyz_d, pred_d, n_points, K_d, H, W, n_inits, is_2d, steps, warmup,
                            flush, peak, smi_index, seed0=1000):
    """Device-resident timing of register_batch on one batch (used for the BASELINE sub-configs): per-step CUDA
    events, solver-kernel events inside the steps, roofline fraction from the solver's own pass counters."""
    S = xyz_d.shape[0]
    sampler = ClockSampler(smi_index)
    sampler.start()
    outs = [None] * max(steps, 1)
    for w in range(max(warmup, 1)):
        outs[w % len(outs)] = frustum.register_batch(xyz_d, pred_d, n_points, K_d, H, W, n_inits=n_inits, seed=seed0 + w,
                                                     max_iter=500, is_2d=is_2d, return_all=True, out=outs[w % len(outs)])
    for k in range(len(outs)):
        if outs[k] is None:
            outs[k] = frustum.register_batch(xyz_d, pred_d, n_points, K_d, H, W, n_inits=n_inits, seed=seed0, max_iter=500,
                                             is_2d=is_2d, return_all=True)
    torch.cuda.synchronize()
    step_ms, kern_ms, tails = [], [], []
    sampler.mark_begin()
    with SolveTimer(torch, lib) as st:
        for k in range(steps):
            flush()
            torch.cuda.synchronize()
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            frustum.register_batch(xyz_d, pred_d, n_points, K_d, H, W, n_inits=n_inits, seed=seed0 + 100 + k, max_iter=500,
                                   is_2d=is_2d, return_all=True, out=outs[k])
            e1.record(); e1.synchronize()
            step_ms.append(e0.elapsed_time(e1))
            kern_ms.append(st.ms())
            tl = frustum.last_solve_timeline(dev, register_shape=(S, n_inits, n_points))
            tails.append((tl[2] - tl[1]) * 1e-6)
    sampler.mark_end()
    clocks = sampler.stop()
    pts_evals = 0.0
    passes_mean = 0.0
    for k in range(steps):
        passes = outs[k]["stats"][:, :, 1].to(torch.float64)
        pts_evals += float((passes * outs[k]["n_pts"].to(torch.float64)[:, None]).sum().item())
        passes_mean += float(passes.mean().item()) / steps
    ms = sum(step_ms) / steps
    kms = sum(kern_ms) / steps
    achieved = BYTES_PER_POINT * pts_evals / (sum(kern_ms) * 1e-3) / 1e9
    return {"value": S / (ms * 1e-3), "unit": "registrations/s", "ms_per_step": ms, "kernel_ms": kms,
            "tail_ms": sum(tails) / steps, "mean_cloud_passes_per_solve": passes_mean,
            "achieved_GBps": achieved, "frac": achieved / peak, "steps": steps, "warmup": max(warmup, 1), "clocks": clocks}


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write every array as out_dir/<name>.npy, integers as float64 (exact), floats as they are.  If they come to more
    than DUMP_MAX_BYTES in all, a fixed seeded sample of the leading (per-cloud) axis is written instead, and the
    sampled row numbers go to sample_rows.npy."""
    arrays = {k: v if v.dtype in (np.float32, np.float64) else v.astype(np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        n = next(iter(arrays.values())).shape[0]
        rows = np.sort(np.random.default_rng(0).choice(n, max(1, n * (DUMP_MAX_BYTES // 2) // total), replace=False))
        arrays = {k: v[rows] for k, v in arrays.items()}
        arrays["sample_rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


_JSON_OUT = None


def emit(line):
    """The ONE JSON line, on the process's original stdout."""
    print(json.dumps(line), file=_JSON_OUT if _JSON_OUT is not None else sys.stdout, flush=True)


def main():
    global _JSON_OUT
    args = parse_args()
    # stdout carries the JSON line and nothing else: libraries that print to file descriptor 1 (NCCL's version banner
    # when NCCL_DEBUG is set in the environment) are sent to stderr, the line goes to a private copy of the descriptor
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    from deepi2p_b200 import frustum, sharding, synthetic as syn, _native

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=dev)
    lib = _native.load()
    peak, peak_src = load_measured_peaks()

    if args.ops_only:
        emit({"ops": bench_ops(torch, dev, peak)})
        return
    S_local, n_inits = workload_shape(args)
    is_2d = not args.is_3d
    n_points = args.points
    xyz_h, pred_h = make_host_batch_threads(rank * S_local, S_local, n_points)
    meta = syn.make_sample(0, 16)
    Kmat, H, W = meta["K"], meta["H"], meta["W"]
    xyz_pin = torch.from_numpy(xyz_h).pin_memory()
    pred_pin = torch.from_numpy(pred_h).pin_memory()
    xyz_d = xyz_pin.to(dev)
    pred_d = pred_pin.to(dev)
    K_d = torch.as_tensor(Kmat, dtype=torch.float64).reshape(1, 9).expand(S_local, 9).contiguous().to(dev)
    n_total = S_local * world
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def flush_l2():
        flush_buf.fill_(1)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    smi_index = vis.split(",")[local_rank].strip() if vis else str(local_rank)

    # result buffers, one set per timed step (register_batch's out= reuse: no allocation inside the timed region)
    n_bufs = max(args.steps, 2)
    outs = [frustum.register_batch(xyz_d, pred_d, n_points, K_d, H, W, n_inits=n_inits, seed=1, max_iter=500, is_2d=is_2d,
                                   return_all=True) for _ in range(n_bufs)]
    gathered = [torch.empty((n_total, 17), dtype=torch.float64, device=dev) for _ in range(2)] if world > 1 else None
    seed_box = [1]

    def step_resident(k):
        seed_box[0] += 1
        out = frustum.register_batch(xyz_d, pred_d, n_points, K_d, H, W, n_inits=n_inits, seed=seed_box[0], max_iter=500,
                                     is_2d=is_2d, return_all=True, out=outs[k % n_bufs])
        if world > 1:
            sharding.gather_poses(out["P"], out["cost"], n_total=n_total, out=gathered[k & 1])

    # ---- warm-up (>= 3), then the timed region: per-step CUDA events, solver-kernel events inside each step
    sampler = ClockSampler(smi_index)
    if rank == 0:
        sampler.start()
    for w in range(max(args.warmup, 0)):
        step_resident(w)
    barrier()
    step_ms, kern_ms, tails = [], [], []
    sampler.mark_begin()
    with SolveTimer(torch, lib) as stimer:
        for k in range(args.steps):
            flush_l2()
            barrier()
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            step_resident(k)
            e1.record(); e1.synchronize()
            step_ms.append(e0.elapsed_time(e1))
            kern_ms.append(stimer.ms())
            tl = frustum.last_solve_timeline(dev, register_shape=(S_local, n_inits, n_points))
            tails.append((tl[2] - tl[1]) * 1e-6)
            ce = frustum.last_solve_cta_end_times(dev, register_shape=(S_local, n_inits, n_points))
            cta_tail = ((ce.astype(np.float64) - float(tl[1])) * 1e-6) if ce is not None and len(ce) else np.zeros(1)
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step_serial = float(t.item()) / args.steps
    value_serial = n_total / (ms_per_step_serial * 1e-3)

    # ---- the headline: the same K steps issued back to back on two alternating streams, ONE bracket around all of
    # them.  The solver is a persistent kernel with one CTA per SM; an SM that has run out of problems releases its CTA,
    # so the next step's CTAs start there while the current step's last long solves finish elsewhere -- the
    # end-of-kernel tail (tail_ms below) of one batch is filled with the head of the next, as in any deployment that
    # registers more than one batch.  Every step still does all of its work on its own inputs/outputs/workspace.
    pipe_streams = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]

    def timed_overlapped(steps):
        flush_l2()
        barrier()
        cur = torch.cuda.current_stream()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for st_ in pipe_streams:
            st_.wait_stream(cur)
        for k in range(steps):
            with torch.cuda.stream(pipe_streams[k & 1]):
                step_resident(k)
        for st_ in pipe_streams:
            cur.wait_stream(st_)
        e1.record(); e1.synchronize()
        tt = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    timed_overlapped(2)                                  # warm-up of the two streams' workspaces
    sampler2 = ClockSampler(smi_index)
    if rank == 0:
        sampler2.start()
        time.sleep(0.4)                                  # nvidia-smi needs a moment before it emits samples
    sampler2.mark_begin()
    ms_total = timed_overlapped(args.steps)
    sampler2.mark_end()
    clocks_overlapped = sampler2.stop() if rank == 0 else None
    # what the headline's last step returned, copied now: the passes below write into the same result buffers
    dumped = ({k: v.cpu().numpy() for k, v in outs[(args.steps - 1) % n_bufs].items()}
              if args.dump_outputs and rank == 0 else None)
    ms_per_step = ms_total / args.steps
    value = n_total / (ms_per_step * 1e-3)
    k_ms = sum(kern_ms) / args.steps
    # per-rank solver-kernel times: separates rank imbalance (slowest rank's kernel) from collective cost
    kr = torch.tensor([k_ms], dtype=torch.float64, device=dev)
    k_ranks = [kr.clone() for _ in range(world)]
    if world > 1:
        dist.all_gather(k_ranks, kr)
    k_ranks = [float(x.item()) for x in k_ranks]

    # ---- roofline of the dominant kernel from the timed steps themselves
    pts_evals = 0.0
    passes_mean = iters_mean = 0.0
    for k in range(args.steps):
        st_k = outs[k % n_bufs]["stats"].to(torch.float64)
        passes = st_k[:, :, 1]
        pts_evals += float((passes * outs[k % n_bufs]["n_pts"].to(torch.float64)[:, None]).sum().item())
        passes_mean += float(passes.mean().item()) / args.steps
        iters_mean += float(st_k[:, :, 0].mean().item()) / args.steps
    alg_bytes = BYTES_PER_POINT * pts_evals / args.steps
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9
    compulsory = float(outs[0]["n_pts"].sum().item()) * BYTES_PER_POINT + S_local * (72 + 8 * 4 * n_inits + 136)

    # ---- end to end through the public API with HOST buffers.  Every step copies ITS inputs from pinned host memory
    # and returns ITS result records to pinned host memory; copies run on a second stream into a second device buffer,
    # so step k+1's host->device copy overlaps step k's solve (double buffering).  One event pair around the K steps.
    copy_stream = torch.cuda.Stream(device=dev)
    comp_streams = pipe_streams                      # consecutive steps alternate between two compute streams (see above)
    x_bufs = [torch.empty_like(xyz_d) for _ in range(2)]
    p_bufs = [torch.empty_like(pred_d) for _ in range(2)]
    out_pins = [torch.empty((n_total, 17), dtype=torch.float64).pin_memory() for _ in range(2)]
    pin_P = [torch.empty((n_total, 4, 4), dtype=torch.float64).pin_memory() for _ in range(2)]
    pin_c = [torch.empty((n_total,), dtype=torch.float64).pin_memory() for _ in range(2)]

    def run_e2e(steps):
        copied = [None, None]
        freed = [None, None]
        for k in range(steps):
            b = k & 1
            with torch.cuda.stream(copy_stream):
                if freed[b] is not None:
                    copy_stream.wait_event(freed[b])          # the solve that last read this buffer is done
                x_bufs[b].copy_(xyz_pin, non_blocking=True)
                p_bufs[b].copy_(pred_pin, non_blocking=True)
                copied[b] = torch.cuda.Event(); copied[b].record(copy_stream)
            comp_stream = comp_streams[b]
            with torch.cuda.stream(comp_stream):
                comp_stream.wait_event(copied[b])
                seed_box[0] += 1
                out = frustum.register_batch(x_bufs[b], p_bufs[b], n_points, K_d, H, W, n_inits=n_inits, seed=seed_box[0],
                                             max_iter=500, is_2d=is_2d, return_all=True, out=outs[k % n_bufs])
                freed[b] = torch.cuda.Event(); freed[b].record(comp_stream)
                if world > 1:
                    sharding.gather_poses(out["P"], out["cost"], n_total=n_total, out=gathered[b])
                    out_pins[b].copy_(gathered[b], non_blocking=True)      # the gathered [S,17] records
                else:
                    pin_P[b].copy_(out["P"], non_blocking=True)           # two plain device->host copies, no kernel
                    pin_c[b].copy_(out["cost"], non_blocking=True)

    def timed_e2e(steps):
        flush_l2()
        barrier()
        cur = torch.cuda.current_stream()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        copy_stream.wait_stream(cur)
        for st_ in comp_streams:
            st_.wait_stream(cur)
        run_e2e(steps)
        cur.wait_stream(copy_stream)
        for st_ in comp_streams:
            cur.wait_stream(st_)
        e1.record(); e1.synchronize()
        tt = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    timed_e2e(2)
    ms_e2e = timed_e2e(args.steps) / args.steps
    e2e_value = n_total / (ms_e2e * 1e-3)
    h2d = xyz_pin.numel() * 4 + pred_pin.numel()
    d2h = n_total * 17 * 8

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    ncu = load_ncu_fractions(S_local, n_inits, is_2d)
    line = {
        "metric": "registrations/sec", "value": value, "unit": "registrations/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {
            "workload": "%s: %d KITTI-shaped clouds/GPU x %d pts x %d inits (%s, max_iter 500); N=8 is BASELINE "
                        "config 4" % (args.workload, S_local, n_points, n_inits, "4-DoF" if is_2d else "6-DoF"),
            "samples_per_gpu": S_local, "points": n_points, "inits": n_inits, "parallelism": "dp%d" % world,
            "why_this_workload": "the per-GPU shard of BASELINE configs[3] (4096 x 20480 x 60 over 8 GPUs), so that "
                                 "N=1,2,4,8 time the same per-GPU work; configs[0], [1], [2] and the 6-DoF variant are the "
                                 "`configs` sub-records of this line",
            "l2": "value and e2e: %d steps issued back to back on two alternating streams inside ONE event bracket (the tail of "
                  "one step's persistent kernel overlaps the head of the next); no flush between them -- each step streams "
                  "136 MB of inputs + a 168 MB packed copy, more than the 126 MB L2; `serial` = the same steps one at a time "
                  "with an L2 flush before each" % args.steps,
            "step": "ONE C-ABI call frustum_register_batch_f32 = prepare (initial guess + front filter + Morton sort + "
                    "Philox inits) + boxes + order + LM solve + arg-min/degenerate rule"
                    + (" + one NCCL all_gather_into_tensor of [S,17] f64" if world > 1 else ""),
        },
        "e2e": {"value": e2e_value, "unit": "registrations/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "vs_resident": e2e_value / value,
                "note": "per step: pinned host xyz f32 + pred int8 -> device buffer (copy stream, double-buffered), "
                        "register_batch, [S,17] poses+cost -> pinned host; step k+1's copy overlaps step k's solve"},
        "gpu_launches": 5 * args.steps,   # prepare, boxes, order, solve, finalize per step -- all this repo's kernels
        "clocks": clocks_overlapped,
        "serial": {"value": value_serial, "unit": "registrations/s", "ms_per_step": ms_per_step_serial, "clocks": clocks,
                   "note": "the same steps one at a time: L2 flushed (256 MiB write) before every step, per-step CUDA events "
                           "summed, max over ranks; the roofline block below is measured on these steps"},
        "roofline": {
            "bound": "issue",
            "bound_note": "limiter per ncu = instruction issue / dependent fp64 latency (profiles/); DRAM moves ~1.3x the "
                          "compulsory bytes. achieved/peak/frac below are SURVEY 8d's streamed-model HBM-equivalent: 13 B x "
                          "points x cloud passes, divided by the measured copy bandwidth",
            "kernel": "frustum_solve_kernel<float,%d>" % (4 if is_2d else 6),
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": k_ms, "kernel_ms_all": kern_ms,
            "kernel_ms_per_rank": {"min": min(k_ranks), "max": max(k_ranks), "all": k_ranks},
            "kernel_timing": "CUDA events recorded by the library around the solver kernel inside each timed step "
                             "(dib_profile_solve_events), rank 0; ms_per_step is the max over ranks",
            "tail_ms": sum(tails) / len(tails),
            "tail_note": "queue empty -> last CTA exit, from the kernel's own globaltimer words",
            "cta_exit_after_queue_empty_ms": {"p10": float(np.percentile(cta_tail, 10)), "p50": float(np.percentile(cta_tail, 50)),
                                              "p90": float(np.percentile(cta_tail, 90)), "max": float(cta_tail.max()),
                                              "mean": float(cta_tail.mean()), "ctas": int(cta_tail.size)},
            "point_evals_per_s": pts_evals / args.steps / (k_ms * 1e-3),
            "mean_cloud_passes_per_solve": passes_mean, "mean_lm_iterations_per_solve": iters_mean,
            "compulsory_bytes_per_launch": compulsory,
            "traffic": load_traffic(S_local, n_inits, is_2d),
            "secondary": ncu,
        },
    }

    # ---- the other BASELINE configs, each a short device-resident run (world == 1 only: they are single-GPU configs)
    if world == 1 and not args.no_configs:
        cfgs = {}
        try:
            cfgs["single_sample_60_calls"] = bench_config1(torch, frustum, lib, dev, n_points, is_2d, flush_l2, peak, smi_index)
        except Exception as e:  # noqa: BLE001
            cfgs["single_sample_60_calls"] = {"error": repr(e)}
        try:
            S2 = args.config2_samples
            x2, p2 = make_host_batch_threads(100000, S2, n_points)
            x2d, p2d = torch.from_numpy(x2).to(dev), torch.from_numpy(p2).to(dev)
            K2 = torch.as_tensor(Kmat, dtype=torch.float64).reshape(1, 9).expand(S2, 9).contiguous().to(dev)
            r = run_registration_config(torch, frustum, lib, dev, x2d, p2d, n_points, K2, H, W, 1, True, 3, 3, flush_l2, peak,
                                        smi_index)
            r["workload"] = "BASELINE configs[1]: %d samples x %d pts x 1 init, 1 GPU" % (S2, n_points)
            cfgs["single_init_4096"] = r
            del x2d, p2d, x2, p2
        except Exception as e:  # noqa: BLE001
            cfgs["single_init_4096"] = {"error": repr(e)}
        try:
            S6 = min(512, S_local)
            r = run_registration_config(torch, frustum, lib, dev, xyz_d[:S6].contiguous(), pred_d[:S6].contiguous(), n_points,
                                        K_d[:S6].contiguous(), H, W, n_inits, False, 2, 2, flush_l2, peak, smi_index)
            r["workload"] = "6-DoF (is_2d=False): %d samples x %d pts x %d inits" % (S6, n_points, n_inits)
            cfgs["sixdof"] = r
        except Exception as e:  # noqa: BLE001
            cfgs["sixdof"] = {"error": repr(e)}
        try:
            cfgs["ops_config3"] = bench_ops(torch, dev, peak)
        except Exception as e:  # noqa: BLE001
            cfgs["ops_config3"] = {"error": repr(e)}
        line["configs"] = cfgs

    # ---- CPU baseline + pose parity on a bounded sample (oracle port, all host cores), THROUGH the product path:
    # the GPU side is register_batch (device initial guess, Morton sort, device-made inits); the oracle gets the original
    # clouds, its own get_initial_guess filter and the same inits
    if not args.no_cpu_baseline and world == 1 and args.cpu_samples > 0:
        line.update(cpu_and_parity(torch, frustum, dev, args, xyz_d, pred_d, n_points, K_d, H, W, n_inits, is_2d))

    if args.ops and "configs" not in line:
        line["ops"] = bench_ops(torch, dev, peak)
    emit(line)
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def bench_config1(torch, frustum, lib, dev, n_points, is_2d, flush, peak, smi_index):
    """BASELINE configs[0]: ONE sample, 60 inits.  (a) exactly as evaluation/registration_lsq.py:132-135 calls the
    extension: 60 sequential FrustumRegistration.solvePGivenK calls with numpy float64 in / (P, cost, residuals) out,
    arg-min on the host -- wall-clocked, because the call is host-synchronous by contract; (b) the batched replacement,
    register_batch(S=1, I=60), device-timed."""
    import importlib
    from deepi2p_b200 import synthetic as syn
    FR = importlib.import_module("deepi2p_b200.dropin.FrustumRegistration")
    smp = syn.make_sample(424242, n_points)
    pts64 = smp["points"].astype(np.float64)
    # host-side get_initial_guess exactly as the reference caller does it (registration_lsq.py:196-220), numpy
    inside = smp["pred"] == 1
    mean = pts64[:, inside].mean(axis=1)
    a = math.fmod(math.atan2(mean[2], mean[0]) - math.pi / 2 + math.pi, 2 * math.pi)
    iy = (a + 2 * math.pi if a < 0 else a) - math.pi
    c, s_ = math.cos(iy), math.sin(iy)
    rz = -s_ * pts64[0] + c * pts64[2]
    keep = rz > rz[inside].min() - 10
    pf, lf = np.ascontiguousarray(pts64[:, keep]), smp["pred"][keep].astype(np.int64)
    ry, t = syn.make_inits(424242, iy, 60)
    lb, ub = list(syn.T_LB), list(syn.T_UB)
    for i in range(3):                                                   # warm-up calls
        FR.solvePGivenK(pf, lf, smp["K"], ry[i], t[i], smp["H"], smp["W"], lb, ub, 500, False, is_2d)
    torch.cuda.synchronize()
    sampler = ClockSampler(smi_index)
    sampler.start()
    sampler.mark_begin()
    reps, walls = 3, []
    for _ in range(reps):
        t0 = time.perf_counter()
        best = None
        for i in range(60):
            P, cost, res = FR.solvePGivenK(pf, lf, smp["K"], ry[i], t[i], smp["H"], smp["W"], lb, ub, 500, False, is_2d)
            if best is None or cost < best[1]:
                best = (P, cost)
        walls.append(time.perf_counter() - t0)
    sampler.mark_end()
    clocks = sampler.stop()
    wall = min(walls)
    # (b) the batched call on the same sample
    Ns = (n_points + 15) // 16 * 16
    xyz1 = np.zeros((1, 3, Ns), dtype=np.float32); xyz1[0, :, :n_points] = smp["points"]
    pred1 = np.full((1, Ns), -1, dtype=np.int8); pred1[0, :n_points] = smp["pred"]
    x1, p1 = torch.from_numpy(xyz1).to(dev), torch.from_numpy(pred1).to(dev)
    K1 = torch.as_tensor(smp["K"], dtype=torch.float64).reshape(1, 9).to(dev)
    rb = run_registration_config(torch, frustum, lib, dev, x1, p1, n_points, K1, smp["H"], smp["W"], 60, is_2d, 5, 3, flush,
                                 peak, smi_index)
    return {"workload": "BASELINE configs[0]: single sample, %d pts, 60 inits" % n_points,
            "dropin_60_sequential_solvePGivenK": {"value": 1.0 / wall, "unit": "registrations/s", "ms_per_registration": wall * 1e3,
                                                   "ms_per_call": wall * 1e3 / 60, "timing": "host wall clock, best of %d x 60 calls "
                                                   "(numpy f64 in, numpy out, residual vector returned every call)" % reps,
                                                   "all_ms": [w * 1e3 for w in walls], "clocks": clocks,
                                                   "best_cost": float(best[1])},
            "register_batch_S1_I60": rb}


def cpu_and_parity(torch, frustum, dev, args, xyz_d, pred_d, n_points, K_d, H, W, n_inits, is_2d):
    import oracle  # noqa: F401
    from concurrent.futures import ThreadPoolExecutor
    from deepi2p_b200 import synthetic as syn
    cores = os.cpu_count() or 1
    count = max(args.cpu_samples, cpu_batch_size(cores, n_inits))
    seed = 777
    g = frustum.register_batch(xyz_d[:count].contiguous(), pred_d[:count].contiguous(), n_points, K_d[:count].contiguous(), H, W,
                               n_inits=n_inits, seed=seed, max_iter=500, is_2d=is_2d, return_all=True)
    inits = g["init"].cpu().numpy()
    gp = g["params"].cpu().numpy()
    gc = g["costs"].cpu().numpy()
    gbest = g["best"].cpu().numpy()
    per, jobs = [], []
    for c_ in range(count):
        smp = syn.make_sample(c_, n_points)          # rank 0, first samples of the batch (seed = global sample id)
        iy, pf, lf, _ = oracle.initial_guess(smp["points"], smp["pred"])
        per.append((smp, pf, lf))
        jobs += [(c_, i) for i in range(n_inits)]

    def one(job):
        c_, i = job
        smp, pf, lf = per[c_]
        return oracle.solve(pf, lf, smp["K"], inits[c_, i, 0], inits[c_, i, 1:4], smp["H"], smp["W"], syn.T_LB, syn.T_UB, 500,
                            is_2d, want_residuals=False)

    dts, outs = [], None
    for _ in range(max(1, args.cpu_repeats)):
        t0 = time.perf_counter()
        with ThreadPoolExecutor(max(1, cores)) as ex:
            outs = list(ex.map(one, jobs))
        dts.append(time.perf_counter() - t0)
    dt = min(dts)
    Pn = 4 if is_2d else 6
    nr = Pn - 3
    op = np.stack([o[4] for o in outs]).reshape(count, n_inits, 6)
    oc = np.array([o[1] for o in outs]).reshape(count, n_inits)
    d_rot = np.linalg.norm(gp[:, :, :nr] - op[:, :, :nr], axis=2).ravel()
    d_tr = np.linalg.norm(gp[:, :, nr:Pn] - op[:, :, nr:Pn], axis=2).ravel()
    within = (d_rot < 1e-4) & (d_tr < 1e-3)
    reg_ok = cost_le = 0
    worst_r = worst_t = 0.0
    for c_ in range(count):
        bo, bg = int(np.argmin(oc[c_])), int(gbest[c_])
        er = float(np.linalg.norm(gp[c_, bg, :nr] - op[c_, bo, :nr])); et = float(np.linalg.norm(gp[c_, bg, nr:Pn] - op[c_, bo, nr:Pn]))
        worst_r, worst_t = max(worst_r, er), max(worst_t, et)
        reg_ok += int(er < 1e-4 and et < 1e-3)
        cost_le += int(gc[c_, bg] <= oc[c_, bo] * (1 + 1e-9))
    res = {"cpu_baseline": {
        "value": count / dt, "unit": "registrations/s", "cores": cores, "kind": "port",
        "sample": "%d registrations x %d inits of the same workload (first samples of the GPU batch, device-made inits), oracle "
                  "port of the Ceres path (Ceres is installed neither here nor on the GPU box: profiles/r02_probe_ceres_gpu_box.txt), "
                  "all solves spread over %d threads, best of %d runs" % (count, n_inits, cores, len(dts)),
        "spread": {"runs_s": dts, "min_value": count / max(dts), "max_value": count / min(dts)}},
        "parity": {
        "gate": "1e-4 rad / 1e-3 m vs the CPU oracle (Ceres unavailable offline)",
        "path": "GPU: register_batch (device initial guess + Morton sort + device-made inits); oracle: original clouds, own "
                "get_initial_guess, same inits",
        "solves": int(within.size), "solves_within_gate": int(within.sum()),
        "solve_median_rot_rad": float(np.median(d_rot)), "solve_median_trans_m": float(np.median(d_tr)),
        "solve_max_rot_rad": float(d_rot.max()), "solve_max_trans_m": float(d_tr.max()),
        "registrations": count, "registrations_within_gate": reg_ok,
        "registrations_gpu_cost_le_oracle": cost_le,
        "best_of_I_max_rot_err_rad": worst_r, "best_of_I_max_trans_err_m": worst_t,
        "note": "trajectories are chaotic at rounding level; every out-of-gate solve of a 1440-solve run is traced to its first "
                "divergent evaluation in profiles/r02_trace_divergence.md"}}
    return res


def bench_ops(torch, dev, peak):
    """BASELINE config 3: index_max + ball_query forward, B=64, C=M=64, N=16384, K=64.
    Inputs are 2 x 268 MB per op (> 126 MB L2) and the timed iterations alternate between two
    distinct input sets, so every byte comes from HBM and no dirty flush lines compete with it."""
    from deepi2p_b200 import point_ops
    B, C, N, K = 64, 64, 16384, 64
    g = torch.Generator(device=dev).manual_seed(0)
    sets = []
    for _ in range(2):
        data = torch.randn((B, C, N), device=dev, generator=g)
        index = torch.randint(0, K, (B, N), device=dev, generator=g, dtype=torch.int32)
        pts = torch.rand((B, N, 3), device=dev, generator=g) * 20
        nodes = torch.rand((B, C, 3), device=dev, generator=g) * 20
        dist_m = torch.cdist(nodes, pts).contiguous()
        sets.append((data, index, dist_m, pts.transpose(1, 2).contiguous(), nodes.transpose(1, 2).contiguous()))
        del pts, nodes
    radius = float(torch.kthvalue(sets[0][2], K, dim=2).values.median().item())

    def t(fn, reps=5, inner=10):
        """Mean device time per launch: `inner` back-to-back launches (alternating input sets) inside one CUDA
        event pair, so that the host's launch latency (Python + ctypes, tens of us) is not billed to a ~60 us
        kernel; repeated `reps` times."""
        for w in range(4):
            fn(w & 1)
        ms = 0.0
        for _ in range(reps):
            torch.cuda.synchronize()
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            for it in range(inner):
                fn(it & 1)
            e1.record(); e1.synchronize()
            ms += e0.elapsed_time(e1) / inner
        return ms / reps

    im_ms = t(lambda i: point_ops.index_max_forward(sets[i][0], sets[i][1], K))
    bq_ms = t(lambda i: point_ops.ball_query_forward(sets[i][2], radius, K))
    xyz_ms = t(lambda i: point_ops.ball_query_xyz_forward(sets[i][3], sets[i][4], radius, K))
    im_bytes = 4 * B * C * N + 4 * B * N + 4 * B * C * K
    # algorithmic bytes of ball_query: up to each row's K-th hit (mean over the two sets)
    bq_bytes = 0.0
    for _, _, dist_m, _, _ in sets:
        csum = (dist_m <= radius).cumsum(2)
        kth = torch.where(csum[:, :, -1] >= K, (csum >= K).float().argmax(2) + 1, torch.full_like(csum[:, :, -1], N))
        bq_bytes += 0.5 * (float(kth.sum().item()) * 4 + 4 * B * C * K)
        del csum, kth
    res = {
        "index_max": {"us": im_ms * 1e3, "GBps": im_bytes / (im_ms * 1e-3) / 1e9, "frac": im_bytes / (im_ms * 1e-3) / 1e9 / peak,
                      "bytes": im_bytes},
        "ball_query": {"us": bq_ms * 1e3, "GBps_algorithmic": bq_bytes / (bq_ms * 1e-3) / 1e9,
                       "frac_algorithmic": bq_bytes / (bq_ms * 1e-3) / 1e9 / peak, "bytes_algorithmic": bq_bytes,
                       "bytes_upper_bound": 4 * B * C * N + 4 * B * C * K, "radius": radius},
        "ball_query_xyz": {"us": xyz_ms * 1e3, "note": "grid-hash radius search from coordinates (grid build + query); reads "
                           "%.1f MB instead of the %.0f MB distance matrix the dense op needs" % (
                               (12 * B * N + 12 * B * C) / 1e6, 4 * B * C * N / 1e6)},
        "shape": {"B": B, "C": C, "M": C, "N": N, "K": K},
        "l2": "two alternating 268 MB input sets per op (> L2), no flush; 10 back-to-back launches per event pair",
    }
    # 8(f) N4: clustering front-end at the shipped encoder shape (kitti/options.py:28-35): B=8, N=20480, Ma=128, k=3
    cb, cn, cm, ck = 8, 20480, 128, 3
    cpc = [(torch.rand((cb, 3, cn), device=dev, generator=g) * 80 - 40) for _ in range(2)]
    cnode = [c[:, :, torch.randperm(cn, device=dev, generator=g)[:cm]].contiguous() for c in cpc]
    ca_ms = t(lambda i: point_ops.cluster_assign_forward(cpc[i], cnode[i], ck))

    def torch_clustering(i):            # the reference's formulation, networks_pc.py:60-82 (torch library ops)
        pc, node = cpc[i], cnode[i]
        diff = torch.norm(pc.unsqueeze(3) - node.unsqueeze(2), dim=1, p=2)
        _, mk = torch.topk(diff, k=ck, dim=2, largest=False, sorted=True)
        mi = mk[:, :, 0]
        mask = torch.eq(mi.unsqueeze(2), torch.arange(cm, device=dev).view(1, 1, cm))
        mf = mask.unsqueeze(1).float()
        mean = torch.sum(pc.unsqueeze(3) * mf, dim=2) / (torch.sum(mf, dim=2) + 1e-5)
        return pc - torch.gather(mean, index=mi.unsqueeze(1).expand(cb, 3, cn), dim=2)

    res["cluster_assign"] = {"us": ca_ms * 1e3, "reference_torch_us": 1e3 * t(torch_clustering, 2, 3),
                             "shape": {"B": cb, "N": cn, "Ma": cm, "k": ck},
                             "bytes": (12 * 2 + 4 * ck + 4 + 24) * cb * cn,
                             "note": "3 launches (assign+sums, means, decenter); inputs are L2-resident at this size, "
                                     "so this is a latency/issue-bound op, not an HBM one; the torch formulation "
                                     "materialises several B x N x Ma tensors"}
    try:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import build_ref
        if build_ref.built("index_max") and build_ref.built("ball_query"):
            ref_im = build_ref.load("index_max")
            ref_bq = build_ref.load("ball_query")
            res["index_max"]["reference_kernel_us"] = 1e3 * t(lambda i: ref_im.forward_cuda_shared_mem(sets[i][0], sets[i][1], K), 2, 3)
            res["ball_query"]["reference_kernel_us"] = 1e3 * t(lambda i: ref_bq.forward_cuda_shared_mem(sets[i][2], radius, K), 2, 3)
    except Exception as e:  # noqa: BLE001
        res["reference_kernels"] = "unavailable: %s" % e
    return res


if __name__ == "__main__":
    main()
