#!/usr/bin/env python
"""bench.py -- throughput of the B200 NCC matcher on BASELINE.json's headline configuration.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --steps K --warmup W --dump-outputs DIR  (also writes the last timed step's results to DIR/*.npy)

Workload (config.workload = "cfg1"): 4024x3036 u8 source (seeded synthetic stand-in for the missing
Src7.bmp: blurred noise + Dst7 at three jittered README poses), the real 762x521 Dst7 template,
TargetNum 3, Score 0.8, ToleranceAngle 180, MinReducedArea 256.  One "step" = one pass of
TemplateMatcher::match over a batch of `--batch` frames per GPU.

value  : images/sec, whole job, frames resident in HBM when the timed region starts.
e2e    : same metric through the C ABI with HOST (pinned) frames, H2D + D2H inside the timed region.
p50_ms_per_match: wall-clock around one fpm_match call with a HOST frame (pinned and pageable), like the reference's own
         timer around match() (src/TemplateMatcher.cpp:117,403-404).
roofline / cpu_baseline: see DESIGN.md "Measurement".

    python bench.py --mode latency [--workload cfg5]        (torchrun for N>1)
the angle-sharded latency mode (BASELINE.json config 5): ONE frame, N GPUs, fpm_match_sharded (two ncclAllGather calls on
device buffers); prints p50 ms/match at N GPUs with the single-GPU p50 of the same run beside it.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True        # the bench writes nothing into the tree (which may be read-only)

METRIC = "images/sec (4024x3036 src, 762x521 tpl, +-180deg)"
UNIT = "images/s"
WORKLOADS = {
    # BASELINE.json configs; cfg1 is the one the metric is quoted on (the default), the others are informational
    "cfg1": dict(w=4024, h=3036, tpl="762x521 (Dst7.bmp)", max_pos=3, score=0.8, tol=180.0, mra=256, overlap=0.0, batch=64,
                 expect=3, metric="images/sec (4024x3036 src, 762x521 tpl, +-180deg)"),
    "cfg2": dict(w=3648, h=3648, tpl="54x54 (Dst10.jpg)", max_pos=200, score=0.7, tol=0.0, mra=256, overlap=0.0, batch=32,
                 expect=205, metric="images/sec (3648x3648 src, 54x54 tpl x576, angle 0, TargetNum 200)"),
    "cfg3": dict(w=4096, h=3000, tpl="848x446 (Dst6.bmp)", max_pos=15, score=0.8, tol=180.0, mra=256, overlap=0.0, batch=32,
                 expect=15, metric="images/sec (Src6.jpg 4096x3000, Dst6 848x446, +-180deg, TargetNum 15)"),
    "cfg4": dict(w=4096, h=3072, tpl="512x512 synthetic", max_pos=4, score=0.8, tol=180.0, mra=256, overlap=0.0, batch=32,
                 expect=4, metric="images/sec (4096x3072 synthetic, 512x512 tpl, +-180deg)"),
    "cfg5": dict(w=8192, h=8192, tpl="1024x1024 synthetic", max_pos=4, score=0.8, tol=180.0, mra=256, overlap=0.0, batch=8,
                 expect=4, metric="images/sec (8192x8192 synthetic, 1024x1024 tpl, +-180deg)"),
}


# ------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------
def make_frames(n_distinct: int, seed0: int, workload: str = "cfg1"):
    """(template, [n, H, W] frames) of a BASELINE.json config (SURVEY.md 8d): seeded synthetic sources, real templates"""
    import numpy as np
    import fpm_workloads as synth
    if workload == "cfg1":
        tpl = synth.load_fixture("Dst7")
        frames = [synth.cfg1_source(seed=seed0 + i, tpl=tpl, jitter=True, fast=True) for i in range(n_distinct)]
    elif workload == "cfg2":
        tpl = synth.load_fixture("Dst10")
        frames = [synth.cfg2_source(seed=seed0 + i, tpl=tpl) for i in range(min(n_distinct, 2))]
    elif workload == "cfg3":
        tpl = synth.load_fixture("Dst6")
        frames = [synth.load_fixture("Src6")]
    elif workload == "cfg4":
        tpl = synth.synth_template(512, 4)
        frames = [synth.synth_frame(4096, 3072, tpl, seed0 + i, 4, fast=True) for i in range(n_distinct)]
    elif workload == "cfg5":
        tpl = synth.synth_template(1024, 4)
        frames = [synth.synth_frame(8192, 8192, tpl, seed0 + i, 4, fast=True) for i in range(min(n_distinct, 2))]
    else:
        raise ValueError(workload)
    return tpl, np.stack(frames)


def configure(m, wl):
    m.setMaxPositions(wl["max_pos"]); m.setScore(wl["score"]); m.setToleranceAngle(wl["tol"])
    m.setMinReduceArea(wl["mra"]); m.setMaxOverlap(wl["overlap"])


# ------------------------------------------------------------------------------------------
# CPU baseline: the oracle (Python/cv2 restatement + SSE2 numerator = the reference's CPU path)
# ------------------------------------------------------------------------------------------
def _cpu_worker(args):
    seed, n_images, wl, workload = args
    import cv2
    import numpy as np  # noqa: F401
    cv2.setNumThreads(1)
    tpl, frames = make_frames(min(n_images, 2), seed, workload)
    try:                                                # CPU Baseline A: the C++ restatement, the reference's Release flags
        from oracle.cpu_match import CpuMatcher
        m = CpuMatcher()
        impl = "cpp"
    except Exception:                                   # not built: the Python/cv2 oracle
        from oracle.oracle import OracleMatcher
        m = OracleMatcher()
        impl = "python"
    m.max_pos, m.score, m.tolerance_angle, m.min_reduce_area, m.max_overlap = wl["max_pos"], wl["score"], wl["tol"], wl["mra"], wl["overlap"]
    m.learn_pattern(tpl)
    m.match(frames[0])                                  # warm-up (page-in)
    t0 = time.perf_counter()
    found = 0
    for i in range(n_images):
        found += len(m.match(frames[i % len(frames)]))
    return time.perf_counter() - t0, found, impl


def cpu_throughput(wl, workers: int, images_per_worker: int, workload: str = "cfg1"):
    """images/sec of the CPU oracle with `workers` processes (one single-threaded matcher each)."""
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    with ctx.Pool(workers) as pool:
        t0 = time.perf_counter()
        res = pool.map(_cpu_worker, [(100 + 10 * r, images_per_worker, wl, workload) for r in range(workers)])
        wall = time.perf_counter() - t0
    busy = max(r[0] for r in res)
    total = workers * images_per_worker
    global CPU_IMPL_NAME
    CPU_IMPL_NAME = CPU_IMPL_NAMES[res[0][2]]
    return total / busy, busy, wall, sum(r[1] for r in res)


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def bind_to_gpu_numa(local_rank: int):
    """Best effort: run this rank (and first-touch its pinned frame buffers) on the NUMA node of its GPU, so that the
    H2D DMA does not cross the socket interconnect.  Returns a short description for the JSON line."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        dev = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev)
        node = int(open(path).read().strip())
        if node < 0:
            return "numa node unknown"
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return "numa node %d (%d cpus)" % (node, len(allowed))
        return "numa node %d (no allowed cpus)" % node
    except Exception as e:  # pragma: no cover
        return "not bound (%s)" % type(e).__name__


# ------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
def emit(line: dict):
    """the ONE JSON line on the real stdout (fd 1 is pointed at stderr while the bench runs, so that banners
    printed by NCCL / torchrun children / libraries cannot pollute it)"""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def workload_config(workload: str, wl: dict, batch: int) -> dict:
    """the `config` object: identical in both arms (it names the workload, not the implementation)"""
    return {"workload": workload, "src": "%dx%d" % (wl["w"], wl["h"]), "tpl": wl["tpl"], "target_num": wl["max_pos"],
            "score": wl["score"], "tolerance_angle": wl["tol"], "min_reduce_area": wl["mra"], "max_overlap": wl["overlap"],
            "batch_per_gpu": batch,
            "l2": "step input %.0f MB > 126 MB L2; two alternating sets of distinct frames" % (batch * wl["w"] * wl["h"] / 1e6)}


def int8_peak_measured():
    """u8 x u8 -> s32 tensor-core peak of this GPU: scripts/int8_peak.cu run live (1 s), else the committed measurement"""
    exe = os.path.join(ROOT, "scripts", "_bin", "int8_peak")
    try:
        out = subprocess.run([exe], capture_output=True, text=True, timeout=60)
        d = json.loads(out.stdout.strip().splitlines()[-1])
        d["source"] = "scripts/int8_peak.cu, run live before the timed region"
        return d
    except Exception:
        pass
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_int8_peak.json")))
        d["source"] = "profiles/r02_int8_peak.json (scripts/int8_peak.cu on this pool's B200)"
        return d
    except Exception:
        return None


def dump_outputs(out_dir: str, res, counts, B: int, cap: int):
    """What one batch match hands its caller, as float64 .npy files: counts.npy [B] targets per frame, results.npy
    [B, cap, 12] (score, angle, cx, cy, lt, rt, rb, lb per target; slots past a frame's count are zero)."""
    import numpy as np
    n = np.frombuffer(counts, dtype=np.int32, count=B).copy()
    rows = np.frombuffer(res, dtype=np.float64, count=B * cap * 12).reshape(B, cap, 12).copy()
    rows[np.arange(cap)[None, :] >= n[:, None]] = 0.0
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "counts.npy"), n.astype(np.float64))
    np.save(os.path.join(out_dir, "results.npy"), rows)


def percentile(v, q):
    v = sorted(v)
    if not v:
        return None
    k = (len(v) - 1) * q
    lo, hi = int(k), min(int(k) + 1, len(v) - 1)
    return v[lo] + (v[hi] - v[lo]) * (k - lo)


def run_reference_arm(args, wl, METRIC):
    cores = host_cores()
    per_worker = max(1, args.cpu_images or 8)
    vals, times = [], []
    for _ in range(max(args.steps, 1)):
        v, busy, wall, found = cpu_throughput(wl, cores, per_worker, args.workload)
        vals.append(v); times.append(busy)
        if sum(times) > 150:                       # bounded: the whole run must end within minutes
            break
    value = (cores * per_worker * len(vals)) / sum(times)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(vals),
        "warmup": args.warmup, "ms_per_step": 1000.0 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args.workload, wl, args.batch),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d steps x %d processes x %d frames; %s, one single-threaded matcher per core "
                                   "(the reference's full match() needs OpenCV C++/Qt, unbuildable here)"
                                   % (len(vals), cores, per_worker, CPU_IMPL_NAME)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)
    return 0


CPU_IMPL_NAMES = {
    "cpp": "CPU Baseline A = oracle/cpu_match.cpp, a C++ restatement of TemplateMatcher::match with the reference's SSE2 IM_Conv_SIMD, "
           "built with the reference's Release flags (-O3 -ffast-math -msse4.2 -mavx2 ...), over C++ models of the OpenCV calls",
    "python": "Python/cv2 4.13 oracle + SSE2 IM_Conv_SIMD restatement",
}
CPU_IMPL_NAME = CPU_IMPL_NAMES["cpp"]


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=0, help="frames per GPU per step (0 = workload default: 64 for cfg1)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="throughput", choices=["throughput", "latency"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--samples", type=int, default=200, help="matches per p50 latency figure")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--device-steps-only", action="store_true",
                    help="run only warm-up + timed device-resident steps and exit (clean launch list for ncu; prints no bench line)")
    ap.add_argument("--cpu-images", type=int, default=0, help="images per worker for the CPU baseline (0 = auto)")
    ap.add_argument("--h2d-chunk", type=int, default=0, help="frames per H2D chunk of the e2e path (0 = library default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed device-resident step to DIR/*.npy (throughput mode)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.mode != "throughput" or args.device_steps_only):
        ap.error("--dump-outputs needs the default throughput run (--impl b200 --mode throughput)")
    if args.workload is None:
        args.workload = "cfg5" if args.mode == "latency" else "cfg1"
    wl = WORKLOADS[args.workload]
    METRIC = wl["metric"]
    if args.batch <= 0:
        args.batch = wl["batch"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    # ---------------- reference arm: the CPU implementation on all host cores -----------------
    if args.impl == "reference":
        if rank != 0:
            return 0
        return run_reference_arm(args, wl, METRIC)
    if args.mode == "latency":
        return run_latency(args, wl, rank, world, local_rank)

    # ---------------- CPU baseline first (before CUDA is initialised in this process) ----------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.device_steps_only:
        cores = host_cores()
        workers = cores
        per_worker = args.cpu_images or 48        # ~10 s of CPU work per core on cfg1
        v, busy, wall, found = cpu_throughput(wl, workers, per_worker, args.workload)
        cpu_baseline = {"value": v, "unit": UNIT, "cores": workers, "kind": "port",
                        "sample": "%d processes x %d frames of the workload (%.1f s); %s, "
                                  "single-threaded per process like the reference's own loops" % (workers, per_worker, busy, CPU_IMPL_NAME),
                        "single_core_ms_per_match": 1000.0 * busy / per_worker}

    import numpy as np
    import torch
    import ctypes as C
    from fastest_image_pattern_matching_b200 import TemplateMatcher
    from fastest_image_pattern_matching_b200 import _lib as L

    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        dist = None
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa(local_rank) if world > 1 else "single process, not bound"
    B, K, W = args.batch, args.steps, max(args.warmup, 3)
    int8_peak = int8_peak_measured() if rank == 0 and not args.device_steps_only else None

    # distinct frames: B frames per step, every one its own seeded scene; 12.2 MB each -> one step reads 782 MB (> 126 MB
    # L2), and the steps alternate between two such sets so nothing survives in L2 from one step to the next
    n_distinct = B if args.workload in ("cfg1", "cfg4") else 2
    H, Wd = wl["h"], wl["w"]
    pitch = (Wd + 127) // 128 * 128
    dev_sets, host_sets = [], []
    tpl = None
    for s in range(2):
        tpl, frames_np = make_frames(n_distinct, 1000 * (rank + 1) + 100 * s, args.workload)
        assert frames_np.shape[1:] == (H, Wd)
        src = torch.from_numpy(frames_np)
        d = torch.empty((B, H, pitch), dtype=torch.uint8, device="cuda")
        hbuf = torch.empty((B, H, Wd), dtype=torch.uint8).pin_memory()
        for b in range(B):
            d[b, :, :Wd].copy_(src[(b + s) % src.shape[0]])
            hbuf[b].copy_(src[(b + s) % src.shape[0]])
        dev_sets.append(d)
        host_sets.append(hbuf)
        del frames_np, src

    m = TemplateMatcher(local_rank, result_capacity=16 if wl["expect"] <= 16 else 256)
    configure(m, wl)
    assert m.learnPattern(tpl)
    if args.h2d_chunk:
        m.setH2DChunk(args.h2d_chunk)
    if os.environ.get("FPM_TC"):
        m.setTensorCores(int(os.environ["FPM_TC"]))
    if os.environ.get("FPM_SPLIT") is not None:
        m.setSplitBatch(int(os.environ["FPM_SPLIT"]))
    if os.environ.get("FPM_WS_MB"):
        m.setWorkspaceMB(float(os.environ["FPM_WS_MB"]))
    cap = m.result_capacity
    res = (L.fpm_result * (cap * B))()
    counts = (C.c_int * B)()

    def step_device(i):
        d = dev_sets[i & 1]
        m.matchBatchRaw(d.data_ptr(), B, Wd, H, pitch, H * pitch, True, res, counts)

    def step_host(i):
        hb = host_sets[i & 1]
        m.matchBatchRaw(hb.data_ptr(), B, Wd, H, Wd, H * Wd, False, res, counts)

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn):
        """K steps inside ONE timed region (CUDA events on the library's stream, max over ranks)"""
        for i in range(W):
            step_fn(i)
        barrier()
        l0 = m.launchCount()
        m.timerRecord(0)
        t0 = time.perf_counter()
        for i in range(K):
            step_fn(i)
        m.timerRecord(1)
        ms = m.timerElapsedMs()
        wall_ms = (time.perf_counter() - t0) * 1000.0
        launches = m.launchCount() - l0
        barrier()
        ms = max(ms, 0.0)
        if dist:
            t = torch.tensor([ms, wall_ms, float(launches)], device="cuda", dtype=torch.float64)
            tmax = t.clone()
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            tsum = t.clone()
            dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
            return float(tmax[0]), float(tmax[1]), int(tsum[2])
        return ms, wall_ms, launches

    if args.device_steps_only:
        for i in range(max(args.warmup, 1) + K):
            step_device(i)
        torch.cuda.synchronize()
        sys.stderr.write("device-steps-only: %d steps of %d frames done\n" % (max(args.warmup, 1) + K, B))
        if dist:
            dist.destroy_process_group()
        return 0

    # sanity: every frame must yield the expected number of targets
    step_device(0)
    found = [counts[b] for b in range(B)]
    ok_found = all(f == wl["expect"] for f in found)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    dev_ms, dev_wall_ms, launches = timed(step_device)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, counts, B, cap)
    e2e_ms, e2e_wall_ms, _ = timed(step_host)
    clocks = sampler.stop() if rank == 0 else None

    # raw pinned-host -> device copy rate of one step's frames (context for e2e: the PCIe bound)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    scratch = torch.empty_like(host_sets[0], device="cuda")
    scratch.copy_(host_sets[0], non_blocking=True)
    ev0.record()
    for _ in range(3):
        scratch.copy_(host_sets[0], non_blocking=True)
    ev1.record()
    torch.cuda.synchronize()
    h2d_gbps = 3 * B * H * Wd / (ev0.elapsed_time(ev1) * 1e-3) / 1e9
    del scratch

    # per-kernel device time over K steps, CUDA events around every launch on the launch stream
    # (whole batch on one handle here: with the two concurrent half-batches of the timed steps the event-bracketed
    #  durations of overlapping kernels would not add up)
    split_default = m.getSplitBatch()
    m.setSplitBatch(0)
    m.setProfile(True)
    m.profileReset()
    for i in range(K):
        step_device(i)
    prof = m.profile()
    m.setProfile(False)
    m.setSplitBatch(split_default)

    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return 0

    total_images = world * B * K
    value = total_images / (dev_ms / 1000.0)
    e2e_value = world * B * K / (e2e_ms / 1000.0)

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    if int8_peak and int8_peak.get("int8_tops_m128n256", 0) > 0:
        int8_tops, int8_src = int8_peak["int8_tops_m128n256"], "measured: " + int8_peak["source"]
    else:
        int8_tops, int8_src = 2.0 * peaks.get("bf16_tflops_sustained", 1400.0), "NOT measured: 2 x bf16_tflops_sustained"

    traffic = {}
    for tf in ("r02_traffic.json", "r01_traffic.json"):
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", tf)))
            if tj.get("config", {}).get("batch_per_gpu") == B and tj.get("config", {}).get("workload") == args.workload:
                traffic = {k: v["dram_bytes_per_launch"] for k, v in tj["kernels"].items()}
                traffic_src = "ncu dram__bytes_read+write per launch, profiles/" + tf
                break
        except Exception:
            pass
    kern = {}
    step_ms = sum(v[0] for v in prof.values()) / max(K, 1)
    for name, (ms, n, work) in prof.items():
        if n == 0:
            continue
        kern[name] = {"ms_per_step": ms / K, "launches_per_step": n / K, "avg_launch_us": 1000.0 * ms / n,
                      "share": (ms / K) / step_ms if step_ms > 0 else None, "work_per_launch": work / n}
    dom = max(kern, key=lambda k: kern[k]["ms_per_step"]) if kern else None
    roofline = None
    if dom:
        kd = kern[dom]
        per_launch_s = kd["avg_launch_us"] * 1e-6
        if "corr" in dom or "top_score" in dom:
            ach = 2.0 * kd["work_per_launch"] / per_launch_s / 1e12
            roofline = {"kernel": dom, "bound": "tensor", "achieved": ach, "peak": int8_tops, "unit": "TFLOP/s", "frac": ach / int8_tops,
                        "traffic": traffic.get(dom), "peak_source": int8_src,
                        "note": "u8xu8->s32; algorithmic ops = 2*49*w*h per eval (SURVEY 8d)"}
        else:
            ach = kd["work_per_launch"] / per_launch_s / 1e9
            roofline = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                        "traffic": traffic.get(dom), "traffic_source": traffic_src if traffic else None,
                        "peak_source": hbm_src}
            if dom.startswith("fpm_warp_kernel"):
                # SURVEY 8d counts this stage in bytes, so the contract's fraction is against HBM -- but HBM is not what limits it
                roofline["limiter"] = ("bilinear gather kernel bound by instruction issue (80 % of peak) and the shared-memory pipe "
                                       "(77 %), not by HBM: its DRAM traffic is 0.6x the algorithmic bytes (ncu: "
                                       "profiles/r02_ncu_final_l0_warp_mma_finalize_summary.txt); 34 thread-instructions per ROI pixel")
    # the HBM-bound stages the north_star names (pyramid, rotation): always reported beside the dominant kernel
    hbm_kernels = {}
    for name in ("fpm_pyrdown_kernel", "fpm_warp_kernel(roi)"):
        if name in kern:
            kd = kern[name]
            ach = kd["work_per_launch"] / (kd["avg_launch_us"] * 1e-6) / 1e9
            hbm_kernels[name] = {"achieved_GBps": ach, "frac_of_hbm_peak": ach / hbm_peak, "traffic": traffic.get(name)}
    # the tensor-core correlation: algorithmic int8 ops against the measured int8 dense peak
    for name in ("fpm_corr_mma_kernel", "fpm_corr_fused_kernel", "fpm_corr_warp_kernel"):
        if name in kern:
            kd = kern[name]
            tops = 2.0 * kd["work_per_launch"] / (kd["avg_launch_us"] * 1e-6) / 1e12
            hbm_kernels[name] = {"achieved_TOPS": tops, "frac_of_int8_peak": tops / int8_tops, "int8_peak_TOPS": int8_tops,
                                 "int8_peak_source": int8_src, "traffic": traffic.get(name)}

    # p50 latency of ONE match through the host API (fpm_match, blocking, results on the host), wall clock around the call
    # like the reference's own timer (src/TemplateMatcher.cpp:117,403-404): pinned and pageable host frame (the Qt caller
    # hands a pageable cv::Mat), and device-resident for reference
    ns = max(args.samples, 20)
    one = (L.fpm_result * cap)()
    n1 = C.c_int(0)
    pageable = np.ascontiguousarray(host_sets[0][0].numpy().copy())

    def lat(fn):
        v = []
        for i in range(5 + ns):
            t0 = time.perf_counter()
            fn(i)
            v.append((time.perf_counter() - t0) * 1000.0)
        return v[5:]
    lib, hnd = m._lib, m._h
    l_pin = lat(lambda i: lib.fpm_match(hnd, host_sets[0][i % B].data_ptr(), Wd, H, Wd, one, cap, C.byref(n1)))
    l_pag = lat(lambda i: lib.fpm_match(hnd, pageable.ctypes.data, Wd, H, Wd, one, cap, C.byref(n1)))
    l_dev = lat(lambda i: m.matchBatchRaw(dev_sets[0][i % B].data_ptr(), 1, Wd, H, pitch, H * pitch, True, res, counts))

    pcie_bound = world * h2d_gbps * 1e9 / (H * Wd)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args.workload, wl, B),
        "run": {"global_batch": world * B, "sharding": "frames over ranks, no data-path collective",
                "concurrent_half_batches": bool(split_default and B >= split_default and wl["tol"] > 0),
                "timed_region_ms": dev_ms, "e2e_timed_region_ms": e2e_ms,
                "distinct_frames_per_set": n_distinct},
        "p50_ms_per_match": percentile(l_pin, 0.5),
        "latency": {"what": "wall clock around one blocking fpm_match call, %d samples" % ns,
                    "host_pinned_p50_ms": percentile(l_pin, 0.5), "host_pinned_p90_ms": percentile(l_pin, 0.9),
                    "host_pageable_p50_ms": percentile(l_pag, 0.5), "host_pageable_p90_ms": percentile(l_pag, 0.9),
                    "device_resident_p50_ms": percentile(l_dev, 0.5), "h2d_bytes": H * Wd},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * H * Wd, "d2h_bytes_per_step": B * cap * 96 + B * 4,
                "ms_per_step": e2e_ms / K, "h2d_copy_only_GBps": h2d_gbps, "host_numa": numa,
                "pcie_bound_images_per_s": pcie_bound, "bound": "h2d", "frac_of_bound": e2e_value / pcie_bound,
                "note": "bound by the host->device copy of the frames (measured copy-only rate of the same pinned buffers); "
                        "at N>1 the ranks share the VM's host memory / PCIe root, see h2d_copy_only_GBps per N"},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": roofline,
        "kernels": kern,
        "hbm_kernels": hbm_kernels,
        "int8_peak_measured": int8_peak,
        "cpu_baseline": cpu_baseline,
        "targets_found_per_frame_ok": ok_found,
        "wall_ms_per_step": dev_wall_ms / K,
    }
    emit(line)
    m.close()
    if dist:
        dist.destroy_process_group()
    return 0


# ------------------------------------------------------------------------------------------
# latency mode: ONE frame, N GPUs, angle-sharded (BASELINE.json config 5)
# ------------------------------------------------------------------------------------------
def run_latency(args, wl, rank, world, local_rank):
    import ctypes as C
    import numpy as np
    import torch
    from fastest_image_pattern_matching_b200 import TemplateMatcher
    from fastest_image_pattern_matching_b200 import dist as D
    from fastest_image_pattern_matching_b200 import _lib as L

    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        dist = None
    torch.cuda.set_device(local_rank)
    ns, W = max(args.samples, 20), max(args.warmup, 3)
    tpl, frames_np = make_frames(1, 4242, args.workload)          # the SAME frame on every rank
    frame = np.ascontiguousarray(frames_np[0])
    H, Wd = frame.shape
    pinned = torch.empty((H, Wd), dtype=torch.uint8).pin_memory()
    pinned.copy_(torch.from_numpy(frame))
    dev = torch.from_numpy(frame).cuda()
    m = TemplateMatcher(local_rank, result_capacity=64)
    configure(m, wl)
    assert m.learnPattern(tpl)
    single = D.results_to_rows(m.match(frame))                     # every rank: plain single-GPU match of the same frame
    D.init_sharded(m, dist)                                        # ncclCommInitRank through the C ABI
    cap = m.result_capacity
    lib, hnd = m._lib, m._h
    out = (L.fpm_result * cap)()
    n = C.c_int(0)

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()

    def check(rc):
        if rc != 0:
            raise RuntimeError(lib.fpm_last_error(hnd).decode())

    def series(fn, collective):
        """p50 of the wall clock around one blocking call; for a collective call every rank runs in lockstep and the
        per-sample time is the max over ranks"""
        v = []
        for i in range(W + ns):
            if collective:
                barrier()
            t0 = time.perf_counter()
            check(fn())
            v.append((time.perf_counter() - t0) * 1000.0)
        v = v[W:]
        if collective and dist:
            t = torch.tensor(v, device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            v = t.tolist()
        return v

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    c0, l0 = m.collectiveCount(), m.launchCount()
    sh_dev = series(lambda: lib.fpm_match_sharded(hnd, dev.data_ptr(), Wd, H, Wd, 1, out, cap, C.byref(n)), True)
    per_match_coll = (m.collectiveCount() - c0) / float(W + ns)
    per_match_launches = (m.launchCount() - l0) / float(W + ns)
    rows = D.results_to_rows(m.matchSharded(ptr=dev.data_ptr(), shape=frame.shape, stride=Wd, on_device=True))
    identical = bool(rows.shape == single.shape and np.array_equal(rows, single))
    sh_pin = series(lambda: lib.fpm_match_sharded(hnd, pinned.data_ptr(), Wd, H, Wd, 0, out, cap, C.byref(n)), True)
    rows = D.results_to_rows(m.matchSharded(ptr=pinned.data_ptr(), shape=frame.shape, stride=Wd))
    identical = identical and bool(rows.shape == single.shape and np.array_equal(rows, single))
    sh_pag = series(lambda: lib.fpm_match_sharded(hnd, frame.ctypes.data, Wd, H, Wd, 0, out, cap, C.byref(n)), True)
    m.setShardUpload(False)
    sh_pin_full = series(lambda: lib.fpm_match_sharded(hnd, pinned.data_ptr(), Wd, H, Wd, 0, out, cap, C.byref(n)), True)
    m.setShardUpload(True)
    clocks = sampler.stop() if rank == 0 else None
    # per-kernel device time of the sharded match on this rank (CUDA events around every launch)
    m.setProfile(True); m.profileReset()
    for _ in range(10):
        barrier()
        check(lib.fpm_match_sharded(hnd, dev.data_ptr(), Wd, H, Wd, 1, out, cap, C.byref(n)))
    prof_sh = {k: v[0] / 10 for k, v in m.profile().items() if v[1]}
    m.setProfile(False)
    if dist:
        ok = torch.tensor([1.0 if identical else 0.0], device="cuda")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        identical = bool(ok.item() > 0)
    barrier()
    # the single-GPU figures of the same run: rank 0 alone, the other ranks wait at the barrier
    one = {}
    if rank == 0:
        one["device_resident"] = series(lambda: lib.fpm_match_batch_device(hnd, dev.data_ptr(), 1, Wd, H, Wd, H * Wd, out, cap, C.byref(n)), False)
        one["host_pinned"] = series(lambda: lib.fpm_match(hnd, pinned.data_ptr(), Wd, H, Wd, out, cap, C.byref(n)), False)
        one["host_pageable"] = series(lambda: lib.fpm_match(hnd, frame.ctypes.data, Wd, H, Wd, out, cap, C.byref(n)), False)
        m.setProfile(True); m.profileReset()
        for _ in range(10):
            check(lib.fpm_match_batch_device(hnd, dev.data_ptr(), 1, Wd, H, Wd, H * Wd, out, cap, C.byref(n)))
        prof_one = {k: v[0] / 10 for k, v in m.profile().items() if v[1]}
        m.setProfile(False)
    barrier()
    if rank == 0:
        p50 = lambda v: percentile(v, 0.5)
        s_dev, s_pin, s_pag = p50(one["device_resident"]), p50(one["host_pinned"]), p50(one["host_pageable"])
        line = {
            "metric": "p50 ms/match (%dx%d src, %s tpl, +-%g deg, one frame angle-sharded over N GPUs)" % (Wd, H, wl["tpl"], wl["tol"]),
            "value": p50(sh_pin), "unit": "ms", "n_gpus": world, "steps": ns, "warmup": W, "ms_per_step": p50(sh_pin),
            "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "mode": "latency",
            "config": dict(workload_config(args.workload, wl, 1), sharding="top-layer angle schedule split contiguously over ranks; "
                           "candidate k -> rank k mod N; 2 ncclAllGather on device buffers (+1 for the row-sliced host frame)"),
            "sharded": {"host_pinned_p50_ms": p50(sh_pin), "host_pinned_p90_ms": percentile(sh_pin, 0.9),
                        "host_pageable_p50_ms": p50(sh_pag), "device_resident_p50_ms": p50(sh_dev),
                        "host_pinned_full_upload_per_rank_p50_ms": p50(sh_pin_full),
                        "collectives_per_match_device_resident": per_match_coll, "kernel_launches_per_match_rank0": per_match_launches,
                        "kernel_ms_rank0": prof_sh, "kernel_ms_sum_rank0": sum(prof_sh.values())},
            "single_gpu": {"host_pinned_p50_ms": s_pin, "host_pageable_p50_ms": s_pag, "device_resident_p50_ms": s_dev,
                           "kernel_ms": prof_one, "kernel_ms_sum": sum(prof_one.values())},
            "speedup_vs_single_gpu": {"host_pinned": s_pin / p50(sh_pin), "host_pageable": s_pag / p50(sh_pag),
                                      "device_resident": s_dev / p50(sh_dev)},
            "results_identical_to_single_gpu_on_every_rank": identical,
            "targets_found": int(single.shape[0]),
            "e2e": {"value": p50(sh_pin), "unit": "ms", "h2d_bytes_per_step": H * Wd // max(world, 1), "d2h_bytes_per_step": cap * 96 + 4},
            "gpu_launches": int(per_match_launches * ns),
            "clocks": clocks,
            "timing": "wall clock around one blocking fpm_match_sharded call (results on the host), barrier before every "
                      "sample, per-sample max over ranks, p50 of %d samples" % ns,
        }
        emit(line)
    m.close()
    if dist:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
