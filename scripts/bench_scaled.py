"""Scale-tolerant matching (FPM_PARAM_SCALE_MIN / MAX) at the ranges [1, 1], [0.9, 1.1] and [0.8, 1.25]:
  batch      device-resident batch of 64 frames, images/s (host clock around calls that end in a device synchronise), the
             three ranges alternating in one process after warm-up
  launches   kernel launches per batch
  kernels    per-kernel device time of one profiled batch (FPM_PARAM_PROFILE)
  found      targets found per frame, and the top-layer candidates of frame 0 (FPM_PARAM_TRACE)
Workloads: cfg1-like (4024 x 3036, the Dst7 template, +-180 deg, Score 0.8, 3 targets) and cfg4-like (2048 x 2048, a 128 x 128
synthetic template, +-180 deg, 4 targets), with seeded instances pasted at scales drawn from [0.8, 1.25] (16 distinct frames,
each used four times).  Writes one JSON file (default profiles/scaled_b200.json) with the card name and power limit.
    python scripts/bench_scaled.py [--out PATH] [--reps 3]"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import fpm_workloads as synth  # noqa: E402
from fastest_image_pattern_matching_b200 import TemplateMatcher  # noqa: E402
from tests.scaled_oracle import paste_scaled  # noqa: E402

RANGES = [(1.0, 1.0), (0.9, 1.1), (0.8, 1.25)]
KERNELS = ("fpm_warp_kernel(top)", "fpm_top_score_kernel", "fpm_top_peaks_kernel", "fpm_collect_sort_kernel", "fpm_warp_kernel(roi)",
           "fpm_corr_rows_kernel", "fpm_corr_mma_kernel", "fpm_corr_fused_kernel", "fpm_refine_finalize_kernel", "fpm_final_kernel")


def card():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                               timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                                   # noqa: BLE001
        power = "unknown (%s)" % e
    return name, power


def frames_for(w, h, tpl, k, seed, n=16):
    rng = np.random.default_rng(seed)
    diag = math.hypot(*tpl.shape) * 1.25
    out = []
    for f in range(n):
        img = synth.background(w, h, seed + f, 3.0)
        centres = []
        while len(centres) < k:
            cx, cy = rng.uniform(diag / 2 + 2, w - diag / 2 - 2), rng.uniform(diag / 2 + 2, h - diag / 2 - 2)
            if all(math.hypot(cx - x, cy - y) >= diag for x, y in centres):
                centres.append((cx, cy))
        for cx, cy in centres:
            r = int(diag / 2) + 3
            x0, y0 = int(cx) - r, int(cy) - r
            sub = img[y0:y0 + 2 * r + 1, x0:x0 + 2 * r + 1]
            paste_scaled(sub, tpl, cx - x0, cy - y0, float(rng.uniform(-180, 180)), float(rng.uniform(0.8, 1.25)))
        out.append(img)
    return np.stack(out)


def run_workload(name, w, h, tpl, k, reps):
    frames = frames_for(w, h, tpl, k, seed=11)
    batch = np.concatenate([frames] * 4)                     # 64 frames
    d = torch.from_numpy(batch).cuda()
    B = batch.shape[0]
    m = TemplateMatcher(0)
    m.setMaxPositions(k); m.setScore(0.8); m.setToleranceAngle(180); m.setMinReduceArea(256)
    assert m.learnPattern(tpl)
    res = {}
    for rng in RANGES:                                       # warm-up, found counts, launches
        m.setScaleRange(*rng)
        l0 = m.launchCount()
        _, n = m.matchBatchRaw(d.data_ptr(), B, w, h, w, w * h, True)
        torch.cuda.synchronize()
        res[rng] = dict(found=[int(n[b]) for b in range(len(frames))], launches_per_batch=m.launchCount() - l0, times=[])
    for _ in range(reps):
        for rng in RANGES:
            m.setScaleRange(*rng)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            m.matchBatchRaw(d.data_ptr(), B, w, h, w, w * h, True)
            torch.cuda.synchronize()
            res[rng]["times"].append(time.perf_counter() - t0)
    for rng in RANGES:
        m.setScaleRange(*rng)
        m.setProfile(True); m.profileReset()
        m.matchBatchRaw(d.data_ptr(), B, w, h, w, w * h, True)
        prof = m.profile()
        m.setProfile(False)
        res[rng]["kernels_ms"] = {kk: round(prof[kk][0], 3) for kk in KERNELS if kk in prof and prof[kk][1] > 0}
        m.setTrace(True)
        m.match(batch[0])
        res[rng]["top_candidates_frame0"] = int(len(m.traceCandidates()))
        m.setTrace(False)
        t = sorted(res[rng].pop("times"))
        res[rng]["images_per_s"] = round(B / t[len(t) // 2], 1)
        res[rng]["images_per_s_all"] = [round(B / x, 1) for x in t]
    m.close()
    return {"%g-%g" % r: v for r, v in res.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "scaled_b200.json"))
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    name, power = card()
    out = dict(gpu=name, power_limit=power, batch=64, ranges=["%g-%g" % r for r in RANGES],
               cfg1=run_workload("cfg1", 4024, 3036, synth.load_fixture("Dst7"), 3, a.reps),
               cfg4=run_workload("cfg4", 2048, 2048, synth.synth_template(128), 4, a.reps))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out)[:2000])


if __name__ == "__main__":
    main()
