"""Masked templates (fpm_learn_masked) against the same template unmasked, on the cfg1 and cfg4 workloads of bench.py:
  batch      device-resident batch of 64 frames, images/s (host clock around calls that end in a device synchronise)
  latency    one frame, fpm_match p50 ms
  kernels    per-kernel device time of one profiled batch (FPM_PARAM_PROFILE): fpm_mask_window_kernel (refinement window sums),
             fpm_top_score_kernel(masked) against fpm_top_score_kernel, and the correlation kernels
  evals      the refinement evals of frame 0 per layer (FPM_PARAM_TRACE): a mask changes which candidates pass each layer
The mask is the disc inscribed in the template.  The two arms alternate in one process after warm-up; the found counts are
recorded.  Writes one JSON file (default profiles/masked_b200.json) with the card name and power limit.
    python scripts/bench_masked.py [--out PATH] [--reps 10]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import bench  # noqa: E402
from fastest_image_pattern_matching_b200 import TemplateMatcher  # noqa: E402
from tests.masked_oracle import disc_mask  # noqa: E402

KERNELS = ("fpm_mask_window_kernel", "fpm_top_score_kernel", "fpm_top_score_kernel(masked)", "fpm_corr_rows_kernel",
           "fpm_corr_mma_kernel", "fpm_corr_fused_kernel", "fpm_refine_finalize_kernel", "fpm_warp_kernel(roi)")


def card():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                               timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                                   # noqa: BLE001
        power = "unknown (%s)" % e
    return name, power


def run_workload(workload, reps):
    wl = bench.WORKLOADS[workload]
    B = 64
    tpl, frames = bench.make_frames(B, 100, workload)
    d = torch.from_numpy(frames).cuda()
    H, W = frames.shape[1:]
    mask = disc_mask(tpl.shape[1], tpl.shape[0])
    arms = {}
    for arm in ("unmasked", "disc"):
        m = TemplateMatcher(0)
        bench.configure(m, wl)
        assert m.learnPattern(tpl) if arm == "unmasked" else m.learnPattern(tpl, mask)
        arms[arm] = m

    def batch(m):
        res, cnt = m.matchBatchRaw(d.data_ptr(), B, W, H, W, H * W, True)
        torch.cuda.synchronize()
        return sum(min(cnt[b], m.result_capacity) for b in range(B))

    out = {"workload": workload, "frames": B, "template": list(tpl.shape[::-1]), "mask_kept": int(mask.sum())}
    found = {k: batch(m) for k, m in arms.items()}                       # warm-up
    bt = {k: [] for k in arms}
    for _ in range(reps):
        for k, m in arms.items():
            t0 = time.perf_counter()
            batch(m)
            bt[k].append(time.perf_counter() - t0)
    lt = {k: [] for k in arms}
    for k, m in arms.items():
        m.match(frames[0])
    for _ in range(reps * 3):
        for k, m in arms.items():
            t0 = time.perf_counter()
            m.match(frames[0])
            lt[k].append((time.perf_counter() - t0) * 1e3)
    evals = {}
    for k, m in arms.items():                                            # refinement evals of frame 0 per layer (traced)
        m.setTrace(True)
        m.match(frames[0])
        evals[k] = [int(len(m.traceEvals(l))) for l in range(len(m.templateLevels()) - 1)]
        m.setTrace(False)
    for k, m in arms.items():
        m.setProfile(True)
        m.profileReset()
        batch(m)
        prof = m.profile()
        m.setProfile(False)
        out[k] = dict(found_in_batch=int(found[k]), frame0_refine_evals_per_layer=evals[k],
                      batch_images_per_s=B / float(np.median(bt[k])),
                      batch_images_per_s_all=[round(B / t, 1) for t in bt[k]],
                      single_frame_p50_ms=float(np.median(lt[k])),
                      kernels_ms={n: round(prof[n][0], 4) for n in KERNELS if n in prof and prof[n][1] > 0},
                      kernel_launches={n: int(prof[n][1]) for n in KERNELS if n in prof and prof[n][1] > 0})
        m.close()
    out["masked_over_unmasked_throughput"] = out["disc"]["batch_images_per_s"] / out["unmasked"]["batch_images_per_s"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "masked_b200.json"))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--workloads", default="cfg1,cfg4")
    a = ap.parse_args()
    name, power = card()
    res = dict(gpu=name, power_limit=power, results=[run_workload(w, a.reps) for w in a.workloads.split(",")])
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
