"""Scale-tolerant template sets on the 36-glyph M12 set: 64 M12-like frames (scripts/bench_template_set.py m12_frames: shifted,
noised), each resized about its centre by a seeded scale drawn from [0.9, 1.1], device-resident and pinned-host.  Arms,
alternating in one process after warm-up:
  set_1        fpm_match_set_batch at [1, 1]
  scaled_1     fpm_match_set_scaled at [1, 1]
  scaled_r     fpm_match_set_scaled at [0.9, 1.1]
  merged_1     fpm_match_set_scaled_merged at [1, 1], Score 0.7, overlap 0.3
  merged_r     fpm_match_set_scaled_merged at [0.9, 1.1], Score 0.7, overlap 0.3
  multi_r      a loop of fpm_match_multi (36 single-glyph handles) over the frames at [0.9, 1.1] (host frames only)
Each (Score, range) has its own set handle, so no timed call changes a handle's range, and every arm writes into result
buffers allocated once outside the timed calls.  Per arm: images/s (host clock around calls that end in a device synchronise,
median of --reps), launches per batch, per-kernel ms of one profiled batch (FPM_PARAM_PROFILE) and their sum, and the frames
whose read (fpm_ocr_assemble of the merged list, or of all per-glyph lists for the unmerged arms) equals the known text.  The plain arms use the M12 case's parameters (Score 0.85).
Writes one JSON file (default profiles/scaled_set_b200.json) with the card name and power limit.
    python scripts/bench_scaled_set.py [--out PATH] [--reps 5]"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import cv2  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402
import fpm_workloads as synth  # noqa: E402
from oracle import oracle as O  # noqa: E402
from bench_template_set import card, m12_frames  # noqa: E402
from fastest_image_pattern_matching_b200 import TemplateMatcher  # noqa: E402
from fastest_image_pattern_matching_b200 import _lib as L  # noqa: E402
from fastest_image_pattern_matching_b200.matcher import _convert, ocr_assemble  # noqa: E402
from tests.helpers import configure  # noqa: E402
from tests.test_ocr import KNOWN_TEXT  # noqa: E402

RANGE = (0.9, 1.1)
B = 64


def resized_frames(src, seed):
    """m12_frames, each frame resized about its centre by a seeded scale in [0.9, 1.1] (edge pixels replicated)"""
    rng = np.random.default_rng(seed)
    frames = m12_frames(src, B, seed)
    H, W = src.shape
    scales = [float(s) for s in rng.uniform(0.9, 1.1, size=B)]
    out = [cv2.warpAffine(f, cv2.getRotationMatrix2D(((W - 1) / 2.0, (H - 1) / 2.0), 0.0, s), (W, H), flags=cv2.INTER_LINEAR,
                          borderMode=cv2.BORDER_REPLICATE) for f, s in zip(frames, scales)]
    return np.stack(out), scales


def text_of(per_glyph):
    centres, labels = [], []
    for ch, lst in zip(O.OCR_LETTERS, per_glyph):
        for r in lst:
            centres.append(r.ptCenter)
            labels.append(ch)
    return ocr_assemble(centres, labels)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "scaled_set_b200.json"))
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    name, power = card()
    with open(os.path.join(ROOT, "tests", "golden", "cases.json")) as f:
        case = json.load(f)["ocr_m12"]
    glyphs = [synth.load_fixture("M12/" + ch) for ch in O.OCR_LETTERS]
    src = synth.load_fixture(case["src"])
    H, W = src.shape
    frames, scales = resized_frames(src, 7)
    dev = torch.from_numpy(frames).cuda()
    pinned = torch.from_numpy(frames).pin_memory()
    srcs = {"device": (dev.data_ptr(), True), "pinned": (pinned.data_ptr(), False)}
    T, cap = len(glyphs), 256

    def set_handle(params, rng):
        m = configure(TemplateMatcher(0, result_capacity=cap), params)
        m.setScaleRange(*rng)
        m.learnPatternSet(glyphs)
        return m
    # one handle per (Score, range): no timed call changes a handle's range (that would re-plan every group)
    plain_1, plain_r = set_handle(case["params"], (1.0, 1.0)), set_handle(case["params"], RANGE)
    merged_1, merged_r = set_handle(dict(case["params"], score=0.7), (1.0, 1.0)), set_handle(dict(case["params"], score=0.7), RANGE)
    singles = []
    for g in glyphs:
        m = configure(TemplateMatcher(0, result_capacity=cap), case["params"])
        m.setScaleRange(*RANGE)
        m.learnPattern(g)
        singles.append(m)

    # every arm writes into buffers allocated once, outside the timed calls
    def set_arm(m, scaled, ptr, on_dev):
        res, counts, sc = (L.fpm_result * (cap * B * T))(), (C.c_int * (B * T))(), (C.c_double * (cap * B * T))()

        def run():
            if scaled:
                rc = m._lib.fpm_match_set_scaled(m._h, ptr, int(on_dev), B, W, H, W, H * W, res, sc, cap, counts)
            else:
                rc = m._lib.fpm_match_set_batch(m._h, ptr, int(on_dev), B, W, H, W, H * W, res, cap, counts)
            m._check(rc)
            torch.cuda.synchronize()
        return [m], run, lambda: m._set_results(res, counts, B, T)

    def merged_arm(m, ptr, on_dev):
        res, labels, counts = (L.fpm_result * (cap * B))(), (C.c_int * (cap * B))(), (C.c_int * B)()
        setc, sc = (C.c_int * (B * T))(), (C.c_double * (cap * B))()

        def run():
            m._check(m._lib.fpm_match_set_scaled_merged(m._h, ptr, int(on_dev), B, W, H, W, H * W, 0.3, res, sc, labels, cap,
                                                        counts, setc))
            torch.cuda.synchronize()

        def per_glyph():
            out = []
            for lst in m._merged_results(res, labels, counts, B):
                per = [[] for _ in range(T)]
                for t, r in lst:
                    per[t].append(r)
                out.append(per)
            return out
        return [m], run, per_glyph

    def multi_arm():
        lib = singles[0]._lib
        hs = (C.c_void_p * T)(*[m._h for m in singles])
        res, counts = (L.fpm_result * (cap * T))(), (C.c_int * T)()

        def one(f):
            rc = lib.fpm_match_multi(hs, T, f.ctypes.data, W, H, W, res, cap, counts)
            if rc != 0:
                raise RuntimeError("fpm_match_multi error %d" % rc)

        def run():
            for f in frames:
                one(f)
            torch.cuda.synchronize()

        def per_glyph():                                     # an untimed pass that keeps every frame's lists
            out = []
            for f in frames:
                one(f)
                out.append([_convert(res[t * cap:(t + 1) * cap], min(counts[t], cap)) for t in range(T)])
            return out
        return singles, run, per_glyph

    arms = {}
    for where, (ptr, on_dev) in srcs.items():
        arms[where + "/set_1"] = set_arm(plain_1, False, ptr, on_dev)
        arms[where + "/scaled_1"] = set_arm(plain_1, True, ptr, on_dev)
        arms[where + "/scaled_r"] = set_arm(plain_r, True, ptr, on_dev)
        arms[where + "/merged_1"] = merged_arm(merged_1, ptr, on_dev)
        arms[where + "/merged_r"] = merged_arm(merged_r, ptr, on_dev)
    arms["host/multi_r"] = multi_arm()
    res = {}
    for k, (handles, run, per_glyph) in arms.items():         # warm-up, launches, reads
        l0 = sum(h.launchCount() for h in handles)
        run()
        launches = sum(h.launchCount() for h in handles) - l0
        reads = [text_of(p) == KNOWN_TEXT for p in per_glyph()]
        res[k] = dict(launches_per_batch=launches, frames_reading_known_text=int(sum(reads)), times=[])
    for _ in range(a.reps):
        for k, (_, run, _) in arms.items():
            t0 = time.perf_counter()
            run()
            res[k]["times"].append(time.perf_counter() - t0)
    for k, (handles, run, _) in arms.items():
        for h in handles:
            h.setProfile(True)
            h.profileReset()
        run()
        prof = {}
        for h in handles:
            for kk, (ms, n, _) in h.profile().items():
                if n > 0:
                    prof[kk] = round(prof.get(kk, 0.0) + ms, 3)
            h.setProfile(False)
        res[k]["kernels_ms"] = prof
        res[k]["kernels_ms_total"] = round(sum(prof.values()), 3)
        t = sorted(res[k].pop("times"))
        res[k]["images_per_s"] = round(B / t[len(t) // 2], 1)
        res[k]["images_per_s_all"] = [round(B / x, 1) for x in t]
    for m in singles + [plain_1, plain_r, merged_1, merged_r]:
        m.close()
    out = dict(gpu=name, power_limit=power, batch=B, frame=[W, H], glyphs=T, range=list(RANGE),
               frame_scales=[round(s, 4) for s in scales], merge=dict(score=0.7, overlap=0.3), arms=res)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: (v["images_per_s"], v["launches_per_batch"], v["frames_reading_known_text"]) for k, v in res.items()}))


if __name__ == "__main__":
    main()
