"""Template sets against today's multi-template paths, in one process, alternating the two arms of each comparison:
  m12_read     one M12 read (36 glyphs on M12_D_Test): fpm_match_set_batch of one frame vs fpm_match_multi (p50, launches)
  m12_frames   64 seeded M12-like frames (shifted, noised), host-pinned and device-resident: one set call vs a loop of
               fpm_match_multi over the frames (images/s)
  m12_merged   the same 64 frames at Score 0.7, device-resident and pinned: fpm_match_set_batch_merged (NMS across the glyphs
               at overlap 0.3) vs fpm_match_set_batch (images/s), and the fpm_set_merge_kernel time of one profiled call
  rot128       8 templates of 128x128 at +-180 deg on 64 frames of 2048x1536 (device-resident): one set call (dp4a refinement)
               vs one handle per template (tensor cores where they apply)
Every timing is a host clock around calls that end in a device synchronise, after warm-up.  Results of the two arms are
checked equal; the merged lists of the first and last frame are checked against the host reference of the merge
(tests/test_gpu_set_merge.py).  Writes one JSON file (default profiles/template_set_b200.json) with the card name and power limit.
    python scripts/bench_template_set.py [--out PATH] [--reps 20]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
import cv2  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402
import fpm_workloads as synth  # noqa: E402
from oracle import oracle as O  # noqa: E402
from fastest_image_pattern_matching_b200 import TemplateMatcher, match_multi  # noqa: E402
from tests.helpers import configure  # noqa: E402
from tests.test_gpu_set_merge import merge_reference  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                               timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                                   # noqa: BLE001
        power = "unknown (%s)" % e
    return name, power


def alternate(arms, reps):
    """{name: fn} run in turn reps times after one warm-up each; per-call ms lists"""
    for fn in arms.values():
        fn()
    ms = {k: [] for k in arms}
    for _ in range(reps):
        for k, fn in arms.items():
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ms[k].append((time.perf_counter() - t0) * 1e3)
    return ms


def rows(lst):
    return [(r.dMatchScore, r.dMatchedAngle) + tuple(r.ptCenter) for r in lst]


def m12_frames(src, n, seed):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        dx, dy = (int(v) for v in rng.integers(-6, 7, size=2))
        f = np.roll(np.roll(src, dy, axis=0), dx, axis=1).astype(np.int16) + rng.integers(-4, 5, size=src.shape).astype(np.int16)
        out.append(np.clip(f, 0, 255).astype(np.uint8))
    return np.stack(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "template_set_b200.json"))
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    name, power = card()
    with open(os.path.join(ROOT, "tests", "golden", "cases.json")) as f:
        case = json.load(f)["ocr_m12"]
    glyphs = [synth.load_fixture("M12/" + ch) for ch in O.OCR_LETTERS]
    src = synth.load_fixture(case["src"])
    H, W = src.shape
    singles = []
    for g in glyphs:
        m = configure(TemplateMatcher(0, result_capacity=256), case["params"])
        m.learnPattern(g)
        singles.append(m)
    sm = configure(TemplateMatcher(0, result_capacity=256), case["params"])
    sm.learnPatternSet(glyphs)
    out = {"card": name, "power_limit": power, "reps": a.reps}

    # ---- one M12 read
    assert [rows(x) for x in sm.matchSet(src)] == [rows(x) for x in match_multi(singles, src)]
    l0 = sm.launchCount(); sm.matchSet(src); set_launches = sm.launchCount() - l0
    l0 = sum(m.launchCount() for m in singles); match_multi(singles, src); multi_launches = sum(m.launchCount() for m in singles) - l0
    ms = alternate({"set": lambda: sm.matchSet(src), "multi": lambda: match_multi(singles, src)}, 3 * a.reps)
    out["m12_read"] = {"set_p50_ms": round(float(np.median(ms["set"])), 3), "multi_p50_ms": round(float(np.median(ms["multi"])), 3),
                       "set_launches": set_launches, "multi_launches": multi_launches}

    # ---- 64 M12-like frames
    B = 64
    frames = m12_frames(src, B, 5)
    pinned = torch.from_numpy(frames).pin_memory()
    dev = pinned.cuda()
    got = sm.matchSetBatch(frames)
    for b in (0, B - 1):
        assert [rows(x) for x in got[b]] == [rows(x) for x in match_multi(singles, frames[b])]
    res_c = sm.matchSetBatchRaw(pinned.data_ptr(), B, W, H, W, H * W, False)
    arms = {"set_pinned": lambda: sm.matchSetBatchRaw(pinned.data_ptr(), B, W, H, W, H * W, False, *res_c),
            "set_device": lambda: sm.matchSetBatchRaw(dev.data_ptr(), B, W, H, W, H * W, True, *res_c),
            "multi_loop": lambda: [match_multi(singles, frames[b]) for b in range(B)]}
    ms = alternate(arms, max(3, a.reps // 4))
    out["m12_frames"] = {k + "_images_per_s": round(B / (float(np.median(v)) / 1e3), 1) for k, v in ms.items()}
    out["m12_frames"]["batch"] = B

    # ---- merged set results: the same frames at Score 0.7, where similar glyphs hit the same character cells
    s7 = configure(TemplateMatcher(0, result_capacity=256), dict(case["params"], score=0.7))
    s7.learnPatternSet(glyphs)
    rs7 = s7.matchSetBatchRaw(dev.data_ptr(), B, W, H, W, H * W, True)
    rm7 = s7.matchSetBatchMergedRaw(dev.data_ptr(), B, W, H, W, H * W, True, 0.3)
    T, cap = len(glyphs), 256
    for b in (0, B - 1):                                     # the merged lists against the host reference of the merge
        lists = [[rs7[0][(b * T + t) * cap + i] for i in range(min(rs7[1][b * T + t], cap))] for t in range(T)]
        want = [(t, bytes(r)) for t, r in merge_reference(lists, 0.3)]
        assert rm7[2][b] == len(want)
        assert [(rm7[1][b * cap + k], bytes(rm7[0][b * cap + k])) for k in range(min(rm7[2][b], cap))] == want[:cap]
    arms = {"set_device": lambda: s7.matchSetBatchRaw(dev.data_ptr(), B, W, H, W, H * W, True, *rs7),
            "merged_device": lambda: s7.matchSetBatchMergedRaw(dev.data_ptr(), B, W, H, W, H * W, True, 0.3, *rm7),
            "set_pinned": lambda: s7.matchSetBatchRaw(pinned.data_ptr(), B, W, H, W, H * W, False, *rs7),
            "merged_pinned": lambda: s7.matchSetBatchMergedRaw(pinned.data_ptr(), B, W, H, W, H * W, False, 0.3, *rm7)}
    ms = alternate(arms, a.reps)
    out["m12_merged"] = {k + "_images_per_s": round(B / (float(np.median(v)) / 1e3), 1) for k, v in ms.items()}
    out["m12_merged"].update(batch=B, score=0.7, merge_overlap=0.3, per_template_hits=int(sum(rs7[1])), merged_hits=int(sum(rm7[2])))
    s7.setProfile(True); s7.profileReset()
    s7.matchSetBatchMergedRaw(dev.data_ptr(), B, W, H, W, H * W, True, 0.3, *rm7)
    out["m12_merged"]["merged_profile_ms"] = {k: round(v[0], 4) for k, v in s7.profile().items() if v[0] > 0}
    s7.close()
    for m in singles:
        m.close()

    # ---- 8 templates of 128x128 at +-180 deg on 64 frames of 2048x1536
    tpls = [synth.synth_template(128, 40 + k) for k in range(8)]
    rng = np.random.default_rng(9)
    fr = []
    for i in range(64):
        f = synth.background(2048, 1536, 500 + i)
        for t in tpls:
            if rng.random() < 0.5:
                synth.paste_rotated(f, t, float(rng.uniform(150, 1900)), float(rng.uniform(150, 1390)), float(rng.uniform(-180, 180)), fast=True)
        fr.append(f)
    fr = np.stack(fr)
    d = torch.from_numpy(fr).cuda()
    params = {"max_pos": 5, "score": 0.8, "tolerance_angle": 180, "max_overlap": 0.5}
    hs = []
    for t in tpls:
        m = configure(TemplateMatcher(0, result_capacity=64), params)
        m.learnPattern(t)
        hs.append(m)
    s8 = configure(TemplateMatcher(0, result_capacity=64), params)
    s8.learnPatternSet(tpls)
    n, (Hh, Ww) = len(fr), fr.shape[1:]
    rs = s8.matchSetBatchRaw(d.data_ptr(), n, Ww, Hh, Ww, Hh * Ww, True)
    ri = [m.matchBatchRaw(d.data_ptr(), n, Ww, Hh, Ww, Hh * Ww, True) for m in hs]
    for t in range(len(tpls)):
        for b in range(n):
            k = b * len(tpls) + t
            assert rs[1][k] == ri[t][1][b]
            for i in range(min(rs[1][k], 64)):
                assert bytes(rs[0][k * 64 + i]) == bytes(ri[t][0][b * 64 + i])
    arms = {"set": lambda: s8.matchSetBatchRaw(d.data_ptr(), n, Ww, Hh, Ww, Hh * Ww, True, *rs),
            "per_template": lambda: [m.matchBatchRaw(d.data_ptr(), n, Ww, Hh, Ww, Hh * Ww, True, *r) for m, r in zip(hs, ri)]}
    ms = alternate(arms, max(3, a.reps // 4))
    out["rot128"] = {k + "_images_per_s": round(n / (float(np.median(v)) / 1e3), 1) for k, v in ms.items()}
    out["rot128"]["frames"] = n
    # where the set's time goes (separate, profiled call)
    s8.setProfile(True); s8.profileReset()
    s8.matchSetBatchRaw(d.data_ptr(), n, Ww, Hh, Ww, Hh * Ww, True, *rs)
    out["rot128"]["set_profile_ms"] = {k: round(v[0], 3) for k, v in s8.profile().items() if v[0] > 0}
    hs[0].setProfile(True); hs[0].profileReset()
    hs[0].matchBatchRaw(d.data_ptr(), n, Ww, Hh, Ww, Hh * Ww, True, *ri[0])
    out["rot128"]["one_template_profile_ms"] = {k: round(v[0], 3) for k, v in hs[0].profile().items() if v[0] > 0}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
