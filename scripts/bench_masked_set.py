"""Masked template sets (fpm_learn_set_masked) against masked single handles, in one process, alternating the two arms of
each comparison:
  m12_read     one M12 read, every glyph under its stroke mask (its ink dilated by 2 pixels): fpm_match_set_batch of one
               frame vs 36 masked handles through fpm_match_multi (p50, launches)
  m12_frames   64 seeded M12-like frames (shifted, noised), device-resident and host-pinned: the masked set per template
               (fpm_match_set_batch) and merged (fpm_match_set_batch_merged, NMS across the glyphs at overlap 0.3), images/s
  parts128     6 masked parts of 128x128 at +-180 deg on 64 frames of 2048x1536 (device-resident): one masked set call
               (dp4a refinement) vs one masked handle per template (tensor cores where they apply)
Every timing is a host clock around calls that end in a device synchronise, after warm-up.  Results of the two arms are
checked equal.  Per-kernel times come from separate FPM_PARAM_PROFILE calls.  Writes one JSON file (default
profiles/masked_set_b200.json) with the card name and power limit.
    python scripts/bench_masked_set.py [--out PATH] [--reps 20]"""
import argparse
import json
import os
import sys

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
import cv2  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402
import fpm_workloads as synth  # noqa: E402
from oracle import oracle as O  # noqa: E402
from fastest_image_pattern_matching_b200 import TemplateMatcher, match_multi  # noqa: E402
from scripts.bench_template_set import alternate, card, m12_frames, rows  # noqa: E402
from tests.helpers import configure  # noqa: E402
from tests.masked_oracle import MASKS, EDGE_MASKS  # noqa: E402


def stroke_mask(g):
    thr, _ = cv2.threshold(g, 0, 255, cv2.THRESH_BINARY + cv2.THRESH_OTSU)
    return cv2.dilate((g < thr).astype(np.uint8), np.ones((5, 5), np.uint8))


def profile_ms(m, call):
    m.setProfile(True); m.profileReset()
    call()
    p = {k: round(v[0], 3) for k, v in m.profile().items() if v[0] > 0}
    m.setProfile(False)
    return p


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "masked_set_b200.json"))
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    name, power = card()
    with open(os.path.join(ROOT, "tests", "golden", "cases.json")) as f:
        case = json.load(f)["ocr_m12"]
    glyphs = [synth.load_fixture("M12/" + ch) for ch in O.OCR_LETTERS]
    masks = [stroke_mask(g) for g in glyphs]
    src = synth.load_fixture(case["src"])
    H, W = src.shape
    singles = []
    for g, mk in zip(glyphs, masks):
        m = configure(TemplateMatcher(0, result_capacity=256), case["params"])
        m.learnPattern(g, mk)
        singles.append(m)
    sm = configure(TemplateMatcher(0, result_capacity=256), case["params"])
    sm.learnPatternSet(glyphs, masks)
    out = {"card": name, "power_limit": power, "reps": a.reps, "stroke_mask": "Otsu ink dilated by a 5x5 square"}

    # ---- one M12 read
    assert [rows(x) for x in sm.matchSet(src)] == [rows(x) for x in match_multi(singles, src)]
    l0 = sm.launchCount(); sm.matchSet(src); set_launches = sm.launchCount() - l0
    l0 = sum(m.launchCount() for m in singles); match_multi(singles, src); multi_launches = sum(m.launchCount() for m in singles) - l0
    ms = alternate({"set": lambda: sm.matchSet(src), "multi": lambda: match_multi(singles, src)}, 3 * a.reps)
    out["m12_read"] = {"set_p50_ms": round(float(np.median(ms["set"])), 3), "multi_p50_ms": round(float(np.median(ms["multi"])), 3),
                       "set_launches": set_launches, "multi_launches": multi_launches,
                       "hits": int(sum(len(x) for x in sm.matchSet(src)))}
    out["m12_read"]["set_profile_ms"] = profile_ms(sm, lambda: sm.matchSet(src))

    # ---- 64 M12-like frames, per template and merged
    B = 64
    frames = m12_frames(src, B, 5)
    pinned = torch.from_numpy(frames).pin_memory()
    dev = pinned.cuda()
    got = sm.matchSetBatch(frames)
    for b in (0, B - 1):
        assert [rows(x) for x in got[b]] == [rows(x) for x in match_multi(singles, frames[b])]
    rs = sm.matchSetBatchRaw(dev.data_ptr(), B, W, H, W, H * W, True)
    rm = sm.matchSetBatchMergedRaw(dev.data_ptr(), B, W, H, W, H * W, True, 0.3)
    arms = {"set_device": lambda: sm.matchSetBatchRaw(dev.data_ptr(), B, W, H, W, H * W, True, *rs),
            "merged_device": lambda: sm.matchSetBatchMergedRaw(dev.data_ptr(), B, W, H, W, H * W, True, 0.3, *rm),
            "set_pinned": lambda: sm.matchSetBatchRaw(pinned.data_ptr(), B, W, H, W, H * W, False, *rs),
            "merged_pinned": lambda: sm.matchSetBatchMergedRaw(pinned.data_ptr(), B, W, H, W, H * W, False, 0.3, *rm)}
    ms = alternate(arms, a.reps)
    out["m12_frames"] = {k + "_images_per_s": round(B / (float(np.median(v)) / 1e3), 1) for k, v in ms.items()}
    out["m12_frames"].update(batch=B, merge_overlap=0.3, per_template_hits=int(sum(rs[1])), merged_hits=int(sum(rm[2])))
    out["m12_frames"]["set_device_profile_ms"] = profile_ms(sm, lambda: sm.matchSetBatchRaw(dev.data_ptr(), B, W, H, W, H * W, True, *rs))
    sm.close()
    for m in singles:
        m.close()

    # ---- 6 masked parts of 128x128 at +-180 deg on 64 frames of 2048x1536
    names = ["disc", "ring", "corner_cut", "holed", "blob", "comb"]
    pmasks = [dict(MASKS, **EDGE_MASKS)[k](128, 128) for k in names]
    tpls = [synth.synth_template(128, 40 + k) for k in range(len(names))]
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
    for t, mk in zip(tpls, pmasks):
        m = configure(TemplateMatcher(0, result_capacity=64), params)
        m.learnPattern(t, mk)
        hs.append(m)
    s6 = configure(TemplateMatcher(0, result_capacity=64), params)
    s6.learnPatternSet(tpls, pmasks)
    n, (Hh, Ww) = len(fr), fr.shape[1:]
    rs = s6.matchSetBatchRaw(d.data_ptr(), n, Ww, Hh, Ww, Hh * Ww, True)
    ri = [m.matchBatchRaw(d.data_ptr(), n, Ww, Hh, Ww, Hh * Ww, True) for m in hs]
    for t in range(len(tpls)):
        for b in range(n):
            k = b * len(tpls) + t
            assert rs[1][k] == ri[t][1][b]
            for i in range(min(rs[1][k], 64)):
                assert bytes(rs[0][k * 64 + i]) == bytes(ri[t][0][b * 64 + i])
    arms = {"set": lambda: s6.matchSetBatchRaw(d.data_ptr(), n, Ww, Hh, Ww, Hh * Ww, True, *rs),
            "per_template": lambda: [m.matchBatchRaw(d.data_ptr(), n, Ww, Hh, Ww, Hh * Ww, True, *r) for m, r in zip(hs, ri)]}
    ms = alternate(arms, max(3, a.reps // 4))
    out["parts128"] = {k + "_images_per_s": round(n / (float(np.median(v)) / 1e3), 1) for k, v in ms.items()}
    out["parts128"].update(frames=n, masks=names, hits=int(sum(rs[1])))
    out["parts128"]["set_profile_ms"] = profile_ms(s6, lambda: s6.matchSetBatchRaw(d.data_ptr(), n, Ww, Hh, Ww, Hh * Ww, True, *rs))
    out["parts128"]["one_template_profile_ms"] = profile_ms(hs[0], lambda: hs[0].matchBatchRaw(d.data_ptr(), n, Ww, Hh, Ww, Hh * Ww, True, *ri[0]))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
