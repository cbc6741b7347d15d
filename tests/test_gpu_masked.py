"""Masked templates on the GPU (fpm_learn_masked) against the masked CPU oracle (tests/masked_oracle.py).

- A full mask gives results bit-identical to fpm_learn on every golden case, every correlation path and the batch paths.
- Disc, ring, holed, blob and corner-cut masks: results at the project tolerances, all 49 refinement scores of every eval and
  the top-layer map above reject_below bit for bit, the mask pyramid and level statistics exactly.
- A disc-shaped part pasted at random angles on a background unlike the template's corners is found by the masked matcher.
- Batch, ingested-batch and angle-sharded results equal per-frame fpm_match; sub-pixel and MFC-compat runs match the oracle.
- Refusals, unmasked re-learns and MinReduceArea re-learns.
"""
import cv2
import numpy as np
import pytest

import fpm_workloads as synth
from fastest_image_pattern_matching_b200 import _lib as L
from tests.helpers import assert_results_match, configure, get_image
from tests.masked_oracle import MASKS, MaskedOracleMatcher, disc_mask

pytestmark = pytest.mark.gpu

GOLDEN = ["src8", "src9", "test4_src3", "src4", "src9_subpix", "cfg3_src6"]
MASKED_CASES = ["src8", "src9", "test4_src3", "src4"]


def _key(r):
    return (r.dMatchScore, r.dMatchedAngle, r.ptCenter, r.ptLT, r.ptRT, r.ptRB, r.ptLB)


def _case(golden_cases, name):
    c = golden_cases[name]
    return get_image(c["tpl"]), get_image(c["src"]), c["params"]


def _learn(m, tpl, mask):
    return m.learnPattern(tpl) if mask is None else m.learnPattern(tpl, mask)


# ---------------- 1. a full mask is fpm_learn, bit for bit ----------------
@pytest.mark.parametrize("name", GOLDEN)
def test_full_mask_bit_identical(matcher, golden_cases, name):
    tpl, src, params = _case(golden_cases, name)
    configure(matcher, params)
    full = np.ones(tpl.shape, np.uint8)
    try:
        for mode in (0, 1, 2, 3, 4):
            matcher.setTensorCores(mode)
            runs = []
            for mask in (None, full):
                assert _learn(matcher, tpl, mask)
                one = matcher.match(src)
                batch = matcher.matchBatch(np.stack([src, src]))
                runs.append(([_key(r) for r in one], [[_key(r) for r in b] for b in batch]))
            assert runs[0][0], (name, mode)
            assert runs[0] == runs[1], (name, mode)
            assert runs[0][1] == [runs[0][0], runs[0][0]]
        import torch
        d = torch.from_numpy(np.stack([src] * 3)).cuda()
        outs = []
        for mask in (None, full):
            assert _learn(matcher, tpl, mask)
            res, cnt = matcher.matchBatchRaw(d.data_ptr(), 3, src.shape[1], src.shape[0], src.shape[1], src.size, True)
            outs.append([tuple(tuple(getattr(res[b * matcher.result_capacity + i], f) for f, _ in L.fpm_result._fields_)
                               for i in range(min(cnt[b], matcher.result_capacity))) for b in range(3)])
        assert outs[0] == outs[1] and outs[0][0]
    finally:
        matcher.setTensorCores(1)


# ---------------- 2. masks against the masked oracle ----------------
_oracles = {}


def _oracle(golden_cases, name, mask_name, **extra):
    key = (name, mask_name, tuple(sorted(extra.items())))
    if key not in _oracles:
        tpl, src, params = _case(golden_cases, name)
        m = MASKS[mask_name](tpl.shape[1], tpl.shape[0])
        om = configure(MaskedOracleMatcher(), dict(params, **extra))
        om.trace = {}
        assert om.learn_pattern(tpl, m)
        res = om.match(src)
        _oracles[key] = (om, res, m)
    return _oracles[key]


def _gpu_evals(matcher, levels):
    evals = {}
    for layer in range(levels - 1):
        rows, scores = matcher.traceEvals(layer), matcher.traceEvalScores(layer)
        seen = {}
        for i, r in enumerate(rows):
            cid = int(r[0])
            j = seen.get(cid, 0)
            seen[cid] = j + 1
            evals[(layer, cid, j)] = scores[i]
    return evals


@pytest.mark.parametrize("mask_name", sorted(MASKS))
@pytest.mark.parametrize("name", MASKED_CASES)
@pytest.mark.parametrize("mode", (0, 1, 6))
def test_masked_matches_oracle(matcher, golden_cases, oracle_lib, name, mask_name, mode):
    om, want, m = _oracle(golden_cases, name, mask_name)
    tpl, src, params = _case(golden_cases, name)
    configure(matcher, params)
    matcher.setTensorCores(mode)
    try:
        assert matcher.learnPattern(tpl, m)
        assert_results_match(matcher.match(src), want, ordered=False)
        matcher.setTrace(True)
        matcher.match(src)
        levels = matcher.templateLevels()
        got = _gpu_evals(matcher, len(levels))
    finally:
        matcher.setTrace(False)
        matcher.setTensorCores(1)
    ref = {(e["layer"], e["cand"], e["j"]): np.asarray(e["score"], np.float32) for e in om.trace["refine"]}
    assert set(ref) == set(got), (name, mask_name, sorted(set(ref) ^ set(got))[:6])
    bad = [k for k in ref if not np.array_equal(ref[k].view(np.uint32), np.asarray(got[k], np.float32).reshape(7, 7).view(np.uint32))]
    assert not bad, "%d of %d evals differ, first %s" % (len(bad), len(ref), bad[:4])
    # level masks and statistics, exactly
    for l, lv in enumerate(levels):
        assert np.array_equal(lv["mask"], om.masks[l]) and lv["n_kept"] == int(om.masks[l].sum())
        assert (lv["mean"], lv["norm"], lv["inv_area"], lv["result_equal1"]) == (
            om.td.templ_mean[l], om.td.templ_norm[l], om.td.inv_area[l], om.td.result_equal1[l])
        assert np.array_equal(lv["pixels"], om.td.pyramid[l])
    assert matcher.borderColor() == om.td.border_color


@pytest.mark.parametrize("mask_name", sorted(MASKS))
@pytest.mark.parametrize("name", MASKED_CASES)
def test_masked_top_score_production(matcher, golden_cases, name, mask_name):
    om, _, m = _oracle(golden_cases, name, mask_name)
    tpl, src, params = _case(golden_cases, name)
    configure(matcher, params)
    assert matcher.learnPattern(tpl, m)
    for rec in om.trace["top"][:4]:
        rot = rec["rot"]
        got, reject_below = matcher.dbgTopScoreProduction(rot)
        top = len(om.td.pyramid) - 1
        want = om._match_template(rot, top, False, top=True)
        keep = want >= reject_below
        assert np.array_equal(got[keep].view(np.uint32), want[keep].view(np.uint32)), (name, mask_name)
        assert np.all(got[~keep] < reject_below)
        assert np.array_equal(matcher.dbgTopScore(rot).view(np.uint32), want.view(np.uint32))


# ---------------- 4. capability: a disc-shaped part on a foreign background ----------------
def test_disc_part_found_at_every_angle(matcher, oracle_lib, capsys):
    rng = np.random.default_rng(2024)
    D = 96
    part = synth.background(D, D, 5, 1.2)
    disc = disc_mask(D, D)
    tpl = np.where(disc > 0, part, synth.background(D, D, 9, 1.2)).astype(np.uint8)   # the template's corners: another surface
    src = synth.background(900, 700, 6, 3.0)                    # a background unlike those corners
    K = 6
    truth = []
    for k in range(K):
        ang = float(rng.uniform(-180, 180))
        R = cv2.getRotationMatrix2D(((D - 1) / 2, (D - 1) / 2), ang, 1)
        rp = cv2.warpAffine(part, R, (D, D), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_REFLECT)
        x, y = 40 + (k % 3) * 280, 60 + (k // 3) * 330
        region = src[y:y + D, x:x + D]
        region[disc > 0] = rp[disc > 0]
        truth.append((x + (D - 1) / 2, y + (D - 1) / 2))
    params = dict(max_pos=K + 2, score=0.8, tolerance_angle=180, min_reduce_area=256)
    configure(matcher, params)
    assert matcher.learnPattern(tpl)
    plain = matcher.match(src)
    assert matcher.learnPattern(tpl, disc)
    got = matcher.match(src)
    om = configure(MaskedOracleMatcher(), params)
    assert om.learn_pattern(tpl, disc)
    assert_results_match(got, om.match(src), ordered=False)
    found = [min(np.hypot(r.ptCenter[0] - cx, r.ptCenter[1] - cy) for r in got) for cx, cy in truth]
    assert len(got) == K and max(found) < 1.5, found
    configure(matcher, dict(params, score=0.3))
    assert matcher.learnPattern(tpl)
    best = sorted(r.dMatchScore for r in matcher.match(src))[::-1][:K]
    with capsys.disabled():
        print("\n[masked capability] masked scores %s; unmasked matcher at Score 0.8 found %d, best unmasked scores %s" % (
            [round(r.dMatchScore, 3) for r in got], len(plain), [round(s, 3) for s in best]))


# ---------------- 5. every entry point gives per-frame fpm_match ----------------
def test_masked_batch_ingest_sharded_equal_single(matcher, golden_cases):
    from fastest_image_pattern_matching_b200 import TemplateMatcher
    from fastest_image_pattern_matching_b200.matcher import match_sharded_virtual
    tpl, src, params = _case(golden_cases, "src9")
    m = MASKS["ring"](tpl.shape[1], tpl.shape[0])
    frames = [src, np.ascontiguousarray(src[:, ::-1]), np.ascontiguousarray(src[::-1])]
    configure(matcher, params)
    assert matcher.learnPattern(tpl, m)
    single = [[_key(r) for r in matcher.match(f)] for f in frames]
    assert all(single)
    assert [[_key(r) for r in b] for b in matcher.matchBatch(np.stack(frames))] == single
    for split in (0, 2):
        matcher.setSplitBatch(split)
        assert [[_key(r) for r in b] for b in matcher.matchBatch(np.stack(frames * 3))] == single * 3
    matcher.setSplitBatch(8)
    files = [cv2.imencode(".jpg", f)[1].tobytes() for f in frames]
    matcher.ingestJpegBatch(files)
    decoded = [matcher.ingestedFramePixels(i) for i in range(3)]
    want = [[_key(r) for r in matcher.match(f)] for f in decoded]
    assert [[_key(r) for r in b] for b in matcher.matchIngestedBatch()] == want
    others = [TemplateMatcher(0) for _ in range(2)]
    try:
        for o in others:
            configure(o, params)
            assert o.learnPattern(tpl, m)
        for lists in match_sharded_virtual([matcher] + others, src):
            assert [_key(r) for r in lists] == single[0]
    finally:
        for o in others:
            o.close()


@pytest.mark.parametrize("variant", ["subpix", "mfc", "stop1", "bitnot", "range"])
def test_masked_modes_match_oracle(matcher, golden_cases, oracle_lib, variant):
    tpl, src, params = _case(golden_cases, "src9")
    m = MASKS["corner_cut"](tpl.shape[1], tpl.shape[0])
    extra = {"subpix": dict(sub_pixel=True), "mfc": dict(mfc_compat=True), "stop1": dict(stop_layer1=True),
             "bitnot": dict(bitwise_not=True), "range": dict(tolerance_range=(-60.0, 30.0, 100.0, 170.0))}[variant]
    om = configure(MaskedOracleMatcher(), dict(params, **extra))
    assert om.learn_pattern(tpl, m)
    want = om.match(src)
    configure(matcher, dict(params, sub_pixel=variant == "subpix"))
    try:
        matcher.setMfcCompat(variant == "mfc")
        matcher.setStopLayer1(variant == "stop1")
        matcher.setBitwiseNot(variant == "bitnot")
        matcher.setToleranceRange(extra["tolerance_range"] if variant == "range" else None)
        assert matcher.learnPattern(tpl, m)
        assert_results_match(matcher.match(src), want, ordered=False)
    finally:
        matcher.setMfcCompat(False)
        matcher.setStopLayer1(False)
        matcher.setBitwiseNot(False)
        matcher.setToleranceRange(None)


# ---------------- 6. refusals and re-learns ----------------
def test_masked_refusals_and_relearn(matcher, golden_cases):
    from fastest_image_pattern_matching_b200.matcher import FpmError
    tpl, src, params = _case(golden_cases, "src9")
    configure(matcher, params)
    h, w = tpl.shape
    rc = matcher._lib.fpm_learn_masked(matcher._h, tpl.ctypes.data, w, h, w, None, w)
    assert rc == -1 and b"null mask" in matcher._lib.fpm_last_error(matcher._h)
    with pytest.raises(FpmError, match="keeps no pixel"):
        matcher.learnPattern(tpl, np.zeros_like(tpl))
    assert not matcher.isPatternLearned()
    dot = np.zeros_like(tpl)
    dot[0, 0] = 1
    with pytest.raises(FpmError, match="level 1"):
        matcher.learnPattern(tpl, dot)
    assert not matcher.isPatternLearned()
    # a masked learn, then fpm_learn: unmasked again
    m = MASKS["disc"](w, h)
    assert matcher.learnPattern(tpl, m)
    assert matcher.templateLevels()[0]["n_kept"] == int(m.sum())
    assert matcher.learnPattern(tpl)
    assert all(lv["n_kept"] == lv["w"] * lv["h"] and lv["mask"].all() for lv in matcher.templateLevels())
    plain = [_key(r) for r in matcher.match(src)]
    configure(matcher, params)
    assert [_key(r) for r in matcher.match(src)] == plain
    # a MinReduceArea change re-learns with the mask
    assert matcher.learnPattern(tpl, m)
    matcher.setMinReduceArea(64)
    got = matcher.match(src)
    om = configure(MaskedOracleMatcher(), dict(params, min_reduce_area=64))
    assert om.learn_pattern(tpl, m)
    assert_results_match(got, om.match(src), ordered=False)
    lv = matcher.templateLevels()
    assert len(lv) == len(om.td.pyramid) and all(np.array_equal(a["mask"], b) for a, b in zip(lv, om.masks))
    matcher.setMinReduceArea(256)
