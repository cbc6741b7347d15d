"""GPU parity tests (run on the B200 box): every CUDA stage and the whole match() against the CPU
oracle / cv2 on the same inputs, through the C ABI.

Bars (BASELINE.json north_star): bit-exact pyramid, warp, integer correlation sums and window
sums; scores within 1e-4; positions within 0.05 px; angles within 0.01 deg; identical accepted set.
"""
import math

import cv2
import numpy as np
import pytest

from oracle import oracle as O
from tests.helpers import assert_results_match, configure, get_image

pytestmark = pytest.mark.gpu


# ---------------- T0: pyramid, bit-exact ----------------
@pytest.mark.parametrize("shape", [(7, 9), (1, 1), (1, 5), (2, 2), (3, 300), (480, 640), (101, 333), (64, 47), (259, 517),
                                   (1519, 2013), (3036, 4024)])
def test_pyrdown_bit_exact(matcher, shape):
    rng = np.random.default_rng(shape[0] * 31 + shape[1])
    img = rng.integers(0, 256, shape, dtype=np.uint8)
    assert np.array_equal(matcher.dbgPyrDown(img), cv2.pyrDown(img))


def test_pyrdown_unaligned_stride(matcher):
    rng = np.random.default_rng(9)
    big = rng.integers(0, 256, (200, 301), dtype=np.uint8)
    view = big[3:150, 5:222]                       # stride 301, odd offset -> byte path
    assert np.array_equal(matcher.dbgPyrDown(view), cv2.pyrDown(np.ascontiguousarray(view)))


@pytest.mark.parametrize("shape", [(7, 9), (1, 1), (2, 2), (5, 3), (3, 300), (101, 333), (259, 517), (129, 257), (130, 258),
                                   (131, 261), (257, 1030), (1519, 2013), (3036, 4024)])
def test_pyrdown_two_levels_per_launch_bit_exact(matcher, shape):
    """fpm_pyrdown_kernel<TWO>: level 2 comes from the level-1 tile in shared memory (halo recomputed, REFLECT_101 fix-up)."""
    rng = np.random.default_rng(shape[0] * 17 + shape[1])
    img = rng.integers(0, 256, shape, dtype=np.uint8)
    want1 = cv2.pyrDown(img)
    want2 = cv2.pyrDown(want1)
    for misalign in (0, 8, 4, 3):                      # 16- / 8- / 4-byte cp.async staging, byte staging
        got1, got2 = matcher.dbgPyrDown2(img, misalign)
        assert np.array_equal(got1, want1), (shape, misalign, int((got1 != want1).sum()))
        assert np.array_equal(got2, want2), (shape, misalign, int((got2 != want2).sum()))
        assert np.array_equal(matcher.dbgPyrDown2(img, misalign, two=False), want1), (shape, misalign)


def test_pyrdown_saturated_image(matcher):
    img = np.full((300, 700), 255, np.uint8)           # largest packed 16-bit sums (16 * 4080 + 128) must not carry
    img[::3, ::5] = 0
    got1, got2 = matcher.dbgPyrDown2(img)
    assert np.array_equal(got1, cv2.pyrDown(img)) and np.array_equal(got2, cv2.pyrDown(cv2.pyrDown(img)))


def test_source_pyramid_chain(matcher, golden_cases):
    c = golden_cases["src8"]
    src = get_image(c["src"])
    lv = src
    for _ in range(4):
        nxt = matcher.dbgPyrDown(lv)
        assert np.array_equal(nxt, cv2.pyrDown(lv))
        lv = nxt


# ---------------- T2: warpAffine, bit-exact ----------------
def test_warp_affine_bit_exact(matcher):
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (190, 253), dtype=np.uint8)
    for ang in [0.0, 9.462, 90.0, -37.3, 180.0, 123.456, 270.0, 359.9]:
        for border in (0, 255):
            m = cv2.getRotationMatrix2D((126.0, 94.5), ang, 1)
            m[0, 2] += 13.5
            m[1, 2] -= 7.25
            want = cv2.warpAffine(img, m, (280, 220), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=border)
            got = matcher.dbgWarpAffine(img, m, (280, 220), border)
            assert np.array_equal(got, want), (ang, border, int((got != want).sum()))


def test_warp_affine_roi_geometry(matcher):
    """getRotatedROI-style calls (src/TemplateMatcher.cpp:1074-1090) incl. ROIs hanging over the border."""
    rng = np.random.default_rng(6)
    src = rng.integers(0, 256, (759, 1006), dtype=np.uint8)
    for (w, h, ltx, lty, ang) in [(191, 131, 400.3, 300.7, 33.2), (96, 66, -20.0, 10.0, -100.0), (381, 261, 800.5, 600.25, 179.9),
                                  (48, 33, 990.0, 740.0, 12.0), (24, 17, 3.0, 5.0, 0.0)]:
        roi = O.OracleMatcher._get_rotated_roi(src, (w, h), (np.float32(ltx), np.float32(lty)), ang)
        ptc = (np.float32((src.shape[1] - 1) / 2.0), np.float32((src.shape[0] - 1) / 2.0))
        lt = O.pt_rotate_pt2f((np.float32(ltx), np.float32(lty)), ptc, ang * O.D2R)
        m = cv2.getRotationMatrix2D((float(ptc[0]), float(ptc[1])), ang, 1)
        m[0, 2] -= float(np.float32(lt[0] - np.float32(3)))
        m[1, 2] -= float(np.float32(lt[1] - np.float32(3)))
        got = matcher.dbgWarpAffine(src, m, (w + 6, h + 6), 0)
        assert np.array_equal(got, roi), (w, h, ang)


def test_warp_affine_large(matcher):
    rng = np.random.default_rng(8)
    img = rng.integers(0, 256, (1500, 2048), dtype=np.uint8)
    m = cv2.getRotationMatrix2D((1023.5, 749.5), -119.979, 1)
    m[0, 2] += 120.5
    m[1, 2] += 300.0
    want = cv2.warpAffine(img, m, (2300, 2100), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=255)
    got = matcher.dbgWarpAffine(img, m, (2300, 2100), 255)
    assert np.array_equal(got, want)


# ---------------- T3: integer correlation row sums + window sums, bit-exact ----------------
@pytest.mark.parametrize("tw,th", [(12, 9), (24, 17), (48, 33), (54, 54), (27, 27), (14, 14), (96, 66), (191, 131), (1, 1), (5, 3),
                                   (381, 261), (130, 7)])
def test_corr_rows_bit_exact(matcher, tw, th):
    rng = np.random.default_rng(tw * 1000 + th)
    tpl = rng.integers(0, 256, (th, tw), dtype=np.uint8)
    roi = rng.integers(0, 256, (th + 6, tw + 6), dtype=np.uint8)
    rowsum, rowS, rowQ = matcher.dbgCorrRows(roi, tpl)
    want = O.ccorr_exact_rows(roi, tpl)                      # [7, 7, th]
    assert np.array_equal(rowsum.astype(np.int64), np.transpose(want, (2, 0, 1)))
    r64 = roi.astype(np.int64)
    for c in range(7):
        assert np.array_equal(rowS[:, c], r64[:, c:c + tw].sum(axis=1))
        assert np.array_equal(rowQ[:, c], (r64[:, c:c + tw] ** 2).sum(axis=1))


def test_corr_rows_saturated_large(matcher):
    """all-255 rows of the cfg1 template size: the s32 row sums must not overflow (762*255*255 < 2^31)."""
    tw, th = 762, 64
    tpl = np.full((th, tw), 255, np.uint8)
    roi = np.full((th + 6, tw + 6), 255, np.uint8)
    rowsum, rowS, rowQ = matcher.dbgCorrRows(roi, tpl)
    assert (rowsum == 762 * 255 * 255).all() and (rowS == 762 * 255).all() and (rowQ == 762 * 255 * 255).all()


# ---------------- T1: template learning ----------------
@pytest.mark.parametrize("case", ["cfg3_src6", "src8", "cfg1_synth", "cfg2_synth", "src4"])
def test_learn_pattern_matches_golden(matcher, golden_cases, case):
    c = golden_cases[case]
    configure(matcher, c["params"])
    assert matcher.learnPattern(get_image(c["tpl"]))
    lv = matcher.templateLevels()
    assert len(lv) == len(c["tpl_levels"])
    assert matcher.borderColor() == c["border_color"]
    import hashlib
    for got, want in zip(lv, c["tpl_levels"]):
        assert (got["w"], got["h"]) == (want["w"], want["h"])
        assert hashlib.sha256(got["pixels"].tobytes()).hexdigest()[:16] == want["sha"]       # bit-exact pyramid
        assert got["mean"] == want["mean"] and got["norm"] == want["norm"] and got["inv_area"] == want["inv_area"]
        assert got["result_equal1"] == want["equal1"]


# ---------------- T4: top-layer score map ----------------
@pytest.mark.parametrize("case", ["src8", "cfg3_src6"])
def test_top_score_map_bit_exact_vs_exact_oracle(matcher, golden_cases, case):
    c = golden_cases[case]
    configure(matcher, c["params"])
    tpl = get_image(c["tpl"])
    matcher.learnPattern(tpl)
    om = configure(O.OracleMatcher(), c["params"])
    om.learn_pattern(tpl)
    top = len(om.td.pyramid) - 1
    src = get_image(c["src"])
    pyr = O.build_pyramid(src, top)
    img = pyr[top]
    got = matcher.dbgTopScore(img)
    want = O.ccoeff_denominator(img, om.td, O.ccorr_exact_dense(img, om.td.pyramid[top]), top)
    assert got.shape == want.shape
    assert np.array_equal(got, want), float(np.abs(got - want).max())
    # reported delta against the cv::matchTemplate-fed map (DFT float numerator), tolerance only
    cvmap = O.ccoeff_denominator(img, om.td, cv2.matchTemplate(img, om.td.pyramid[top], cv2.TM_CCORR), top)
    assert float(np.abs(got - cvmap).max()) < 1e-3


# ---------------- T5: peak extraction ----------------
@pytest.mark.parametrize("block", [False, True])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_peaks_match_oracle(matcher, block, seed):
    rng = np.random.default_rng(seed)
    rows, cols = (211, 300) if block else (57, 66)
    score = rng.uniform(-0.2, 0.9, (rows, cols)).astype(np.float32)
    score = cv2.GaussianBlur(score, (0, 0), 1.5)
    # exact ties, including clamped +-1 plateaus
    for _ in range(12):
        y, x = int(rng.integers(0, rows)), int(rng.integers(0, cols))
        score[y, x] = 1.0
    tw, th = 9, 7
    om = O.OracleMatcher()
    om.max_pos, om.max_overlap = 20, 0.25 if seed == 2 else 0.0
    want = om.top_picks(score.copy(), (tw, th), 0.3, block)
    got = matcher.dbgPeaks(score, tw, th, block, 0.3, om.max_overlap, om.max_pos + 5)
    assert len(got) == len(want)
    for g, (loc, val) in zip(got, want):
        assert (int(g[0]), int(g[1])) == loc and np.float32(g[2]) == np.float32(val)


@pytest.mark.parametrize("shape", [(211, 300), (216, 288), (216, 300), (211, 288), (30, 300), (211, 17)])
@pytest.mark.parametrize("seed", [0, 1])
def test_peaks_match_oracle_mfc_blocks(matcher, shape, seed):
    """MFC s_BlockMax (MatchToolDlg.h:109-213): 2x template blocks, residue strips, last maximal block on ties,
    whole-map search when the table is empty"""
    rng = np.random.default_rng(100 + seed)
    rows, cols = shape
    score = rng.uniform(-0.2, 0.9, (rows, cols)).astype(np.float32)
    score = cv2.GaussianBlur(score, (0, 0), 1.5)
    for _ in range(12):
        y, x = int(rng.integers(0, rows)), int(rng.integers(0, cols))
        score[y, x] = 1.0
    tw, th = 9, 9 if shape[0] == 216 else 7        # 216 = 12 * 18, 288 = 16 * 18: shapes without residue
    om = O.OracleMatcher()
    om.mfc_compat = True
    om.max_pos, om.max_overlap = 20, 0.25 * seed
    want = om.top_picks(score.copy(), (tw, th), 0.3, True)
    got = matcher.dbgPeaks(score, tw, th, 2, 0.3, om.max_overlap, om.max_pos + 5)
    assert len(got) == len(want)
    for g, (loc, val) in zip(got, want):
        assert (int(g[0]), int(g[1])) == loc and np.float32(g[2]) == np.float32(val)


def test_peaks_nothing_above_threshold(matcher):
    score = np.full((20, 30), 0.1, np.float32)
    assert len(matcher.dbgPeaks(score, 5, 5, False, 0.5, 0.0, 10)) == 0
    assert len(matcher.dbgPeaks(score, 5, 5, True, 0.5, 0.0, 10)) == 0


# ---------------- T5..T7: the whole match() ----------------
ALL_CASES = ["src8", "src9", "test4_src3", "cfg3_src6", "cfg1_synth", "src4", "cfg2_synth", "src9_subpix"]


@pytest.mark.parametrize("case", ALL_CASES)
def test_match_against_golden(matcher, golden_cases, case):
    c = golden_cases[case]
    configure(matcher, c["params"])
    matcher.setTrace(True)
    assert matcher.learnPattern(get_image(c["tpl"]))
    src = get_image(c["src"])
    res = matcher.match(src)
    matcher.setTrace(False)
    # T0: source pyramid bit-exact
    import hashlib
    for l, sha in enumerate(c["src_pyr_sha"]):
        lv = matcher.traceLevel(l)
        assert lv is not None and hashlib.sha256(lv.tobytes()).hexdigest()[:16] == sha, "pyramid level %d" % l
    # T5: ordered top-layer candidate list (exact ties may permute: compare per score class)
    cand = matcher.traceCandidates()
    assert len(cand) == c["n_candidates"]
    want = np.array(c["candidates"])[:, :3] if c["n_candidates"] else np.zeros((0, 3))
    if c["n_candidates"]:
        assert np.array_equal(cand[:, 2].astype(np.float32), want[:, 2].astype(np.float32))
        ties = len(set(want[:, 2].tolist())) != len(want)
        if not ties:
            assert np.array_equal(cand[:, :2].astype(np.float32), want[:, :2].astype(np.float32))
    # T7: accepted set, order, score / angle / pose
    ties = len({r["score"] for r in c["results"]}) != len(c["results"])
    if case == "src9_subpix":
        assert_results_match(res, c["results"], 1e-4, 0.5, 0.1)     # ill-conditioned LSQ fit, see DESIGN.md
    else:
        assert_results_match(res, c["results"], ordered=not ties)


def test_match_equals_live_oracle_on_jittered_cfg1(matcher, golden_cases):
    """a pose set that is not in the golden file: oracle and GPU run on the same seeded input here."""
    import fpm_workloads as synth
    c = golden_cases["cfg1_synth"]
    tpl = get_image("Dst7")
    src = synth.cfg1_source(seed=21, tpl=tpl, jitter=True)
    configure(matcher, c["params"])
    matcher.learnPattern(tpl)
    got = matcher.match(src)
    om = configure(O.OracleMatcher(), c["params"])
    om.learn_pattern(tpl)
    want = om.match(src)
    assert len(want) == 3
    assert_results_match(got, want)


def test_batch_equals_single(matcher, golden_cases):
    c = golden_cases["src8"]
    configure(matcher, c["params"])
    matcher.learnPattern(get_image(c["tpl"]))
    a = get_image("Src8")
    b = get_image("Src9")
    frames = np.stack([a, b, a, np.zeros_like(a), b])
    single = [matcher.match(f) for f in frames]
    batch = matcher.matchBatch(frames)
    assert [len(x) for x in batch] == [len(x) for x in single]
    for x, y in zip(batch, single):
        assert_results_match(x, y, 0, 0, 0)
    assert len(single[0]) == 3 and len(single[3]) == 0


def test_device_batch_in_two_concurrent_halves_equals_single(matcher, golden_cases):
    """fpm_match_batch_device splits large batches into two half-batches on two internal handles (FPM_PARAM_SPLIT_BATCH)"""
    import ctypes as C
    import torch
    from fastest_image_pattern_matching_b200 import _lib as L
    from fastest_image_pattern_matching_b200.matcher import _convert
    c = golden_cases["src8"]
    configure(matcher, c["params"])
    matcher.learnPattern(get_image(c["tpl"]))
    a, b = get_image("Src8"), get_image("Src9")
    frames = np.stack([a, b, a, np.zeros_like(a), b])
    single = [matcher.match(f) for f in frames]
    d = torch.from_numpy(frames).cuda()
    B, H, W = frames.shape
    cap = matcher.result_capacity
    try:
        for split in (2, 0):
            matcher.setSplitBatch(split)
            res = (L.fpm_result * (cap * B))()
            counts = (C.c_int * B)()
            matcher.matchBatchRaw(d.data_ptr(), B, W, H, W, H * W, True, res, counts)
            assert [counts[i] for i in range(B)] == [len(x) for x in single]
            for i in range(B):
                assert_results_match(_convert(res[i * cap:(i + 1) * cap], counts[i]), single[i], 0, 0, 0)
        # the template learned later must reach the twin handle too
        matcher.setSplitBatch(2)
        c9 = golden_cases["src9"]
        configure(matcher, c9["params"])
        matcher.learnPattern(get_image(c9["tpl"]))
        single9 = [matcher.match(f) for f in frames]
        res = (L.fpm_result * (cap * B))()
        counts = (C.c_int * B)()
        matcher.matchBatchRaw(d.data_ptr(), B, W, H, W, H * W, True, res, counts)
        for i in range(B):
            assert_results_match(_convert(res[i * cap:(i + 1) * cap], counts[i]), single9[i], 0, 0, 0)
    finally:
        matcher.setSplitBatch(8)


def test_small_workspace_waves_give_same_result(matcher, golden_cases):
    c = golden_cases["src8"]
    configure(matcher, c["params"])
    matcher.learnPattern(get_image(c["tpl"]))
    src = get_image(c["src"])
    ref = matcher.match(src)
    matcher.setWorkspaceMB(0.5)
    try:
        res = matcher.match(src)
    finally:
        matcher.setWorkspaceMB(4096)
    assert_results_match(res, ref, 0, 0, 0)


def test_use_simd_off(matcher, golden_cases):
    """SIMD unchecked: the reference falls back to cv::matchTemplate in refinement; here the exact sum."""
    c = golden_cases["src8"]
    p = dict(c["params"], use_simd=False)
    configure(matcher, p)
    matcher.learnPattern(get_image(c["tpl"]))
    res = matcher.match(get_image(c["src"]))
    matcher.setUseSIMD(True)
    assert_results_match(res, c["results"], 1e-4, 0.05, 0.01)


# ---------------- guards / edge cases (src/TemplateMatcher.cpp:99-114 and SURVEY 8a) ----------------
def test_guards(matcher):
    matcher.clearPattern()
    assert not matcher.isPatternLearned()
    assert matcher.match(np.zeros((50, 50), np.uint8)) == []
    assert not matcher.learnPattern(np.zeros((0, 0), np.uint8))
    tpl = np.full((40, 40), 7, np.uint8)
    tpl[10:30, 10:30] = 200
    assert matcher.learnPattern(tpl) and matcher.isPatternLearned()
    assert matcher.match(np.zeros((20, 100), np.uint8)) == []
    assert matcher.match(np.zeros((30, 30), np.uint8)) == []
    assert matcher.match(np.zeros((0, 0), np.uint8)) == []
    matcher.setUserDefinedRect((1, 2, 3, 4))
    assert matcher.hasUserDefinedRect() and matcher.getUserDefinedRect() == (1, 2, 3, 4)


def _edge_case(matcher, tpl, src, params):
    configure(matcher, params)
    assert matcher.learnPattern(tpl)
    got = matcher.match(src)
    om = configure(O.OracleMatcher(), params)
    om.learn_pattern(tpl)
    want = om.match(src)
    return got, want


def test_flat_template_forces_score_one(matcher):
    tpl = np.full((20, 24), 90, np.uint8)
    rng = np.random.default_rng(2)
    src = rng.integers(0, 256, (90, 120), dtype=np.uint8)
    got, want = _edge_case(matcher, tpl, src, dict(max_pos=3, score=0.9, tolerance_angle=0, min_reduce_area=64))
    assert len(want) > 0
    assert_results_match(got, want, ordered=False)


def test_top_layer_zero_no_refinement(matcher):
    """template area <= MinReduceArea: iTopLayer == 0, top-layer picks are final (:272-276)."""
    rng = np.random.default_rng(3)
    src = cv2.GaussianBlur(rng.integers(0, 256, (120, 160), dtype=np.uint8), (0, 0), 2)
    tpl = src[40:55, 60:76].copy()
    got, want = _edge_case(matcher, tpl, src, dict(max_pos=2, score=0.8, tolerance_angle=20, min_reduce_area=256))
    assert len(want) >= 1
    assert_results_match(got, want)


def test_zero_tolerance_single_angle(matcher):
    rng = np.random.default_rng(4)
    src = cv2.GaussianBlur(rng.integers(0, 256, (300, 400), dtype=np.uint8), (0, 0), 2)
    tpl = src[100:164, 200:280].copy()
    got, want = _edge_case(matcher, tpl, src, dict(max_pos=2, score=0.8, tolerance_angle=0, min_reduce_area=256))
    assert len(want) == 1 and abs(want[0].ptLT[0] - 200) < 0.01
    assert_results_match(got, want)


def test_candidate_near_border(matcher):
    rng = np.random.default_rng(5)
    src = cv2.GaussianBlur(rng.integers(0, 256, (300, 400), dtype=np.uint8), (0, 0), 2)
    tpl = src[0:60, 0:90].copy()                      # ROI taps fall outside -> border 0 (:1089)
    got, want = _edge_case(matcher, tpl, src, dict(max_pos=2, score=0.6, tolerance_angle=30, min_reduce_area=256))
    assert len(want) >= 1
    assert_results_match(got, want)


def test_min_reduce_area_change_relearns(matcher, golden_cases):
    c = golden_cases["src8"]
    configure(matcher, c["params"])
    tpl, src = get_image(c["tpl"]), get_image(c["src"])
    matcher.learnPattern(tpl)
    matcher.setMinReduceArea(1024)                    # reference would index out of range (SURVEY 8a hazard)
    got = matcher.match(src)
    om = configure(O.OracleMatcher(), dict(c["params"], min_reduce_area=1024))
    om.learn_pattern(tpl)
    assert_results_match(got, om.match(src))


def test_tolerance_360_duplicate_orientations(matcher, golden_cases):
    c = golden_cases["src9"]
    p = dict(c["params"], tolerance_angle=360)
    got, want = _edge_case(matcher, get_image(c["tpl"]), get_image(c["src"]), p)
    assert_results_match(got, want)


# ---------------- angle-sharded stage API == whole match ----------------
@pytest.mark.parametrize("case", ["src8", "cfg3_src6"])
def test_stage_api_equals_match(matcher, golden_cases, case):
    c = golden_cases[case]
    configure(matcher, c["params"])
    matcher.learnPattern(get_image(c["tpl"]))
    src = get_image(c["src"])
    whole = matcher.match(src)
    n_ang = matcher.stageNumAngles(src.shape[1], src.shape[0])
    assert n_ang == c["n_angles"]
    world = 3
    per = (n_ang + world - 1) // world
    picks = [matcher.stageTop(src, r * per, min(n_ang, (r + 1) * per)) for r in range(world)]
    allp = np.concatenate(picks)
    cands = matcher.stageSortCandidates(allp)
    assert len(cands) == c["n_candidates"]
    matcher.stageTop(src, 0, 0)                                   # pyramid resident, no angles
    refined = [matcher.stageRefine(cands[r::world]) for r in range(world)]
    res = matcher.stageFinal(np.concatenate(refined))
    assert_results_match(res, whole, 0, 0, 0)


def test_angle_sharded_driver_single_rank(matcher, golden_cases):
    """dist.match_angle_sharded with the real engine (world 1) == match()."""
    from fastest_image_pattern_matching_b200 import dist as D
    c = golden_cases["src8"]
    configure(matcher, c["params"])
    matcher.learnPattern(get_image(c["tpl"]))
    src = get_image(c["src"])
    assert_results_match(D.match_angle_sharded(matcher, src, None), matcher.match(src), 0, 0, 0)
    rows = D.match_frames_sharded(matcher, [src, get_image("Src9")], None)
    assert rows[0].shape == (3, 12) and abs(rows[0][0, 0] - c["results"][0]["score"]) <= 1e-4


# ---------------- BASELINE.json configs 4 and 5 at full size, against the live oracle ----------------
def _cfg45(matcher, W, H, T, seeds):
    import fpm_workloads as synth
    tpl = synth.synth_template(T, 4)
    frames = [synth.synth_frame(W, H, tpl, s, 4) for s in seeds]
    params = dict(max_pos=4, score=0.8, tolerance_angle=180, min_reduce_area=256, max_overlap=0.0)
    configure(matcher, params)
    assert matcher.learnPattern(tpl)
    om = configure(O.OracleMatcher(), params)
    om.learn_pattern(tpl)
    return tpl, frames, om


def test_cfg4_full_size_batch(matcher):
    """cfg4: 4096x3072 frames x 512x512 template, +-180 deg, 4 instances per frame (batch of 3 here)."""
    tpl, frames, om = _cfg45(matcher, 4096, 3072, 512, [11, 12, 13])
    got = matcher.matchBatch(np.stack(frames))
    for f, g in zip(frames, got):
        want = om.match(f)
        assert len(want) == 4
        assert_results_match(g, want)


def test_cfg5_full_size_and_angle_sharded(matcher):
    """cfg5: one 8192x8192 frame x 1024x1024 template (L0 angular step 0.112 deg); whole match and the
    angle-sharded stage pipeline (4 virtual ranks) must both equal the oracle."""
    from fastest_image_pattern_matching_b200 import dist as D
    tpl, frames, om = _cfg45(matcher, 8192, 8192, 1024, [11])
    src = frames[0]
    want = om.match(src)
    assert len(want) == 4
    got = matcher.match(src)
    assert_results_match(got, want)
    n_ang = matcher.stageNumAngles(src.shape[1], src.shape[0])
    world = 4
    picks = np.concatenate([matcher.stageTop(src, *D.angle_range(n_ang, r, world)) for r in range(world)])
    cands = matcher.stageSortCandidates(picks)
    matcher.stageTop(src, 0, 0)
    refined = np.concatenate([matcher.stageRefine(cands[r::world]) for r in range(world)])
    refined = refined[np.argsort(refined[:, 0], kind="stable")]
    assert_results_match(matcher.stageFinal(refined), got, 0, 0, 0)


def test_mfc_compat_result_convention(matcher, golden_cases):
    """upstream MFC convention (MatchTool/MatchToolDlg.cpp:1085-1116): angle = -theta wrapped, TargetNum truncation,
    corners in double -- derived here from the Qt-convention golden results; reproduces the README sign (README.md:47-49)."""
    import math
    c = golden_cases["cfg3_src6"]
    configure(matcher, dict(c["params"], max_pos=7))
    matcher.learnPattern(get_image(c["tpl"]))
    src = get_image(c["src"])
    qt = matcher.match(src)
    matcher.setMfcCompat(True)
    try:
        mfc = matcher.match(src)
    finally:
        matcher.setMfcCompat(False)
    assert len(qt) == 15 and len(mfc) == 7                      # truncated to TargetNum
    w, h = 848, 446
    for q, m in zip(qt, mfc):
        ang = -q.dMatchedAngle
        ang = ang + 360 if ang < -180 else (ang - 360 if ang > 180 else ang)
        assert m.dMatchedAngle == ang and m.dMatchScore == q.dMatchScore and m.ptLT == q.ptLT
        a = -q.dMatchedAngle * math.pi / 180
        rt = (q.ptLT[0] + w * math.cos(a), q.ptLT[1] - w * math.sin(a))
        rb = (rt[0] + h * math.sin(a), rt[1] + h * math.cos(a))
        assert abs(m.ptRT[0] - rt[0]) < 1e-9 and abs(m.ptRT[1] - rt[1]) < 1e-9
        assert abs(m.ptRB[0] - rb[0]) < 1e-9 and abs(m.ptRB[1] - rb[1]) < 1e-9
        assert abs(m.ptCenter[0] - q.ptCenter[0]) < 1e-3


# ---------------- randomized differential test: GPU vs live oracle on small random scenes ----------------
def _random_scene(seed):
    import fpm_workloads as synth
    rng = np.random.default_rng(seed)
    W, H = int(rng.integers(300, 900)), int(rng.integers(240, 700))
    tw, th = int(rng.integers(24, 140)), int(rng.integers(20, 120))
    tpl = synth.background(tw, th, seed + 7, float(rng.uniform(1.0, 3.0)))
    tpl = cv2.normalize(tpl, None, 0, 255, cv2.NORM_MINMAX)
    cv2.circle(tpl, (tw // 3, th // 3), max(3, min(tw, th) // 5), 255, -1)
    cv2.rectangle(tpl, (tw // 2, th // 2), (tw - 3, th - 3), 0, -1)
    src = synth.background(W, H, seed + 13, float(rng.uniform(1.5, 4.0)))
    k = int(rng.integers(1, 5))
    tol = float(rng.choice([0.0, 15.0, 45.0, 180.0]))
    for _ in range(k):
        a = float(rng.uniform(-tol, tol)) if tol > 0 else 0.0
        cx, cy = float(rng.uniform(0.15 * W, 0.85 * W)), float(rng.uniform(0.15 * H, 0.85 * H))
        synth.paste_rotated(src, tpl, cx, cy, a)
    params = dict(max_pos=int(rng.integers(1, 8)), score=float(rng.choice([0.5, 0.7, 0.85])), tolerance_angle=tol,
                  min_reduce_area=int(rng.choice([64, 256, 1024])), max_overlap=float(rng.choice([0.0, 0.3, 0.8])))
    return src, tpl, params


@pytest.mark.parametrize("seed", list(range(16)))
def test_random_scenes_match_live_oracle(matcher, seed):
    src, tpl, params = _random_scene(1000 + seed)
    configure(matcher, params)
    assert matcher.learnPattern(tpl)
    got = matcher.match(src)
    om = configure(O.OracleMatcher(), params)
    om.learn_pattern(tpl)
    want = om.match(src)
    ties = len({r.score for r in want}) != len(want)
    assert_results_match(got, want, ordered=not ties)


def test_unaligned_device_frames(matcher, golden_cases):
    """frames at an odd device address / odd pitch take the byte-granular load paths of pyrDown and warp."""
    import torch
    c = golden_cases["src8"]
    configure(matcher, c["params"])
    matcher.learnPattern(get_image(c["tpl"]))
    src = get_image(c["src"])
    H, W = src.shape
    pitch = W + 3
    buf = torch.zeros(2 * H * pitch + 64, dtype=torch.uint8, device="cuda")
    view = buf[1:1 + 2 * H * pitch].view(2, H, pitch)
    view[:, :, :W] = torch.from_numpy(src).cuda()
    res, counts = matcher.matchBatchRaw(view.data_ptr(), 2, W, H, pitch, H * pitch, True)
    assert counts[0] == 3 and counts[1] == 3
    want = c["results"]
    cap = matcher.result_capacity
    for b in range(2):
        for i, w in enumerate(want):
            r = res[b * cap + i]
            assert abs(r.score - w["score"]) <= 1e-4 and abs(r.cx - w["cx"]) <= 0.05 and abs(r.cy - w["cy"]) <= 0.05


# ---------------- MFC-only modes of the upstream dialog (MatchTool/MatchToolDlg.cpp) vs the oracle ----------------
@pytest.mark.parametrize("mode", ["stop_layer1", "bitwise_not", "tolerance_range", "tolerance_range_invalid", "mfc_compat"])
def test_mfc_only_modes(matcher, golden_cases, mode):
    c = golden_cases["src8"]
    tpl, src = get_image(c["tpl"]), get_image(c["src"])
    om = configure(O.OracleMatcher(), c["params"])
    configure(matcher, c["params"])
    try:
        if mode == "stop_layer1":
            om.stop_layer1 = True
            matcher.setStopLayer1(True)
        elif mode == "bitwise_not":
            om.bitwise_not = True
            matcher.setBitwiseNot(True)
            tpl = 255 - tpl
        elif mode == "tolerance_range":
            om.tolerance_range = (-30.0, 20.0, 40.0, 80.0)
            matcher.setToleranceRange(om.tolerance_range)
        elif mode == "tolerance_range_invalid":
            om.tolerance_range = (30.0, 20.0, 40.0, 80.0)
            matcher.setToleranceRange(om.tolerance_range)
        elif mode == "mfc_compat":
            om.mfc_compat = True
            matcher.setMfcCompat(True)
        om.learn_pattern(tpl)
        assert matcher.learnPattern(tpl)
        want = om.match(src)
        got = matcher.match(src)
    finally:
        matcher.setStopLayer1(False); matcher.setBitwiseNot(False); matcher.setToleranceRange(None); matcher.setMfcCompat(False)
    assert len(want) == {"stop_layer1": 3, "bitwise_not": 3, "tolerance_range": 2, "tolerance_range_invalid": 0, "mfc_compat": 3}[mode]
    assert_results_match(got, want)
