"""CPU checks of the masked-template oracle (tests/masked_oracle.py): a full mask is the unmasked oracle exactly, masked
scores agree with cv2.matchTemplate(TM_CCOEFF_NORMED, mask=M), and the mask pyramid / level statistics equal a plain
numpy restatement of the definition."""
import math

import cv2
import numpy as np
import pytest

import fpm_workloads as synth
from oracle import oracle as O
from tests.helpers import configure
from tests.masked_oracle import (EDGE_MASKS, MASKS, MaskedOracleMatcher, disc_mask, mask_pyramid, mask_runs,
                                 masked_level_stats)


def _pyrdown_numpy(a):
    """cv::pyrDown of u8: 5x5 binomial kernel / 256, BORDER_REFLECT_101, (sum + 128) >> 8, size ((w+1)/2, (h+1)/2)"""
    h, w = a.shape
    k = np.array([1, 4, 6, 4, 1], np.int64)

    def refl(i, n):                                   # BORDER_REFLECT_101
        if n == 1:
            return 0
        while i < 0 or i >= n:
            i = -i if i < 0 else 2 * n - 2 - i
        return i

    s = a.astype(np.int64)
    dw, dh = (w + 1) // 2, (h + 1) // 2
    rows = np.zeros((h, dw), np.int64)
    for x in range(dw):
        for j in range(5):
            rows[:, x] += k[j] * s[:, refl(2 * x + j - 2, w)]
    out = np.zeros((dh, dw), np.int64)
    for y in range(dh):
        for i in range(5):
            out[y] += k[i] * rows[refl(2 * y + i - 2, h)]
    return ((out + 128) >> 8).astype(np.uint8)


def _template(w, h, seed):
    return synth.background(w, h, seed, 1.5)


def _scene(seed=3):
    tpl = _template(48, 40, seed)
    src = synth.background(260, 220, seed + 1, 2.0)
    src[30:70, 40:88] = tpl
    rot = cv2.warpAffine(tpl, cv2.getRotationMatrix2D((23.5, 19.5), 25, 1), (48, 40), borderMode=cv2.BORDER_REFLECT)
    src[120:160, 150:198] = rot
    return tpl, src


def test_full_mask_is_the_unmasked_oracle():
    tpl, src = _scene()
    params = dict(max_pos=5, score=0.5, tolerance_angle=40, min_reduce_area=64)
    a = configure(O.OracleMatcher(), params)
    b = configure(MaskedOracleMatcher(), params)
    assert a.learn_pattern(tpl)
    assert b.learn_pattern(tpl, np.full(tpl.shape, 9, np.uint8))
    assert a.td.templ_mean == b.td.templ_mean and a.td.templ_norm == b.td.templ_norm
    assert a.td.inv_area == b.td.inv_area and a.td.result_equal1 == b.td.result_equal1
    assert a.td.border_color == b.td.border_color
    ra, rb = a.match(src), b.match(src)
    assert len(ra) >= 2 and ra == rb


def _cv_masked(src, tpl, m):
    return cv2.matchTemplate(src, tpl, cv2.TM_CCOEFF_NORMED, mask=m)


def _compare_cv(src, tpl, m, got):
    want = _cv_masked(src, tpl, m).astype(np.float64)
    ok = np.isfinite(want)
    assert ok.mean() > 0.99
    diff = np.abs(got.astype(np.float64) - want)[ok]
    assert diff.max() <= 1e-4, diff.max()


@pytest.mark.parametrize("mask_name", sorted(MASKS))
@pytest.mark.parametrize("seed", [0, 1])
def test_masked_scores_match_cv2(mask_name, seed):
    _masked_scores_match_cv2(MASKS[mask_name], seed)


@pytest.mark.parametrize("mask_name", sorted(EDGE_MASKS))
@pytest.mark.parametrize("seed", [0, 1])
def test_edge_masked_scores_match_cv2(mask_name, seed):
    """comb, banded, frame and sparse masks: many runs, runs of one pixel, empty rows, runs at both edges"""
    _masked_scores_match_cv2(EDGE_MASKS[mask_name], seed)


def _masked_scores_match_cv2(mask_fn, seed):
    rng = np.random.default_rng(100 + seed)
    tpl = _template(37, 29, 200 + seed)
    m = mask_fn(37, 29)
    om = MaskedOracleMatcher()
    om.min_reduce_area = 64
    assert om.learn_pattern(tpl, m)
    src = synth.background(90, 70, 300 + seed, 1.0)
    src = np.clip(src.astype(np.int32) + rng.integers(-20, 21, src.shape), 0, 255).astype(np.uint8)
    for layer in range(len(om.td.pyramid)):
        t, ml = om.td.pyramid[layer], om.masks[layer]
        s = src if layer == 0 else cv2.resize(src, (max(t.shape[1] + 8, src.shape[1] >> layer), max(t.shape[0] + 8, src.shape[0] >> layer)))
        for use_simd in (True, False):           # refinement numerator (float row chain) and top-layer numerator (exact)
            got = om._match_template(s, layer, use_simd).copy()
            if om.td.result_equal1[layer]:       # a flat kept template (a frame's one-pixel top level): cv2 divides by 0
                assert (got == 1).all()
                continue
            _compare_cv(s, t, ml, got)


@pytest.mark.parametrize("name", ["Dst3", "Dst9", "Dst4"])
def test_masked_scores_match_cv2_golden(name):
    tpl = synth.load_fixture(name)
    src = synth.load_fixture({"Dst3": "Src3", "Dst9": "Src9", "Dst4": "Src4"}[name])
    th, tw = tpl.shape
    src = np.ascontiguousarray(src[:th + 24, :tw + 30])
    m = disc_mask(tw, th)
    om = MaskedOracleMatcher()
    assert om.learn_pattern(tpl, m)
    for use_simd in (True, False):
        _compare_cv(src, tpl, m, om._match_template(src, 0, use_simd).copy())


@pytest.mark.parametrize("mask_name", sorted(MASKS))
def test_mask_pyramid_and_stats_restated(mask_name):
    tpl = _template(61, 45, 11)
    m0 = MASKS[mask_name](61, 45)
    om = MaskedOracleMatcher()
    om.min_reduce_area = 64
    assert om.learn_pattern(tpl, m0 * 200)
    top = len(om.td.pyramid) - 1
    ms = [(m0 != 0).astype(np.uint8)]
    for _ in range(top):
        ms.append((_pyrdown_numpy(ms[-1] * 255) >= 128).astype(np.uint8))
    assert all(np.array_equal(a, b) for a, b in zip(ms, om.masks))
    assert all(np.array_equal(a, b) for a, b in zip(ms, mask_pyramid(m0, top)))
    for l, (t, m) in enumerate(zip(om.td.pyramid, ms)):
        v = t[m != 0].astype(np.int64)
        n = v.size
        mean = float(v.sum()) * (1.0 / n)
        var = max(float((v * v).sum()) * (1.0 / n) - mean * mean, 0.0)
        norm = math.sqrt(math.sqrt(var) ** 2) / math.sqrt(1.0 / n)
        assert om.td.templ_mean[l] == mean
        assert om.td.templ_norm[l] == norm
        assert om.td.inv_area[l] == 1.0 / n
        assert om.td.result_equal1[l] == (math.sqrt(var) ** 2 < O.DBL_EPSILON)
        assert np.array_equal(om.masked_pyr[l], t * m)
    kept0 = om.td.pyramid[0][ms[0] != 0].astype(np.int64)
    assert om.td.border_color == (255 if float(kept0.sum()) / kept0.size < 128 else 0)


def test_pyrdown_restatement_is_cv2():
    rng = np.random.default_rng(5)
    for shape in [(45, 61), (23, 31), (12, 16), (7, 9), (3, 2)]:
        a = rng.integers(0, 256, shape, dtype=np.uint8)
        assert np.array_equal(_pyrdown_numpy(a), cv2.pyrDown(a))


def test_refusals():
    tpl = _template(40, 30, 1)
    om = MaskedOracleMatcher()
    with pytest.raises(ValueError, match="keeps no pixel"):
        om.learn_pattern(tpl, np.zeros_like(tpl))
    one = np.zeros_like(tpl)
    one[0, 0] = 1                                # a single corner pixel vanishes at level 1
    with pytest.raises(ValueError, match="level 1"):
        om.learn_pattern(tpl, one)
    assert masked_level_stats(tpl, np.ones_like(tpl))[4] == tpl.size


# the shapes the GPU cell tests refine (tests/test_gpu_refine_cells.py SYNTH) and the wide masked templates
EDGE_SHAPES = [(120, 10, 64), (123, 36, 64), (65, 44, 64), (63, 40, 64), (122, 30, 256), (128, 60, 64), (30, 60, 64),
               (40, 32, 64), (64, 48, 256), (60, 44, 256), (5000, 64, 10000), (6400, 64, 10000)]


@pytest.mark.parametrize("mask_name", sorted(EDGE_MASKS))
def test_edge_masks_have_their_run_table_cases(mask_name):
    """each edge mask learns at every shape (no level empty) and has at level 0 or 1 (both refined when the pyramid has
    three levels) the case it is named for, checked on the level masks and not on the level-0 drawing"""
    for (w, h, mra) in EDGE_SHAPES:
        m0 = EDGE_MASKS[mask_name](w, h)
        om = MaskedOracleMatcher()
        om.min_reduce_area = mra
        assert om.learn_pattern(np.zeros((h, w), np.uint8), m0)
        runs = [mask_runs(ml) for ml in om.masks]
        if mask_name == "comb":
            assert max(len(r) for r in runs[0]) >= 8 and any(e - b == 1 for r in runs[0] for b, e in r), (w, h)
        elif mask_name == "banded":
            assert len(om.masks) > 2 and any(not r for r in runs[1]), (w, h)
        elif mask_name == "frame":
            for ml, lr in zip(om.masks[:2], runs[:2]):
                assert any(len(r) >= 2 and r[0][0] == 0 and r[-1][1] == ml.shape[1] for r in lr), (w, h)
        else:
            assert m0.mean() < 1 / 3 and any(e - b == 1 for r in runs[0] for b, e in r), (w, h)
