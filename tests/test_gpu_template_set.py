"""Template sets (fpm_learn_set / fpm_match_set_batch): n templates in one handle, matched against frame batches in shared
launches.  Every list of frame b / template t must be bit-identical (ordered, tolerance 0) to what a handle holding only
template t returns for frame b."""
import ctypes as C
import json
import os

import cv2
import numpy as np
import pytest

import fpm_workloads as synth
from oracle import oracle as O
from tests.helpers import assert_results_match, configure, get_image
from tests.test_ocr import KNOWN_TEXT

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _rows(lst):
    return [(r.dMatchScore, r.dMatchedAngle) + tuple(r.ptCenter) + tuple(r.ptLT) + tuple(r.ptRT) + tuple(r.ptRB) + tuple(r.ptLB)
            for r in lst]


def _matcher(params, extra=None, cap=512):
    from fastest_image_pattern_matching_b200 import TemplateMatcher
    m = configure(TemplateMatcher(0, result_capacity=cap), params)
    for k, v in (extra or {}).items():
        getattr(m, k)(v)
    return m


def _raw_lists(res, counts, n_lists, cap):
    from fastest_image_pattern_matching_b200.matcher import _convert
    return [_convert(res[i * cap:(i + 1) * cap], min(counts[i], cap)) for i in range(n_lists)]


def _match_frames(m, frames, on_device, set_call):
    """[frame][template] lists of a set handle (set_call) or [frame] lists of a single handle"""
    f = np.ascontiguousarray(frames)
    B, H, W = f.shape
    if on_device:
        import torch
        t = torch.from_numpy(f).cuda()
        ptr = t.data_ptr()
    else:
        ptr = f.ctypes.data
    if set_call:
        T = m.patternSetSize()
        res, counts = m.matchSetBatchRaw(ptr, B, W, H, W, H * W, on_device)
        flat = _raw_lists(res, counts, B * T, m.result_capacity)
        return [flat[b * T:(b + 1) * T] for b in range(B)]
    res, counts = m.matchBatchRaw(ptr, B, W, H, W, H * W, on_device)
    return _raw_lists(res, counts, B, m.result_capacity)


def _singles(tpls, frames, params, extra=None, on_device=True):
    out = [[None] * len(tpls) for _ in range(len(frames))]
    for t, tpl in enumerate(tpls):
        m = _matcher(params, extra)
        m.learnPattern(tpl)
        for b, lst in enumerate(_match_frames(m, frames, on_device, False)):
            out[b][t] = lst
        m.close()
    return out


def _check_set(tpls, frames, params, extra=None, on_device=(False, True), set_extra=None):
    want = _singles(tpls, frames, params, extra)
    m = _matcher(params, dict(extra or {}, **(set_extra or {})))
    m.learnPatternSet(tpls)
    assert m.patternSetSize() == len(tpls)
    got = None
    for dev in on_device:
        got = _match_frames(m, frames, dev, True)
        for b in range(len(frames)):
            for t in range(len(tpls)):
                assert _rows(got[b][t]) == _rows(want[b][t]), (dev, b, t, len(got[b][t]), len(want[b][t]))
    m.close()
    return got


# ---- M12: the reference's OCR test -----------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ocr_case():
    with open(os.path.join(HERE, "golden", "cases.json")) as f:
        return json.load(f)["ocr_m12"]


def _glyphs():
    return [get_image("M12/" + ch) for ch in O.OCR_LETTERS]


def _variants(src, n, seed):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        dx, dy = (int(v) for v in rng.integers(-6, 7, size=2))
        f = np.roll(np.roll(src, dy, axis=0), dx, axis=1).astype(np.int16)
        f += rng.integers(-4, 5, size=f.shape).astype(np.int16)
        out.append(np.clip(f, 0, 255).astype(np.uint8))
    return np.stack(out)


def test_m12_set_equals_single_handles_and_reads_the_text(ocr_case):
    from fastest_image_pattern_matching_b200 import GlyphReader
    src = get_image(ocr_case["src"])
    got = _check_set(_glyphs(), src[None], ocr_case["params"])[0]
    for ch, lst in zip(O.OCR_LETTERS, got):
        assert_results_match(lst, ocr_case["results"][ch], ordered=False)
    reader = GlyphReader({ch: g for ch, g in zip(O.OCR_LETTERS, _glyphs())}, **ocr_case["params"])
    frames = np.concatenate([src[None], _variants(src, 15, 11)])
    batch = reader.readBatch(frames)
    assert batch[0][0] == KNOWN_TEXT
    for f, (text, per) in zip(frames, batch):
        t1, per1 = reader.read(f)
        assert text == t1
        for ch in reader.letters:
            assert _rows(per[ch]) == _rows(per1[ch])


@pytest.mark.parametrize("batch", [3, 16])
@pytest.mark.parametrize("async_descent", [0, 1])
def test_m12_batches_host_and_device(ocr_case, batch, async_descent):
    src = get_image(ocr_case["src"])
    frames = _variants(src, batch, 100 + batch)
    extra = {"setAsyncDescent": async_descent}
    _check_set(_glyphs()[:12], frames, ocr_case["params"], extra)


# ---- rotation: synthetic scenes with the set's templates planted at seeded poses -------------------------------
def _tpl(w, h, seed, dark=False, flat=None):
    if flat is not None:
        return np.full((h, w), flat, np.uint8)
    t = cv2.resize(synth.synth_template(max(w, h), seed), (w, h), interpolation=cv2.INTER_AREA)
    return (t // 2) if dark else (128 + t // 2).astype(np.uint8)


def _rotation_set():
    a = _tpl(72, 40, 1)
    return [a, _tpl(72, 40, 2), a.copy(),                  # width >= 64 (tcgen05 alone, dp4a in the set), the same template twice
            _tpl(120, 10, 3), _tpl(120, 10, 4),            # refinement layer 60x5
            _tpl(30, 30, 5), _tpl(30, 30, 6, flat=200),    # a flat template in a group
            _tpl(30, 30, 7, dark=True),                    # same size, the other border colour: its own group
            _tpl(40, 130, 9), _tpl(40, 130, 10),           # ROI taller than 128 rows: one eval per correlation CTA
            _tpl(44, 26, 8)]                               # a group of one


def _scenes(tpls, n, w=420, h=300, seed=0):
    rng = np.random.default_rng(seed)
    mx, my = min(60, w // 3), min(60, h // 3)
    frames = []
    for i in range(n):
        f = synth.background(w, h, seed * 100 + i)
        for k, t in enumerate(tpls):
            if rng.random() < 0.7:
                synth.paste_rotated(f, t, float(rng.uniform(mx, w - mx)), float(rng.uniform(my, h - my)), float(rng.uniform(-180, 180)))
        frames.append(f)
    return np.stack(frames)


ROT = {"max_pos": 6, "score": 0.6, "tolerance_angle": 180, "max_overlap": 0.3}


def test_rotation_sets_with_mixed_groups():
    tpls = _rotation_set()
    got = _check_set(tpls, _scenes(tpls, 3, seed=1), ROT)
    assert _rows(got[0][0]) == _rows(got[0][2])               # the same template twice: identical lists
    assert sum(len(got[b][t]) for b in range(3) for t in range(len(tpls))) > 0


@pytest.mark.parametrize("async_descent", [0, 1])
def test_rotation_batch_of_16_in_two_half_batches(async_descent):
    # an angle sweep of >= 8 frames runs as two concurrent half-batches: the second handle learns the whole set
    tpls = _rotation_set()
    _check_set(tpls, _scenes(tpls, 16, w=360, h=280, seed=5), ROT, {"setAsyncDescent": async_descent})


@pytest.mark.parametrize("variant", ["no_simd", "subpixel", "mfc", "stop_layer1", "bitwise_not", "tol_range", "target_num",
                                     "small_workspace"])
def test_parameters(variant):
    tpls = _rotation_set()
    frames = _scenes(tpls, 2, seed=2)
    params, extra = dict(ROT), {}
    if variant == "no_simd":
        params["use_simd"] = False
    elif variant == "subpixel":
        params["sub_pixel"] = True
    elif variant == "mfc":
        extra["setMfcCompat"] = True
    elif variant == "stop_layer1":
        extra["setStopLayer1"] = True
    elif variant == "bitwise_not":
        extra["setBitwiseNot"] = True
    elif variant == "tol_range":
        extra["setToleranceRange"] = (-90, 30, 60, 150)
    elif variant == "target_num":
        params["max_pos"] = 2
    elif variant == "small_workspace":
        extra["setWorkspaceMB"] = 0.25
    _check_set(tpls, frames, params, extra, on_device=(True,))


def test_relearn_after_min_reduce_area_change():
    tpls = _rotation_set()
    frames = _scenes(tpls, 2, seed=3)
    m = _matcher(ROT)
    m.learnPatternSet(tpls)
    m.setMinReduceArea(64)
    got = _match_frames(m, frames, True, True)
    want = _singles(tpls, frames, dict(ROT, min_reduce_area=64))
    for b in range(len(frames)):
        for t in range(len(tpls)):
            assert _rows(got[b][t]) == _rows(want[b][t])


def test_score_jobs_beyond_the_grid_limit():
    tpls = [_tpl(16, 16, 20 + k) for k in range(20)]
    frames = _scenes(tpls[:3], 70, w=72, h=64, seed=4)
    params = {"max_pos": 2, "score": 0.7, "tolerance_angle": 180}
    step = np.degrees(np.arctan(2 / 16))                     # angle_schedule of a 16x16 top layer: 26 + 25 angles
    n_ang = int(np.ceil((180 + step) / step)) * 2 - 1
    assert len(frames) * len(tpls) * n_ang > 65535
    _check_set(tpls, frames, params, on_device=(True,))


def test_ingested_set_batch_equals_set_batch(ocr_case):
    src = get_image(ocr_case["src"])
    frames = _variants(src, 4, 7)
    files = [cv2.imencode(".jpg", f, [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes() for f in frames]
    m = _matcher(ocr_case["params"])
    m.learnPatternSet(_glyphs())
    m.ingestJpegBatch(files)
    got = m.matchIngestedSetBatch()
    decoded = np.stack([m.ingestedFramePixels(i) for i in range(len(files))])
    want = m.matchSetBatch(decoded)
    assert [[_rows(x) for x in per] for per in got] == [[_rows(x) for x in per] for per in want]
    m.close()


def test_guards_and_refusals(ocr_case):
    from fastest_image_pattern_matching_b200 import FpmError, match_multi
    from fastest_image_pattern_matching_b200 import _lib as L
    src = get_image(ocr_case["src"])
    glyphs = _glyphs()[:4]
    big = np.zeros((src.shape[0] + 10, 40), np.uint8)
    big[::3] = 255
    m = _matcher(ocr_case["params"])
    m.learnPatternSet(glyphs + [big])
    per = m.matchSet(src)
    assert per[-1] == []
    want = _singles(glyphs, src[None], ocr_case["params"])[0]
    assert [_rows(x) for x in per[:-1]] == [_rows(x) for x in want]
    lib, h = m._lib, m._h
    res = (L.fpm_result * 8)()
    n = (C.c_int * 8)()
    r5 = (C.c_double * 5)()
    u8 = np.zeros(src.size, np.uint8)
    calls = {
        "fpm_match": lambda: lib.fpm_match(h, src.ctypes.data, src.shape[1], src.shape[0], src.shape[1], res, 8, n),
        "fpm_match_batch": lambda: lib.fpm_match_batch(h, src.ctypes.data, 1, src.shape[1], src.shape[0], src.shape[1], src.size, res, 8, n),
        "fpm_match_batch_device": lambda: lib.fpm_match_batch_device(h, 1, 1, src.shape[1], src.shape[0], src.shape[1], src.size, res, 8, n),
        "fpm_match_ingested": lambda: lib.fpm_match_ingested(h, res, 8, n),
        "fpm_match_ingested_batch": lambda: lib.fpm_match_ingested_batch(h, res, 8, n),
        "fpm_learn_ingested": lambda: lib.fpm_learn_ingested(h),
        "fpm_match_sharded": lambda: lib.fpm_match_sharded(h, src.ctypes.data, src.shape[1], src.shape[0], src.shape[1], 0, res, 8, n),
        "fpm_match_sharded_virtual": lambda: lib.fpm_match_sharded_virtual((C.c_void_p * 1)(h), 1, src.ctypes.data, src.shape[1],
                                                                           src.shape[0], src.shape[1], res, 8, n),
        "fpm_stage_num_angles": lambda: lib.fpm_stage_num_angles(h, src.shape[1], src.shape[0]),
        "fpm_stage_top": lambda: lib.fpm_stage_top(h, src.ctypes.data, src.shape[1], src.shape[0], src.shape[1], 0, 0, 1, r5, 1, n),
        "fpm_stage_sort_candidates": lambda: lib.fpm_stage_sort_candidates(h, r5, 1, r5),
        "fpm_stage_refine": lambda: lib.fpm_stage_refine(h, r5, 1, r5, 1, n),
        "fpm_stage_final": lambda: lib.fpm_stage_final(h, r5, 1, res, 8, n),
        "fpm_tpl_levels": lambda: lib.fpm_tpl_levels(h),
        "fpm_tpl_level_info": lambda: lib.fpm_tpl_level_info(h, 0, None, None, None, None, None, None),
        "fpm_tpl_level_pixels": lambda: lib.fpm_tpl_level_pixels(h, 0, u8.ctypes.data),
        "fpm_tpl_border_color": lambda: lib.fpm_tpl_border_color(h),
    }
    for name, call in calls.items():
        assert call() == -1, name
        assert name in lib.fpm_last_error(h).decode() and "set of 5" in lib.fpm_last_error(h).decode(), name
    with pytest.raises(FpmError, match="fpm_match_multi"):
        match_multi([m], src)
    m.setTrace(True)
    with pytest.raises(FpmError, match="TRACE"):
        m.matchSet(src)
    m.setTrace(False)
    # bad sets leave nothing learned; the message names the index
    with pytest.raises(FpmError, match="template 1"):
        m.learnPatternSet([glyphs[0], np.zeros((0, 4), np.uint8)])
    assert m.patternSetSize() == 0 and not m.isPatternLearned()
    assert lib.fpm_learn_set(h, 0, None, None, None, None) == -1
    # fpm_learn after a set: a set of one, today's behaviour
    m.learnPattern(glyphs[0])
    assert m.patternSetSize() == 1
    assert _rows(m.match(src)) == _rows(want[0])
    m.clearPattern()
    assert m.patternSetSize() == 0
    m.close()


def test_a_group_issues_no_more_launches_than_one_template(ocr_case):
    glyphs = _glyphs()
    shapes = [g.shape for g in glyphs]
    common = max(set(shapes), key=shapes.count)
    group = [g for g in glyphs if g.shape == common]
    assert len(group) == 22
    src = get_image(ocr_case["src"])
    one = _matcher(ocr_case["params"])
    one.learnPattern(group[0])
    assert len(one.match(src)) > 0
    n0 = one.launchCount(); one.match(src); single = one.launchCount() - n0
    s = _matcher(ocr_case["params"])
    s.learnPatternSet(group)
    s.matchSet(src)
    n0 = s.launchCount(); s.matchSet(src); grouped = s.launchCount() - n0
    assert grouped <= single, (grouped, single)
    one.close(); s.close()
