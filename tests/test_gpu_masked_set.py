"""Masked template sets (fpm_learn_set_masked): a don't-care mask per template of a set, matched on every set path.

For every (frame, template) the list of a masked set must be bit-identical (ordered, tolerance 0) to what a handle holding
only that template (fpm_learn_masked, or fpm_learn when unmasked) returns through fpm_match_batch_device.  The single masked
handles are checked against the masked oracle cell by cell in test_gpu_masked.py and test_gpu_masked_cells.py; a few pairs
are also compared with MaskedOracleMatcher directly here."""
import ctypes as C
import json
import os

import cv2
import numpy as np
import pytest

from oracle import oracle as O
from tests.helpers import assert_results_match, configure, get_image
from tests.masked_oracle import EDGE_MASKS, MASKS, MaskedOracleMatcher, disc_mask, mask_pyramid
from tests.test_gpu_set_merge import _check_merge
from tests.test_gpu_set_sharded import _check_virtual, _merged_rows
from tests.test_gpu_template_set import ROT, _glyphs, _match_frames, _matcher, _rows, _scenes, _tpl, _variants

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _mask(name, w, h):
    return dict(MASKS, **EDGE_MASKS)[name](w, h)


def _singles(tpls, masks, frames, params, extra=None):
    """[frame][template] lists of one handle per template (fpm_learn_masked / fpm_learn), device frames"""
    out = [[None] * len(tpls) for _ in range(len(frames))]
    for t, (tpl, mk) in enumerate(zip(tpls, masks)):
        m = _matcher(params, extra)
        assert m.learnPattern(tpl, mk)
        for b, lst in enumerate(_match_frames(m, frames, True, False)):
            out[b][t] = lst
        m.close()
    return out


def _set(tpls, masks, params, extra=None):
    m = _matcher(params, extra)
    assert m.learnPatternSet(tpls, masks)
    assert m.patternSetSize() == len(tpls)
    return m


def _check(tpls, masks, frames, params, extra=None, on_device=(False, True)):
    """the masked set's lists against the single handles', host and / or device frames; returns the set's lists"""
    want = _singles(tpls, masks, frames, params, extra)
    m = _set(tpls, masks, params, extra)
    got = None
    for dev in on_device:
        got = _match_frames(m, frames, dev, True)
        for b in range(len(frames)):
            for t in range(len(tpls)):
                assert _rows(got[b][t]) == _rows(want[b][t]), (dev, b, t, len(got[b][t]), len(want[b][t]))
    m.close()
    return got


def _profile(m, frame):
    """{kernel name: launches} of one matchSet"""
    m.setProfile(True)
    m.profileReset()
    m.matchSet(frame)
    p = {k: v[1] for k, v in m.profile().items()}
    m.setProfile(False)
    return p


# ---- 1. masked parts: five masks in one group, an unmasked member of the same size, a masked member of another size --
PART_MASKS = ["disc", "ring", "corner_cut", "holed", "comb"]


def _parts():
    tpls = [_tpl(72, 40, 30 + k) for k in range(len(PART_MASKS))] + [_tpl(72, 40, 40), _tpl(96, 64, 41)]
    masks = [_mask(n, 72, 40) for n in PART_MASKS] + [None, _mask("ring", 96, 64)]
    return tpls, masks


def test_parts_set_equals_single_handles_in_three_groups():
    tpls, masks = _parts()
    frames = _scenes(tpls, 3, seed=1)
    got = _check(tpls, masks, frames, ROT)
    assert sum(len(got[b][t]) for b in range(3) for t in range(len(tpls))) > 0
    # groups: the five masked 72x40, the unmasked 72x40 (the same size and border colour), the masked 96x64 alone
    m = _set(tpls, masks, ROT)
    p = _profile(m, frames[0])
    assert p["fpm_top_score_kernel(masked)"] == 2 and p["fpm_top_score_kernel"] == 1, p
    assert p["fpm_mask_window_kernel"] > 0
    m.close()


@pytest.mark.parametrize("async_descent", [0, 1])
def test_parts_batch_of_16_in_two_half_batches(async_descent):
    # 16 frames with split batch 8: the second handle learns the set with its masks
    tpls, masks = _parts()
    _check(tpls, masks, _scenes(tpls, 16, w=360, h=280, seed=5), ROT, {"setAsyncDescent": async_descent, "setSplitBatch": 8})


@pytest.mark.parametrize("variant", ["tc0", "tc1", "tc6", "small_workspace"])
def test_parts_correlation_paths_and_waves(variant):
    # the masked group of one (96 wide) takes the tensor cores under modes 1 and 6 as a single handle does
    tpls, masks = _parts()
    frames = _scenes(tpls, 2, seed=2)
    extra = {"tc0": {"setTensorCores": 0}, "tc1": {"setTensorCores": 1}, "tc6": {"setTensorCores": 6},
             "small_workspace": {"setWorkspaceMB": 0.25}}[variant]
    _check(tpls, masks, frames, ROT, extra, on_device=(True,))
    if variant == "small_workspace":
        m = _set(tpls, masks, ROT, extra)
        small = _profile(m, frames[0])["fpm_mask_window_kernel"]
        m.setWorkspaceMB(4096)
        assert small > _profile(m, frames[0])["fpm_mask_window_kernel"]      # several waves per layer
        m.close()


# ---- 2. every member walks its own runs ---------------------------------------------------------------------------
def _sprinkled(m):
    m = m.copy()
    m[1::4, 1::4] = 0
    return m


def test_members_use_their_own_runs():
    full = np.ones((40, 72), np.uint8)
    cc = _mask("corner_cut", 72, 40)
    # masks that differ at level 0 only: the runs of the last refinement layer tell them apart
    a, b = mask_pyramid(full, 2), mask_pyramid(_sprinkled(full), 2)
    assert not np.array_equal(a[0], b[0]) and all(np.array_equal(x, y) for x, y in zip(a[1:], b[1:]))
    g1 = ([_tpl(72, 40, 60 + k) for k in range(4)], [full, _sprinkled(full), cc, _sprinkled(cc)])
    # members that keep very different pixel counts at every level, the top layer included
    g2 = ([_tpl(64, 64, 70 + k) for k in range(4)], [disc_mask(64, 64, 0.6), _mask("ring", 64, 64), _mask("holed", 64, 64),
                                                      _mask("sparse", 64, 64)])
    assert len({int(m.sum()) for m in g2[1]}) == 4
    for tpls, masks in (g1, g2):
        got = _check(tpls, masks, _scenes(tpls, 2, seed=8), ROT, on_device=(True,))
        assert sum(len(x) for per in got for x in per) > 0


# ---- 3. flat members ----------------------------------------------------------------------------------------------
def _flat_under_mask(w, seed):
    """a textured template whose middle is one grey: flat under a small disc at every level"""
    t = _tpl(w, w, seed).copy()
    t[6:-6, 6:-6] = 200
    return t, disc_mask(w, w, 0.3)


def test_flat_members():
    # member 0 flat under its mask, the others not: the window sums still run for the group
    f, fm = _flat_under_mask(64, 50)
    om = MaskedOracleMatcher()
    assert om.learn_pattern(f, fm) and all(om.td.result_equal1)
    tpls, masks = [f, _tpl(64, 64, 51), _tpl(64, 64, 52)], [fm, _mask("ring", 64, 64), _mask("corner_cut", 64, 64)]
    frames = _scenes(tpls, 2, seed=9)
    _check(tpls, masks, frames, ROT, on_device=(True,))
    m = _set(tpls, masks, ROT)
    assert _profile(m, frames[0])["fpm_mask_window_kernel"] > 0
    m.close()
    # every member flat: no window sums at all
    (f1, m1), (f2, m2) = _flat_under_mask(48, 53), _flat_under_mask(48, 54)
    m2 = m2.copy()
    m2[:, :24] = 0
    tpls, masks = [f1, f2], [m1, m2]
    _check(tpls, masks, frames, ROT, on_device=(True,))
    m = _set(tpls, masks, ROT)
    assert _profile(m, frames[0]).get("fpm_mask_window_kernel", 0) == 0
    m.close()


# ---- 4. the masked oracle directly --------------------------------------------------------------------------------
def test_set_matches_the_masked_oracle(oracle_lib):
    tpls, masks = _parts()
    pick = [0, 4, 5, 6]                                       # disc, comb, the unmasked member, the masked 96x64
    frame = _scenes(tpls, 1, w=320, h=240, seed=12)[0]
    m = _set(tpls, masks, ROT)
    got = m.matchSet(frame)
    m.close()
    for t in pick:
        om = configure(MaskedOracleMatcher(), ROT)
        assert om.learn_pattern(tpls[t], masks[t])
        assert_results_match(got[t], om.match(frame), ordered=False)
    assert sum(len(got[t]) for t in pick) > 0


# ---- 5. merged, ingested and angle-sharded paths ------------------------------------------------------------------
def test_merged_equals_the_reference_merge():
    tpls, masks = _parts()
    m = _set(tpls, masks, ROT)
    out = _check_merge(m, _scenes(tpls, 3, seed=14), (0.0, 0.3))
    assert any(out[(True, 0.3)][1])
    m.close()


def test_ingested_and_ingested_merged():
    tpls, masks = _parts()
    frames = _scenes(tpls, 4, seed=15)
    files = [cv2.imencode(".jpg", f, [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes() for f in frames]
    m = _set(tpls, masks, ROT)
    m.ingestJpegBatch(files)
    got = m.matchIngestedSetBatch()
    got_m = m.matchIngestedSetBatchMerged(0.3)
    decoded = np.stack([m.ingestedFramePixels(i) for i in range(len(files))])
    want = _singles(tpls, masks, decoded, ROT)
    assert [[_rows(x) for x in per] for per in got] == [[_rows(x) for x in per] for per in want]
    assert [_merged_rows(x) for x in got_m] == [_merged_rows(x) for x in m.matchSetBatchMerged(decoded, 0.3)]
    assert sum(len(x) for per in got for x in per) > 0
    m.close()


@pytest.mark.parametrize("world", [1, 2, 3])
def test_sharded_virtual_ranks(world):
    tpls, masks = _parts()
    ref = _set(tpls, masks, ROT)
    hs = [_set(tpls, masks, ROT) for _ in range(world)]
    try:
        for f in _scenes(tpls, 2, seed=20 + world):
            _check_virtual(hs, f, ref.matchSet(f), {0.3: ref.matchSetMerged(f, 0.3)})
    finally:
        for m in hs + [ref]:
            m.close()


def test_sharded_nccl_single_rank():
    import torch
    from fastest_image_pattern_matching_b200.matcher import comm_available, comm_unique_id
    assert comm_available()
    tpls, masks = _parts()
    f = np.ascontiguousarray(_scenes(tpls, 1, seed=30)[0])
    m = _set(tpls, masks, ROT)
    want = [_rows(x) for x in m.matchSet(f)]
    want_m = _merged_rows(m.matchSetMerged(f, 0.3))
    m.commInit(1, 0, comm_unique_id())
    try:
        d = torch.from_numpy(f).cuda()
        dev = dict(ptr=d.data_ptr(), shape=f.shape, stride=f.shape[1], on_device=True)
        assert [_rows(x) for x in m.matchSetSharded(f)] == want
        assert [_rows(x) for x in m.matchSetSharded(**dev)] == want
        assert _merged_rows(m.matchSetShardedMerged(f, 0.3)) == want_m
        assert _merged_rows(m.matchSetShardedMerged(max_overlap=0.3, **dev)) == want_m
    finally:
        m.commDestroy()
        m.close()


# ---- 6. parameters ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["no_simd", "subpixel", "mfc", "bitwise_not", "tol_range"])
def test_parameters(variant):
    tpls, masks = _parts()
    params, extra = dict(ROT), {}
    if variant == "no_simd":
        params["use_simd"] = False
    elif variant == "subpixel":
        params["sub_pixel"] = True
    elif variant == "mfc":
        extra["setMfcCompat"] = True
    elif variant == "bitwise_not":
        extra["setBitwiseNot"] = True
    elif variant == "tol_range":
        extra["setToleranceRange"] = (-90, 30, 60, 150)
    _check(tpls, masks, _scenes(tpls, 2, seed=2), params, extra, on_device=(True,))


# ---- 7 / 8. M12 glyphs under stroke masks -------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ocr_case():
    with open(os.path.join(HERE, "golden", "cases.json")) as f:
        return json.load(f)["ocr_m12"]


def _stroke_mask(g):
    """the glyph's ink (Otsu), dilated by 2 pixels: it keeps pixels at every pyramid level"""
    thr, _ = cv2.threshold(g, 0, 255, cv2.THRESH_BINARY + cv2.THRESH_OTSU)
    return cv2.dilate((g < thr).astype(np.uint8), np.ones((5, 5), np.uint8))


def test_a_masked_group_issues_no_more_launches_than_one_masked_template(ocr_case):
    glyphs = _glyphs()
    shapes = [g.shape for g in glyphs]
    common = max(set(shapes), key=shapes.count)
    group = [g for g in glyphs if g.shape == common]
    masks = [_stroke_mask(g) for g in group]
    src = get_image(ocr_case["src"])
    one = _set(group[:1], masks[:1], ocr_case["params"])
    assert sum(len(x) for x in one.matchSet(src)) > 0
    n0 = one.launchCount(); one.matchSet(src); single = one.launchCount() - n0
    s = _set(group, masks, ocr_case["params"])
    s.matchSet(src)
    n0 = s.launchCount(); s.matchSet(src); grouped = s.launchCount() - n0
    assert grouped <= single, (grouped, single)
    one.close(); s.close()


def test_m12_stroke_masks(ocr_case):
    from fastest_image_pattern_matching_b200 import GlyphReader
    glyphs = _glyphs()
    masks = [_stroke_mask(g) for g in glyphs]
    src = get_image(ocr_case["src"])
    _check(glyphs, masks, src[None], ocr_case["params"])
    reader = GlyphReader(dict(zip(O.OCR_LETTERS, glyphs)), masks=dict(zip(O.OCR_LETTERS, masks)), **ocr_case["params"])
    frames = np.concatenate([src[None], _variants(src, 3, 13)])
    merged = reader.readBatch(frames, merge_overlap=0.3)
    per_glyph = reader.readBatch(frames)
    for f, (text_m, _), (_, per) in zip(frames, merged, per_glyph):
        text, per1 = reader.read(f)
        assert text_m == text
        for ch in reader.letters:
            assert _rows(per[ch]) == _rows(per1[ch])
    assert merged[0][0]


# ---- 9. refusals and re-learns ------------------------------------------------------------------------------------
def _learn_raw(m, tpls, masks, mask_strides):
    n = len(tpls)
    ptrs = (C.c_void_p * n)(*[t.ctypes.data for t in tpls])
    ws = (C.c_int * n)(*[t.shape[1] for t in tpls])
    hs = (C.c_int * n)(*[t.shape[0] for t in tpls])
    st = (C.c_int * n)(*[t.strides[0] for t in tpls])
    mp = None if masks is None else (C.c_void_p * n)(*[None if k is None else k.ctypes.data for k in masks])
    ms = None if mask_strides is None else (C.c_int * n)(*mask_strides)
    return m._lib.fpm_learn_set_masked(m._h, n, ptrs, ws, hs, st, mp, ms)


def test_refusals_and_relearns():
    from fastest_image_pattern_matching_b200 import FpmError
    tpls, masks = _parts()
    frames = _scenes(tpls, 2, seed=40)
    m = _matcher(ROT)
    err = lambda: m._lib.fpm_last_error(m._h).decode()
    w = [t.shape[1] for t in tpls]
    dot = np.zeros_like(tpls[1])
    dot[0, 0] = 1
    cases = [
        (masks, None, ["mask_strides"]),
        (masks, [w[0], w[1] - 1] + w[2:], ["template 1", "stride"]),
        (masks[:2] + [np.zeros_like(masks[2])] + masks[3:], w, ["template 2", "keeps no pixel"]),
        (masks[:1] + [dot] + masks[2:], w, ["template 1", "keeps no pixel at pyramid level 1"]),
    ]
    for mk, strides, words in cases:
        assert m.learnPatternSet(tpls, masks)
        assert _learn_raw(m, tpls, mk, strides) == -1
        assert all(x in err() for x in words), (words, err())
        assert not m.isPatternLearned() and m.patternSetSize() == 0
    with pytest.raises(ValueError, match="mask 1"):
        m.learnPatternSet(tpls, [masks[0], masks[1][:, :-1]] + masks[2:])
    with pytest.raises(ValueError):
        m.learnPatternSet(tpls, masks[:-1])
    with pytest.raises(FpmError, match="template 1"):
        m.learnPatternSet(tpls, [masks[0], dot] + masks[2:])
    # masks == NULL is fpm_learn_set, bit for bit
    plain = _set(tpls, None, ROT)
    want_plain = [[_rows(x) for x in per] for per in _match_frames(plain, frames, True, True)]
    assert _learn_raw(m, tpls, None, None) == 0
    assert [[_rows(x) for x in per] for per in _match_frames(m, frames, True, True)] == want_plain
    # a MinReduceArea change re-learns with the masks
    assert m.learnPatternSet(tpls, masks)
    m.setMinReduceArea(64)
    got = _match_frames(m, frames, True, True)
    fresh = _set(tpls, masks, dict(ROT, min_reduce_area=64))
    assert [[_rows(x) for x in per] for per in got] == [[_rows(x) for x in per] for per in _match_frames(fresh, frames, True, True)]
    # fpm_learn_set after a masked set: unmasked again
    m.setMinReduceArea(256)
    assert m.learnPatternSet(tpls)
    assert [[_rows(x) for x in per] for per in _match_frames(m, frames, True, True)] == want_plain
    for x in (m, plain, fresh):
        x.close()
