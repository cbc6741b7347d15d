"""Scale-tolerant template sets (fpm_match_set_scaled*, fpm_match_ingested_set_scaled*, fpm_match_set_sharded_scaled*).

- For every (frame, template) the records and scales of a set are bit for bit those of a handle holding only that template
  (fpm_match_scaled with the same parameters and range): ranges [0.8, 1.25] and [0.9, 1.1], the fixed scale 1.2 and [1, 1],
  on a set whose groups have different top-level sizes (so different scale schedules) plus a masked group; host and device
  frames, batches of 1 and 16 (split halves), async descent on and off, workspace waves, the correctness-relevant parameters
  and tensor-core modes 0-4 and 6.
- A range, another, then the first again on one handle equal fresh handles (each group's plan and slot scales are its own).
- A 3-template set at [0.8, 1.25] matches ScaledOracleMatcher per template, with the oracle's scales.
- At [1, 1] the scaled calls are fpm_match_set_batch / _merged bit for bit with every scale 1.0 (M12, the rotation set).
- Merged: the CPU merge of the scaled per-template lists, including two templates that hit one instance at different scales.
- Angle-sharded: virtual ranks 1, 2, 3, 8 and an NCCL rank equal the one-GPU scaled lists with the unscaled call's collectives.
- GlyphReader(scale_range=...) reads the M12 text printed at 0.9 and 1.15 times the glyph size; without a range it does not.
- Refusals: the old set calls keep refusing ranges, the new ones refuse min > max, TRACE, a bad max_overlap, NULL labels.
"""
import ctypes as C
import math

import cv2
import numpy as np
import pytest

import fpm_workloads as synth
from oracle import oracle as O
from tests.helpers import assert_results_match, configure, get_image
from tests.masked_oracle import disc_mask
from tests.scaled_oracle import ScaledOracleMatcher, paste_scaled
from tests.test_gpu_set_merge import merge_reference
from tests.test_gpu_template_set import _glyphs, _matcher, _rotation_set, _scenes, _tpl
from tests.test_ocr import KNOWN_TEXT

pytestmark = pytest.mark.gpu

RANGES = [(0.8, 1.25), (0.9, 1.1), (1.2, 1.2), (1.0, 1.0)]
SROT = {"max_pos": 6, "score": 0.6, "tolerance_angle": 180, "max_overlap": 0.3}
L_ERR = -1


def _set_tpls():
    """groups of different level-0 sizes (72x40, 30x30 with a flat member, 44x26), and a masked 48x48 group"""
    tpls = [_tpl(72, 40, 1), _tpl(72, 40, 2), _tpl(30, 30, 5), _tpl(30, 30, 6, flat=200), _tpl(44, 26, 8),
            _tpl(48, 48, 11), _tpl(48, 48, 12)]
    masks = [None] * 5 + [disc_mask(48, 48), disc_mask(48, 48)]
    return tpls, masks


def _scaled_scenes(tpls, n, w=420, h=300, seed=0):
    """frames with the templates planted at seeded poses and scales in [0.8, 1.25]"""
    rng = np.random.default_rng(seed)
    frames = []
    for i in range(n):
        f = synth.background(w, h, seed * 100 + i)
        for t in tpls:
            if rng.random() < 0.7:
                paste_scaled(f, t, float(rng.uniform(60, w - 60)), float(rng.uniform(60, h - 60)), float(rng.uniform(-180, 180)),
                             float(rng.uniform(0.8, 1.25)))
        frames.append(f)
    return np.stack(frames)


def _ptr(frames, on_device, keep):
    f = np.ascontiguousarray(frames)
    if not on_device:
        keep.append(f)
        return f.ctypes.data
    import torch
    t = torch.from_numpy(f).cuda()
    keep.append(t)
    return t.data_ptr()


def _recs(res, sc, base, n):
    return [(bytes(res[base + i]), sc[base + i]) for i in range(n)]


def _single_lists(tpl, mask, frames, params, rng, extra=None):
    """[frame] lists of (record bytes, scale) of a handle holding only tpl: fpm_match_scaled on device frames"""
    m = _matcher(params, extra)
    m.setScaleRange(*rng)
    assert m.learnPattern(tpl, mask)
    keep = []
    B, H, W = frames.shape
    cap = m.result_capacity
    from fastest_image_pattern_matching_b200 import _lib as L
    res, sc, n = (L.fpm_result * (cap * B))(), (C.c_double * (cap * B))(), (C.c_int * B)()
    rc = m._lib.fpm_match_scaled(m._h, _ptr(frames, True, keep), 1, B, W, H, W, H * W, res, sc, cap, n)
    assert rc == 0, m._lib.fpm_last_error(m._h).decode()
    out = [_recs(res, sc, b * cap, min(n[b], cap)) for b in range(B)]
    m.close()
    return out


def _singles(tpls, masks, frames, params, rng, extra=None):
    per_t = [_single_lists(t, mk, frames, params, rng, extra) for t, mk in zip(tpls, masks)]
    return [[per_t[t][b] for t in range(len(tpls))] for b in range(len(frames))]


def _set_handle(tpls, masks, params, rng, extra=None):
    m = _matcher(params, extra)
    m.setScaleRange(*rng)
    assert m.learnPatternSet(tpls, masks if any(x is not None for x in masks) else None)
    return m


def _set_lists(m, frames, on_device):
    """[frame][template] lists of (record bytes, scale) of fpm_match_set_scaled"""
    keep = []
    B, H, W = frames.shape
    T, cap = m.patternSetSize(), m.result_capacity
    res, counts, sc = m.matchSetBatchRaw(_ptr(frames, on_device, keep), B, W, H, W, H * W, on_device, scaled=True)
    return [[_recs(res, sc, (b * T + t) * cap, min(counts[b * T + t], cap)) for t in range(T)] for b in range(B)]


def _merged_lists(m, frames, on_device, max_overlap):
    """fpm_match_set_scaled_merged: ([frame][(label, record bytes, scale)], counts, [frame][template] set counts)"""
    keep = []
    B, H, W = frames.shape
    T, cap = m.patternSetSize(), m.result_capacity
    res, labels, counts, setc, sc = m.matchSetBatchMergedRaw(_ptr(frames, on_device, keep), B, W, H, W, H * W, on_device,
                                                             max_overlap, scaled=True)
    got = [[(labels[b * cap + k], bytes(res[b * cap + k]), sc[b * cap + k]) for k in range(min(counts[b], cap))] for b in range(B)]
    return got, list(counts), [list(setc[b * T:(b + 1) * T]) for b in range(B)]


def _assert_equal(got, want, what):
    for b in range(len(want)):
        for t in range(len(want[b])):
            assert got[b][t] == want[b][t], (what, b, t, len(got[b][t]), len(want[b][t]))


def _found(lists):
    return sum(len(x) for f in lists for x in f)


# ---- 1. a set equals its single handles, bit for bit, scales included ------------------------------------------
@pytest.mark.parametrize("rng", RANGES)
def test_set_equals_single_handles(rng):
    tpls, masks = _set_tpls()
    frames = _scaled_scenes(tpls, 3, seed=1)
    want = _singles(tpls, masks, frames, SROT, rng)
    m = _set_handle(tpls, masks, SROT, rng)
    try:
        for dev in (False, True, True):                     # the second device call runs every group from its cached plan
            _assert_equal(_set_lists(m, frames, dev), want, (rng, dev))
    finally:
        m.close()
    assert _found(want) > 0
    if rng == (0.8, 1.25):
        assert {s for f in want for x in f for _, s in x} - {1.0}, "no instance found away from scale 1"


@pytest.mark.parametrize("async_descent", [0, 1])
def test_batch_of_16_in_two_half_batches(async_descent):
    tpls, masks = _set_tpls()
    frames = _scaled_scenes(tpls, 16, w=360, h=280, seed=5)
    rng = (0.8, 1.25)
    extra = {"setAsyncDescent": async_descent}
    want = _singles(tpls, masks, frames, SROT, rng, extra)
    m = _set_handle(tpls, masks, SROT, rng, extra)
    try:
        for dev in (False, True):
            _assert_equal(_set_lists(m, frames, dev), want, dev)
        b1 = _set_lists(m, frames[:1], True)                # a batch of one (no split)
        assert b1[0] == want[0]
    finally:
        m.close()


def test_workspace_waves():
    tpls, masks = _set_tpls()
    frames = _scaled_scenes(tpls, 2, seed=7)
    rng = (0.9, 1.1)
    extra = {"setWorkspaceMB": 0.25}
    want = _singles(tpls, masks, frames, SROT, rng, extra)
    m = _set_handle(tpls, masks, SROT, rng, extra)
    try:
        _assert_equal(_set_lists(m, frames, True), want, "waves")
    finally:
        m.close()
    assert want == _singles(tpls, masks, frames, SROT, rng)


# ---- 2. plan and scale caching across ranges --------------------------------------------------------------------
def test_plan_and_scale_cache_across_ranges():
    tpls, masks = _set_tpls()
    frames = _scaled_scenes(tpls, 2, seed=9)
    fresh = {}
    for rng in [(0.8, 1.25), (1.1, 1.1)]:
        m = _set_handle(tpls, masks, SROT, rng)
        fresh[rng] = _set_lists(m, frames, True)
        m.close()
    assert fresh[(0.8, 1.25)] == _singles(tpls, masks, frames, SROT, (0.8, 1.25))
    m = _set_handle(tpls, masks, SROT, (1.0, 1.0))
    try:
        for rng in [(0.8, 1.25), (1.1, 1.1), (0.8, 1.25), (1.1, 1.1)]:
            m.setScaleRange(*rng)
            assert _set_lists(m, frames, True) == fresh[rng], rng
    finally:
        m.close()


# ---- 3. parameters ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["subpixel", "mfc", "stop_layer1", "bitwise_not", "tol_range", "tc0", "tc1", "tc2", "tc3",
                                     "tc4", "tc6"])
def test_parameters(variant):
    tpls, masks = _set_tpls()
    frames = _scaled_scenes(tpls, 1, seed=13)
    params, extra = dict(SROT), {}
    if variant == "subpixel":
        params["sub_pixel"] = True
    elif variant == "mfc":
        extra["setMfcCompat"] = True
    elif variant == "stop_layer1":
        extra["setStopLayer1"] = True
    elif variant == "bitwise_not":
        extra["setBitwiseNot"] = True
        frames = (255 - frames).astype(np.uint8)
    elif variant == "tol_range":
        extra["setToleranceRange"] = (-90, 30, 60, 150)
    else:
        extra["setTensorCores"] = int(variant[2:])
    rng = (0.9, 1.1)
    want = _singles(tpls, masks, frames, params, rng, extra)
    m = _set_handle(tpls, masks, params, rng, extra)
    try:
        _assert_equal(_set_lists(m, frames, False), want, variant)
    finally:
        m.close()
    assert _found(want) > 0


# ---- 4. the oracle anchor --------------------------------------------------------------------------------------
OPARAMS = dict(max_pos=10, score=0.8, tolerance_angle=20, max_overlap=0.2)


def test_three_templates_match_the_scaled_oracle():
    base = synth.synth_template(96, 41)
    tpls = [base[:72, :96].copy(), cv2.resize(synth.synth_template(64, 42), (64, 48), interpolation=cv2.INTER_AREA),
            synth.synth_template(56, 43)[:56, :56].copy()]
    src = synth.background(720, 540, 140, 3.0)
    poses = {0: [(130.0, 120.0, 8.0, 0.8), (560.0, 420.0, -12.0, 1.25)], 1: [(360.0, 110.0, -6.0, 1.0), (130.0, 420.0, 14.0, 1.2)],
             2: [(600.0, 130.0, 5.0, 0.85), (360.0, 330.0, -15.0, 1.1)]}
    for t, ps in poses.items():
        for cx, cy, a, s in ps:
            paste_scaled(src, tpls[t], cx, cy, a, s)
    rng = (0.8, 1.25)
    m = _set_handle(tpls, [None] * 3, OPARAMS, rng)
    try:
        got = m.matchSet(src, scaled=True)
    finally:
        m.close()
    for t, tpl in enumerate(tpls):
        om = configure(ScaledOracleMatcher(), OPARAMS)
        om.scale_min, om.scale_max = rng
        assert om.learn_pattern(tpl)
        want = om.match(src)
        assert len(want) >= 2, t
        assert_results_match(got[t], want)
        assert [r.dScale for r in got[t]] == [r.scale for r in want], t


# ---- 5. [1, 1] through the scaled calls is the unscaled set path ---------------------------------------------------
@pytest.mark.parametrize("case", ["m12", "rotation"])
def test_unit_range_is_the_unscaled_set_path(case):
    if case == "m12":
        import json
        import os
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cases.json")) as f:
            oc = json.load(f)["ocr_m12"]
        params, tpls = dict(oc["params"], score=0.7), _glyphs()
        src = get_image(oc["src"])
        frames = np.stack([src, np.roll(src, 3, axis=1)])
    else:
        params, tpls = SROT, _rotation_set()
        frames = _scenes(tpls, 3, seed=17)
    m = _matcher(params)
    m.learnPatternSet(tpls)
    B, H, W = frames.shape
    T, cap = m.patternSetSize(), m.result_capacity
    keep = []
    try:
        for dev in (False, True):
            ptr = _ptr(frames, dev, keep)
            res, counts = m.matchSetBatchRaw(ptr, B, W, H, W, H * W, dev)
            want = [[bytes(res[i * cap + k]) for k in range(min(counts[i], cap))] for i in range(B * T)]
            res2, counts2, sc = m.matchSetBatchRaw(ptr, B, W, H, W, H * W, dev, scaled=True)
            assert list(counts2) == list(counts)
            assert [[bytes(res2[i * cap + k]) for k in range(min(counts[i], cap))] for i in range(B * T)] == want
            assert all(sc[i * cap + k] == 1.0 for i in range(B * T) for k in range(min(counts[i], cap)))
            for ov in (0.0, 0.3):
                r1, l1, c1, s1 = m.matchSetBatchMergedRaw(ptr, B, W, H, W, H * W, dev, ov)
                r2, l2, c2, s2, sc2 = m.matchSetBatchMergedRaw(ptr, B, W, H, W, H * W, dev, ov, scaled=True)
                assert list(c1) == list(c2) and list(s1) == list(s2)
                for b in range(B):
                    n = min(c1[b], cap)
                    assert [bytes(r1[b * cap + k]) for k in range(n)] == [bytes(r2[b * cap + k]) for k in range(n)]
                    assert list(l1[b * cap:b * cap + n]) == list(l2[b * cap:b * cap + n])
                    assert all(sc2[b * cap + k] == 1.0 for k in range(n))
        assert sum(counts) > 0
    finally:
        m.close()


# ---- 6. merged ----------------------------------------------------------------------------------------------------
def _check_merged(m, frames, overlaps):
    from fastest_image_pattern_matching_b200 import _lib as L
    B = len(frames)
    T, cap = m.patternSetSize(), m.result_capacity
    for dev in (False, True):
        lists = _set_lists(m, frames, dev)
        for ov in overlaps:
            got, counts, setc = _merged_lists(m, frames, dev, ov)
            for b in range(B):
                recs = [[L.fpm_result.from_buffer_copy(x) for x, _ in lists[b][t]] for t in range(T)]
                scale_of = {(t, x): s for t in range(T) for x, s in lists[b][t]}
                ref = merge_reference(recs, ov)
                want = [(t, bytes(r), scale_of[(t, bytes(r))]) for t, r in ref[:cap]]
                assert counts[b] == len(ref) and got[b] == want, (dev, ov, b, counts[b], len(ref))
                assert setc[b] == [len(lists[b][t]) for t in range(T)]
    return got


def test_merged_equals_the_reference_merge():
    tpls, masks = _set_tpls()
    frames = _scaled_scenes(tpls, 4, seed=19)
    m = _set_handle(tpls, masks, SROT, (0.8, 1.25))
    try:
        _check_merged(m, frames, (0.0, 0.3))
    finally:
        m.close()


def test_scaled_rectangles_decide_the_merge():
    """template B is template A at 1.2 times its size; an instance of A at scale 1.2 is hit by A at ~1.2 and by B at ~1.0.
    Both records carry the 1.2-sized rectangle, so the merge keeps one of them."""
    from fastest_image_pattern_matching_b200.matcher import rrect_from3_host, rrect_overlap_host
    a = _tpl(48, 48, 31)
    b = cv2.resize(a, (58, 58), interpolation=cv2.INTER_LINEAR)
    src = synth.background(300, 240, 77, 3.0)
    paste_scaled(src, a, 150.0, 120.0, 10.0, 1.2)
    params = dict(max_pos=2, score=0.7, tolerance_angle=20, max_overlap=0.2)
    m = _set_handle([a, b], [None, None], params, (0.8, 1.25))
    try:
        per = m.matchSet(src, scaled=True)
        assert len(per[0]) == 1 and len(per[1]) == 1, [(len(x), [r.dScale for r in x]) for x in per]
        ra, rb = per[0][0], per[1][0]
        assert 1.1 < ra.dScale < 1.3 and 0.9 < rb.dScale < 1.1, (ra.dScale, rb.dScale)
        wa, wb = (math.hypot(r.ptRT[0] - r.ptLT[0], r.ptRT[1] - r.ptLT[1]) for r in (ra, rb))
        assert abs(wa - 48 * ra.dScale) < 0.01 and abs(wb - 58 * rb.dScale) < 0.01     # the scaled rectangles
        assert abs(wa - wb) < 2.0 and wa > 52.0, (wa, wb)                             # one size, well above A's own 48
        RA = rrect_from3_host(ra.ptLT, ra.ptRT, ra.ptRB)
        RB = rrect_from3_host(rb.ptLT, rb.ptRT, rb.ptRB)
        assert rrect_overlap_host(RA, RB, 0.5)[0] == 1
        merged = m.matchSetMerged(src, 0.5, scaled=True)
        assert len(merged) == 1
        t, r = merged[0]
        assert r.dScale == (ra if t == 0 else rb).dScale
        _check_merged(m, src[None], (0.5,))
    finally:
        m.close()


def test_ingested_and_ingested_merged_equal_the_host_calls():
    tpls, masks = _set_tpls()
    frames = _scaled_scenes(tpls, 1, seed=23)
    m = _set_handle(tpls, masks, SROT, (0.8, 1.25))
    try:
        want = m.matchSetBatch(frames, scaled=True)
        want_m = m.matchSetBatchMerged(frames, 0.3, scaled=True)
        ok, buf = cv2.imencode(".bmp", frames[0])
        m.ingestImage(buf.tobytes())
        key = lambda r: (r.dMatchScore, r.dMatchedAngle, r.ptCenter, r.ptLT, r.ptRT, r.ptRB, r.ptLB, r.dScale)
        assert [[[key(r) for r in x] for x in f] for f in m.matchIngestedSetBatch(scaled=True)] == \
            [[[key(r) for r in x] for x in f] for f in want]
        assert [[(t, key(r)) for t, r in f] for f in m.matchIngestedSetBatchMerged(0.3, scaled=True)] == \
            [[(t, key(r)) for t, r in f] for f in want_m]
        assert _found(want) > 0
    finally:
        m.close()


# ---- 7. angle-sharded -----------------------------------------------------------------------------------------------
def _key(r):
    return (r.dMatchScore, r.dMatchedAngle, r.ptCenter, r.ptLT, r.ptRT, r.ptRB, r.ptLB, r.dScale)


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_sharded_virtual_ranks(world):
    from fastest_image_pattern_matching_b200.matcher import match_set_sharded_virtual
    tpls, masks = _set_tpls()
    rng = (0.8, 1.25)
    f = _scaled_scenes(tpls, 1, seed=29 + world)[0]
    ref = _set_handle(tpls, masks, SROT, rng)
    hs = [_set_handle(tpls, masks, SROT, rng) for _ in range(world)]
    try:
        want = [[_key(r) for r in x] for x in ref.matchSet(f, scaled=True)]
        want_m = [(t, _key(r)) for t, r in ref.matchSetMerged(f, 0.3, scaled=True)]
        assert sum(len(x) for x in want) > 0

        def collectives(call):
            before = [m.collectiveCount() for m in hs]
            call()
            return [m.collectiveCount() - b for m, b in zip(hs, before)]
        # the collectives of the unscaled calls on the same handles (at [1, 1], where they run)
        for m in hs:
            m.setScaleRange(1.0, 1.0)
        plain_n = collectives(lambda: match_set_sharded_virtual(hs, f))
        merged_n = collectives(lambda: match_set_sharded_virtual(hs, f, max_overlap=0.3))
        assert min(plain_n + merged_n) > 0
        for m in hs:
            m.setScaleRange(*rng)
        for _ in range(2):                                   # the second call: cached plans
            got_all = []
            assert collectives(lambda: got_all.append(match_set_sharded_virtual(hs, f, scaled=True))) == plain_n
            for got in got_all[0]:
                assert [[_key(r) for r in x] for x in got] == want
            got_all = []
            assert collectives(lambda: got_all.append(match_set_sharded_virtual(hs, f, max_overlap=0.3, scaled=True))) == merged_n
            for got in got_all[0]:
                assert [(t, _key(r)) for t, r in got] == want_m
    finally:
        for m in hs + [ref]:
            m.close()


def test_sharded_set_of_one_and_nccl_single_rank():
    import torch
    from fastest_image_pattern_matching_b200.matcher import comm_available, comm_unique_id, match_set_sharded_virtual
    assert comm_available()
    tpls, masks = _set_tpls()
    rng = (0.8, 1.25)
    f = np.ascontiguousarray(_scaled_scenes(tpls, 1, seed=37)[0])
    # a set of one: the angle-sharded single-template scaled match
    one = _set_handle(tpls[:1], [None], SROT, rng)
    want1 = [_key(r) for r in one.match(f)]
    hs = [_set_handle(tpls[:1], [None], SROT, rng) for _ in range(3)]
    try:
        assert want1
        for got in match_set_sharded_virtual(hs, f, scaled=True):
            assert [_key(r) for r in got[0]] == want1
    finally:
        for m in hs + [one]:
            m.close()
    m = _set_handle(tpls, masks, SROT, rng)
    want = [[_key(r) for r in x] for x in m.matchSet(f, scaled=True)]
    want_m = [(t, _key(r)) for t, r in m.matchSetMerged(f, 0.3, scaled=True)]
    m.commInit(1, 0, comm_unique_id())
    try:
        d = torch.from_numpy(f).cuda()
        dev = dict(ptr=d.data_ptr(), shape=f.shape, stride=f.shape[1], on_device=True)
        assert [[_key(r) for r in x] for x in m.matchSetSharded(f, scaled=True)] == want
        assert [[_key(r) for r in x] for x in m.matchSetSharded(scaled=True, **dev)] == want
        assert [(t, _key(r)) for t, r in m.matchSetShardedMerged(f, 0.3, scaled=True)] == want_m
        assert [(t, _key(r)) for t, r in m.matchSetShardedMerged(max_overlap=0.3, scaled=True, **dev)] == want_m
    finally:
        m.commDestroy()
        m.close()


# ---- 8. demonstration: M12 text printed smaller and larger than the glyphs ---------------------------------------------
DEMO_SCALES = (0.9, 1.15)


@pytest.mark.parametrize("s", DEMO_SCALES)
def test_glyph_reader_reads_resized_text(s):
    import json
    import os
    from fastest_image_pattern_matching_b200 import GlyphReader
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cases.json")) as f:
        oc = json.load(f)["ocr_m12"]
    src = get_image(oc["src"])
    frame = cv2.resize(src, (round(src.shape[1] * s), round(src.shape[0] * s)), interpolation=cv2.INTER_LINEAR)
    glyphs = {ch: g for ch, g in zip(O.OCR_LETTERS, _glyphs())}
    params = dict(oc["params"], score=0.7)
    line_tol = 10.0 * s
    scaled = GlyphReader(glyphs, scale_range=(0.85, 1.2), **params)
    plain = GlyphReader(glyphs, scale_range=None, **params)          # None: no range, the unscaled reader
    try:
        text, _ = scaled.readBatch(frame[None], line_tol=line_tol, merge_overlap=0.3)[0]
        assert text == KNOWN_TEXT, (s, text)
        assert plain.readBatch(frame[None], line_tol=line_tol, merge_overlap=0.3)[0][0] != KNOWN_TEXT
    finally:
        for r in (scaled, plain):
            for m in r.matchers + ([r._set_matcher] if r._set_matcher else []):
                m.close()


# ---- 9. refusals ------------------------------------------------------------------------------------------------------
def test_refusals():
    from fastest_image_pattern_matching_b200 import FpmError
    from fastest_image_pattern_matching_b200 import _lib as L
    from fastest_image_pattern_matching_b200.matcher import match_set_sharded_virtual
    tpls, masks = _set_tpls()
    f = np.ascontiguousarray(_scaled_scenes(tpls, 1, w=240, h=200, seed=41)[0])
    m = _set_handle(tpls, masks, SROT, (0.9, 1.1))
    lib, h = m._lib, m._h
    try:
        # the old set calls keep refusing ranges with today's messages
        for call, name in ((lambda: m.matchSet(f), "fpm_match_set_batch"), (lambda: m.matchSetMerged(f, 0.3), "fpm_match_set_batch"),
                           (lambda: m.matchSetSharded(f), "fpm_match_set_sharded"),
                           (lambda: m.matchSetShardedMerged(f, 0.3), "fpm_match_set_sharded_merged"),
                           (lambda: match_set_sharded_virtual([m], f), "fpm_match_set_sharded_virtual")):
            with pytest.raises(FpmError, match=name + ": this call matches at scale 1 only"):
                call()
        ok, buf = cv2.imencode(".bmp", f)
        m.ingestImage(buf.tobytes())
        with pytest.raises(FpmError, match="fpm_match_set_batch: this call matches at scale 1 only"):
            m.matchIngestedSetBatch()
        assert m.matchIngestedSetBatch(scaled=True) is not None
        # the new calls: min > max, TRACE, max_overlap, NULL labels
        m.setScaleRange(1.2, 1.1)
        with pytest.raises(FpmError, match="fpm_match_set_scaled: FPM_PARAM_SCALE_MIN .* > FPM_PARAM_SCALE_MAX"):
            m.matchSet(f, scaled=True)
        with pytest.raises(FpmError, match="fpm_match_set_scaled_merged: FPM_PARAM_SCALE_MIN"):
            m.matchSetMerged(f, 0.3, scaled=True)
        with pytest.raises(FpmError, match="fpm_match_set_sharded_scaled: FPM_PARAM_SCALE_MIN"):
            m.matchSetSharded(f, scaled=True)
        with pytest.raises(FpmError, match="FPM_PARAM_SCALE_MIN"):
            match_set_sharded_virtual([m], f, scaled=True)
        m.setScaleRange(0.9, 1.1)
        m.setTrace(True)
        for call in (lambda: m.matchSet(f, scaled=True), lambda: m.matchSetMerged(f, 0.3, scaled=True),
                     lambda: m.matchIngestedSetBatch(scaled=True), lambda: m.matchSetSharded(f, scaled=True),
                     lambda: m.matchSetShardedMerged(f, 0.3, scaled=True)):
            with pytest.raises(FpmError, match="TRACE"):
                call()
        m.setTrace(False)
        for bad in (float("nan"), float("inf")):
            with pytest.raises(FpmError, match="fpm_match_set_scaled_merged: max_overlap must be finite"):
                m.matchSetMerged(f, bad, scaled=True)
            with pytest.raises(FpmError, match="max_overlap"):
                m.matchSetShardedMerged(f, bad, scaled=True)
            with pytest.raises(FpmError, match="max_overlap"):
                match_set_sharded_virtual([m], f, max_overlap=bad, scaled=True)
        T, cap = m.patternSetSize(), 8
        out, cnt, setc = (L.fpm_result * (cap * T))(), (C.c_int * T)(), (C.c_int * T)()
        W, H = f.shape[1], f.shape[0]
        assert lib.fpm_match_set_scaled_merged(h, f.ctypes.data, 0, 1, W, H, W, W * H, 0.3, out, None, None, cap, cnt, setc) == L_ERR
        assert "labels is NULL" in lib.fpm_last_error(h).decode()
        assert lib.fpm_match_set_sharded_scaled_merged(h, f.ctypes.data, W, H, W, 0, 0.3, out, None, None, cap, cnt, setc) == L_ERR
        assert "labels is NULL" in lib.fpm_last_error(h).decode()
        # scales = NULL is accepted, and the records are those of a call with scales
        assert lib.fpm_match_set_scaled(h, f.ctypes.data, 0, 1, W, H, W, W * H, out, None, cap, cnt) == 0
        want = m.matchSet(f, scaled=True)
        assert [min(cnt[t], cap) for t in range(T)] == [min(len(x), cap) for x in want]
        labels = (C.c_int * cap)()
        assert lib.fpm_match_set_scaled_merged(h, f.ctypes.data, 0, 1, W, H, W, W * H, 0.3, out, None, labels, cap, cnt, None) == 0
        assert lib.fpm_match_set_sharded_scaled(h, f.ctypes.data, W, H, W, 0, out, None, cap, cnt) == 0
        assert lib.fpm_match_ingested_set_scaled(h, out, None, cap, cnt) == 0
        # the single-template sharded and stage calls still refuse ranges
        one = _set_handle(tpls[:1], [None], SROT, (0.9, 1.1))
        n = C.c_int(0)
        assert one._lib.fpm_match_sharded(one._h, f.ctypes.data, W, H, W, 0, out, cap, C.byref(n)) == L_ERR
        assert "fpm_match_sharded: this call matches at scale 1 only" in one._lib.fpm_last_error(one._h).decode()
        picks = np.zeros(64, np.float64)
        assert one._lib.fpm_stage_top(one._h, f.ctypes.data, W, H, W, 0, 0, -1, picks.ctypes.data, 16, C.byref(n)) == L_ERR
        assert "fpm_stage_top" in one._lib.fpm_last_error(one._h).decode()
        assert one.matchSetSharded(f, scaled=True) is not None
        # min > max on a set of one: the refusal names the call that was made
        one.setScaleRange(1.2, 1.1)
        with pytest.raises(FpmError, match="^fpm error -1: fpm_match_set_scaled: FPM_PARAM_SCALE_MIN"):
            one.matchSet(f, scaled=True)
        with pytest.raises(FpmError, match="^fpm error -1: fpm_match: FPM_PARAM_SCALE_MIN"):
            one.match(f)
        one.close()
    finally:
        m.close()
