"""Merged set results (fpm_match_set_batch_merged): every frame's per-template lists of fpm_match_set_batch merged into one
labelled list with greedy rotated-rectangle NMS across templates.  Every merged call is compared with merge_reference, a
host restatement of the semantics over the lists fpm_match_set_batch returns with the same capacity, using the library's
host build of the shared geometry: equal counts, equal labels, bit-equal records."""
import ctypes as C
import json
import math
import os

import cv2
import numpy as np
import pytest

import fpm_workloads as synth
from oracle import oracle as O
from tests.helpers import get_image
from tests.test_gpu_template_set import ROT, _glyphs, _matcher, _rotation_set, _rows, _scenes, _tpl, _variants
from tests.test_ocr import KNOWN_TEXT

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def ocr_case():
    with open(os.path.join(HERE, "golden", "cases.json")) as f:
        return json.load(f)["ocr_m12"]


def _rrect(r):
    from fastest_image_pattern_matching_b200.matcher import rrect_from3_host
    return rrect_from3_host((r.ltx, r.lty), (r.rtx, r.rty), (r.rbx, r.rby))


def _far(a, b):
    # conservative: rectangles whose centres are this far apart cannot touch (decision 0)
    ra, rb = 0.5 * math.hypot(a[2], a[3]), 0.5 * math.hypot(b[2], b[3])
    return math.hypot(a[0] - b[0], a[1] - b[1]) > (ra + rb) * 1.01 + 2.0


def merge_reference(lists, max_overlap):
    """lists[t]: the records (fpm_result) of template t for one frame -> [(t, record)] kept, in merged order."""
    from fastest_image_pattern_matching_b200.matcher import rrect_overlap_host
    entries = []
    for t, lst in enumerate(lists):
        for i, r in enumerate(lst):
            assert r.score == float(np.float32(r.score))
            entries.append((-float(np.float32(r.score)), t, i, r))
    entries.sort(key=lambda e: e[:3])
    kept = []
    for _, t, _, r in entries:
        R = _rrect(r)
        if not any(kt != t and not _far(KR, R) and rrect_overlap_host(KR, R, max_overlap)[0] == 1 for kt, KR, _ in kept):
            kept.append((t, R, r))
    return [(t, r) for t, _, r in kept]


def _knife_edges(lists, max_overlap):
    """pairs of different templates whose overlap ratio lies within 1e-5 of the threshold (reported on a mismatch)"""
    from fastest_image_pattern_matching_b200.matcher import rrect_overlap_host
    rs = [(t, _rrect(r)) for t, lst in enumerate(lists) for r in lst]
    out = []
    for a in range(len(rs)):
        for b in range(a + 1, len(rs)):
            if rs[a][0] != rs[b][0] and not _far(rs[a][1], rs[b][1]):
                _, typ, ratio = rrect_overlap_host(rs[a][1], rs[b][1], max_overlap)
                if abs(ratio - max_overlap) < 1e-5:
                    out.append((rs[a][0], rs[b][0], typ, ratio))
    return out


def _device_ptr(frames, on_device, keep):
    f = np.ascontiguousarray(frames)
    if not on_device:
        keep.append(f)
        return f.ctypes.data
    import torch
    t = torch.from_numpy(f).cuda()
    keep.append(t)
    return t.data_ptr()


def _set_inputs(m, ptr, B, W, H, on_device):
    """fpm_match_set_batch with m's capacity: ([frame][template] records, [frame][template] totals)"""
    T, cap = m.patternSetSize(), m.result_capacity
    res, counts = m.matchSetBatchRaw(ptr, B, W, H, W, H * W, on_device)
    lists = [[[res[(b * T + t) * cap + i] for i in range(min(counts[b * T + t], cap))] for t in range(T)] for b in range(B)]
    return lists, [list(counts[b * T:(b + 1) * T]) for b in range(B)]


def _merged(m, ptr, B, W, H, on_device, max_overlap):
    """fpm_match_set_batch_merged: ([frame][(label, record bytes)], counts, [frame][template] set counts)"""
    T, cap = m.patternSetSize(), m.result_capacity
    res, labels, counts, sc = m.matchSetBatchMergedRaw(ptr, B, W, H, W, H * W, on_device, max_overlap)
    got = [[(labels[b * cap + k], bytes(res[b * cap + k])) for k in range(min(counts[b], cap))] for b in range(B)]
    return got, list(counts), [list(sc[b * T:(b + 1) * T]) for b in range(B)]


def _check_merge(m, frames, overlaps, on_device=(False, True)):
    """every frame, overlap and source residency against merge_reference; returns {(dev, overlap): (got, counts)}"""
    B, H, W = frames.shape
    cap = m.result_capacity
    keep, out = [], {}
    for dev in on_device:
        ptr = _device_ptr(frames, dev, keep)
        lists, totals = _set_inputs(m, ptr, B, W, H, dev)
        for ov in overlaps:
            got, counts, sc = _merged(m, ptr, B, W, H, dev, ov)
            for b in range(B):
                ref = merge_reference(lists[b], ov)
                want = [(t, bytes(r)) for t, r in ref[:cap]]
                if counts[b] != len(ref) or got[b] != want:
                    pytest.fail("frame %d, overlap %r, device %r: %d kept vs %d in the reference; knife-edge pairs %r" %
                                (b, ov, dev, counts[b], len(ref), _knife_edges(lists[b], ov)))
                assert sc[b] == totals[b]
            out[(dev, ov)] = (got, counts, lists)
    return out


# ---- M12: the reference's OCR test at Score 0.7 ----------------------------------------------------------------------
def test_m12_merged_read_at_a_lower_score(ocr_case):
    from fastest_image_pattern_matching_b200 import GlyphReader
    params = dict(ocr_case["params"], score=0.7)
    src = get_image(ocr_case["src"])
    H, W = src.shape
    reader = GlyphReader({ch: g for ch, g in zip(O.OCR_LETTERS, _glyphs())}, **params)
    m = _matcher(params, cap=256)
    m.learnPatternSet(_glyphs())
    keep = []
    ptr = _device_ptr(src[None], True, keep)
    lists, totals = _set_inputs(m, ptr, 1, W, H, True)
    assert sum(totals[0]) == 158
    for ov, n_kept in ((0.3, 89), (0.0, 83)):
        got, counts, _ = _merged(m, ptr, 1, W, H, True, ov)
        assert counts[0] == n_kept
        assert got[0] == [(t, bytes(r)) for t, r in merge_reference(lists[0], ov)]
    assert reader.readBatch(src[None])[0][0] != KNOWN_TEXT
    frames = np.concatenate([src[None], _variants(src, 15, 11)])
    batch = reader.readBatch(frames, merge_overlap=0.3)
    assert batch[0][0] == KNOWN_TEXT
    assert sum(len(v) for v in batch[0][1].values()) == 89
    ptr = _device_ptr(frames, True, keep)
    lists, _ = _set_inputs(m, ptr, len(frames), W, H, True)
    for b, (text, per) in enumerate(batch):
        ref = merge_reference(lists[b], 0.3)
        for t, ch in enumerate(reader.letters):
            want = [(r.score, r.angle, r.cx, r.cy, r.ltx, r.lty, r.rtx, r.rty, r.rbx, r.rby, r.lbx, r.lby) for tt, r in ref if tt == t]
            assert _rows(per[ch]) == want, (b, ch)
    m.close()


# ---- the rotation set: mixed groups, both border colours, a flat template, the same template twice -------------------
@pytest.mark.parametrize("batch", [1, 3, 16])
@pytest.mark.parametrize("async_descent", [0, 1])
def test_rotation_set_merges_like_the_reference(batch, async_descent):
    tpls = _rotation_set()
    frames = _scenes(tpls, batch, w=360, h=280, seed=20 + batch)
    m = _matcher(ROT, {"setAsyncDescent": async_descent})
    m.learnPatternSet(tpls)
    out = _check_merge(m, frames, (0.0, 0.3, 1.0))
    saw_copy = False
    for (dev, ov), (got, counts, lists) in out.items():
        for b in range(batch):
            if [bytes(r) for r in lists[b][0]] == [bytes(r) for r in lists[b][2]]:
                saw_copy = saw_copy or len(lists[b][0]) > 0
                assert all(t != 2 for t, _ in got[b]), (dev, ov, b)      # the copy of template 0 never survives it
    assert saw_copy or batch == 1                         # one scene may lack template 0
    m.close()


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
    m = _matcher(params, extra)
    m.learnPatternSet(tpls)
    _check_merge(m, frames, (0.3,), on_device=(True,))
    # a set of one merges to exactly its own list
    one = _matcher(params, extra)
    one.learnPatternSet(tpls[:1])
    B, H, W = frames.shape
    keep = []
    ptr = _device_ptr(frames, True, keep)
    lists, totals = _set_inputs(one, ptr, B, W, H, True)
    got, counts, sc = _merged(one, ptr, B, W, H, True, 0.0)
    assert sum(counts) > 0
    for b in range(B):
        assert counts[b] == totals[b][0] and sc[b] == totals[b]
        assert got[b] == [(0, bytes(r)) for r in lists[b][0]]
    m.close(); one.close()


# ---- capacity ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cap", [1, 3])
def test_capacity_truncates_inputs_and_output(cap):
    tpls = _rotation_set()
    frames = _scenes(tpls, 3, seed=7)
    m = _matcher(ROT, cap=cap)
    m.learnPatternSet(tpls)
    out = _check_merge(m, frames, (0.3,))
    counts = out[(True, 0.3)][1]
    assert max(counts) > cap
    big = _matcher(ROT)
    big.learnPatternSet(tpls)
    B, H, W = frames.shape
    keep = []
    ptr = _device_ptr(frames, True, keep)
    _, totals = _set_inputs(big, ptr, B, W, H, True)
    _, _, sc = _merged(m, ptr, B, W, H, True, 0.3)
    assert sc == totals and any(t > cap for row in totals for t in row)
    m.close(); big.close()


def test_capacity_zero_writes_counts_only():
    tpls = _rotation_set()
    frames = np.ascontiguousarray(_scenes(tpls, 2, seed=8))
    m = _matcher(ROT)
    m.learnPatternSet(tpls)
    B, H, W = frames.shape
    T = len(tpls)
    _, totals = _set_inputs(m, frames.ctypes.data, B, W, H, False)
    counts = (C.c_int * B)(*([-1] * B))
    sc = (C.c_int * (B * T))()
    rc = m._lib.fpm_match_set_batch_merged(m._h, frames.ctypes.data, 0, B, W, H, W, H * W, 0.3, None, None, 0, counts, sc)
    assert rc == 0
    assert list(counts) == [0] * B                             # no input entries survive a capacity of 0
    assert [list(sc[b * T:(b + 1) * T]) for b in range(B)] == totals and sum(map(sum, totals)) > 0
    m.close()


# ---- large merges: the serial NMS above 512 entries and sort keys in global memory above 1024 ------------------------
def test_large_merges():
    # MaxPos 4 on the 53-angle schedule of a 16x16 top layer: no template's list exceeds 53 * (4 + 5) = 477 entries, so the
    # first prefix of the set beyond 512 (1024) merged entries holds at most 1024 (1535)
    tpls = [_tpl(16, 16, 300 + k) for k in range(48)]
    rng = np.random.default_rng(3)
    frame = synth.background(256, 224, 77)
    for t in tpls:
        synth.paste_rotated(frame, t, float(rng.uniform(20, 236)), float(rng.uniform(20, 204)), float(rng.uniform(-180, 180)))
    H, W = frame.shape
    for score in (0.7, 0.6, 0.5, 0.4):
        params = {"max_pos": 4, "score": score, "tolerance_angle": 180, "max_overlap": 0.9}
        m = _matcher(params, cap=1024)
        m.learnPatternSet(tpls)
        _, totals = _set_inputs(m, frame.ctypes.data, 1, W, H, False)
        m.close()
        if sum(totals[0]) > 1100:
            break
    per = totals[0]
    assert sum(per) > 1100 and max(per) < 512, per
    prefix = np.cumsum(per)
    for lo, hi in ((513, 1024), (1025, 1535)):
        k = int(np.argmax(prefix >= lo)) + 1
        m = _matcher(params, cap=1024)
        m.learnPatternSet(tpls[:k])
        out = _check_merge(m, frame[None], (0.0, 0.5), on_device=(False,))
        n_in = sum(len(x) for x in out[(False, 0.0)][2][0])
        assert lo <= n_in <= hi, (k, n_in)
        m.close()


# ---- ingested JPEG batch ---------------------------------------------------------------------------------------------
def test_ingested_merged_equals_merged(ocr_case):
    src = get_image(ocr_case["src"])
    frames = _variants(src, 4, 7)
    files = [cv2.imencode(".jpg", f, [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes() for f in frames]
    m = _matcher(dict(ocr_case["params"], score=0.7))
    m.learnPatternSet(_glyphs())
    m.ingestJpegBatch(files)
    got = m.matchIngestedSetBatchMerged(0.3)
    decoded = np.stack([m.ingestedFramePixels(i) for i in range(len(files))])
    want = m.matchSetBatchMerged(decoded, 0.3)
    assert [[(t, _rows([r])) for t, r in per] for per in got] == [[(t, _rows([r])) for t, r in per] for per in want]
    assert sum(len(x) for x in got) > 0
    m.close()


# ---- refusals and guards ----------------------------------------------------------------------------------------------
def test_refusals_and_skipped_group(ocr_case):
    from fastest_image_pattern_matching_b200 import FpmError
    from fastest_image_pattern_matching_b200 import _lib as L
    src = get_image(ocr_case["src"])
    H, W = src.shape
    glyphs = _glyphs()[:4]
    big = np.zeros((H + 10, 40), np.uint8)
    big[::3] = 255
    m = _matcher(ocr_case["params"])
    m.learnPatternSet(glyphs + [big])
    for bad in (float("nan"), float("inf"), -float("inf")):
        with pytest.raises(FpmError, match="max_overlap"):
            m.matchSetMerged(src, bad)
    res = (L.fpm_result * 8)()
    n = (C.c_int * 1)()
    assert m._lib.fpm_match_set_batch_merged(m._h, src.ctypes.data, 0, 1, W, H, W, H * W, 0.3, res, None, 8, n, None) == -1
    assert "labels" in m._lib.fpm_last_error(m._h).decode()
    m.setTrace(True)
    with pytest.raises(FpmError, match="TRACE"):
        m.matchSetMerged(src, 0.3)
    m.setTrace(False)
    with pytest.raises(FpmError, match="no ingested frame"):
        m.matchIngestedSetBatchMerged(0.3)
    # the big template's group is skipped by the guards: nothing from it, 0 in its set count
    out = _check_merge(m, src[None], (0.3,))
    for (dev, ov), (got, counts, lists) in out.items():
        assert lists[0][4] == [] and counts[0] > 0 and all(t != 4 for t, _ in got[0])
    _, _, sc = _merged(m, src.ctypes.data, 1, W, H, False, 0.3)
    assert sc[0][4] == 0 and sum(sc[0][:4]) > 0
    # nothing learned or an empty source: zero counts
    m.clearPattern()
    assert m.matchSetMerged(src, 0.3) == []
    m.learnPatternSet(glyphs)
    _, _, counts, sc = m.matchSetBatchMergedRaw(0, 1, W, H, W, H * W, False, 0.3)
    assert list(counts) == [0] and list(sc) == [0] * 4
    m.close()


def test_merged_issues_one_launch_more(ocr_case):
    import torch
    src = get_image(ocr_case["src"])
    frames = np.ascontiguousarray(_variants(src, 3, 5))
    B, H, W = frames.shape
    d = torch.from_numpy(frames).cuda()
    m = _matcher(ocr_case["params"])
    m.learnPatternSet(_glyphs())
    m.matchSetBatchRaw(d.data_ptr(), B, W, H, W, H * W, True)
    m.matchSetBatchMergedRaw(d.data_ptr(), B, W, H, W, H * W, True, 0.3)
    n0 = m.launchCount(); m.matchSetBatchRaw(d.data_ptr(), B, W, H, W, H * W, True); plain = m.launchCount() - n0
    n0 = m.launchCount(); m.matchSetBatchMergedRaw(d.data_ptr(), B, W, H, W, H * W, True, 0.3); merged = m.launchCount() - n0
    assert merged == plain + 1, (merged, plain)
    m.close()
