"""Template sets in the angle-sharded latency mode (fpm_match_set_sharded*): one frame against the whole set, the angle
schedule of every group split across the ranks.  Every rank's lists must be bit-identical (ordered, tolerance 0, full
records) to what fpm_match_set_batch / fpm_match_set_batch_merged return for the frame on one GPU.  The virtual-rank calls
let several handles of one GPU play the ranks; the NCCL calls run with a one-rank communicator."""
import ctypes as C
import math

import numpy as np
import pytest

import fpm_workloads as synth
from oracle import oracle as O
from tests.helpers import configure, get_image
from tests.test_gpu_template_set import ROT, _glyphs, _matcher, _rotation_set, _rows, _scenes, _tpl
from tests.test_ocr import KNOWN_TEXT

pytestmark = pytest.mark.gpu


def _merged_rows(lst):
    return [(t,) + _rows([r])[0] for t, r in lst]


def _ranks(world, params, tpls, extra=None, cap=512):
    hs = [_matcher(params, extra, cap) for _ in range(world)]
    for m in hs:
        m.learnPatternSet(tpls)
    return hs


def _close(ms):
    for m in ms:
        m.close()


def _check_virtual(hs, src, want, want_merged, calls=1):
    """every rank == the single-GPU lists; each virtual call adds exactly two exchange rounds to every handle's count"""
    from fastest_image_pattern_matching_b200.matcher import match_set_sharded_virtual
    for _ in range(calls):
        before = [m.collectiveCount() for m in hs]
        per_rank = match_set_sharded_virtual(hs, src)
        assert [m.collectiveCount() - b for m, b in zip(hs, before)] == [2] * len(hs)
        assert len(per_rank) == len(hs)
        for r, got in enumerate(per_rank):
            assert [_rows(x) for x in got] == [_rows(x) for x in want], r
        for ov, wm in want_merged.items():
            before = [m.collectiveCount() for m in hs]
            for r, got in enumerate(match_set_sharded_virtual(hs, src, max_overlap=ov)):
                assert _merged_rows(got) == _merged_rows(wm), (r, ov)
            assert [m.collectiveCount() - b for m, b in zip(hs, before)] == [2] * len(hs)


# ---- M12: 36 glyphs in several groups, tolerance 0 (one angle: more ranks than angles) ---------------------------
@pytest.fixture(scope="module")
def ocr_case():
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cases.json")) as f:
        return json.load(f)["ocr_m12"]


def _text(merged):
    from fastest_image_pattern_matching_b200.matcher import ocr_assemble
    return ocr_assemble([r.ptCenter for _, r in merged], [O.OCR_LETTERS[t] for t, _ in merged])


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_m12_virtual_ranks(ocr_case, world):
    src = get_image(ocr_case["src"])
    params = dict(ocr_case["params"], score=0.7)             # 0.7: look-alike glyphs hit the same cells, the merge matters
    ref = _matcher(params)
    ref.learnPatternSet(_glyphs())
    want = ref.matchSet(src)
    want_merged = {ov: ref.matchSetMerged(src, ov) for ov in (0.0, 0.3)}
    ref.close()
    assert sum(len(x) for x in want) > 0
    assert _text(want_merged[0.3]) == KNOWN_TEXT
    hs = _ranks(world, params, _glyphs())
    try:
        _check_virtual(hs, src, want, want_merged)
    finally:
        _close(hs)


# ---- the +-180 degree rotation set: several groups, a flat template, both border colours, a duplicate, tall ROIs ---
@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_rotation_set_virtual_ranks(world):
    tpls = _rotation_set()
    frames = _scenes(tpls, 2, seed=21 + world)
    ref = _matcher(ROT)
    ref.learnPatternSet(tpls)
    hs = _ranks(world, ROT, tpls)
    try:
        for f in frames:
            want = ref.matchSet(f)
            assert _rows(want[0]) == _rows(want[2])
            _check_virtual(hs, f, want, {0.3: ref.matchSetMerged(f, 0.3)}, calls=2)   # second call: cached plans and buffers
        assert sum(len(x) for x in want) > 0
        # a handle that has just played a rank still sweeps the whole schedule
        assert [_rows(x) for x in hs[-1].matchSet(frames[-1])] == [_rows(x) for x in want]
    finally:
        _close(hs + [ref])


@pytest.mark.parametrize("variant", ["subpixel", "mfc", "stop_layer1", "bitwise_not", "tol_range", "no_simd", "small_workspace"])
def test_parameter_variants_world3(variant):
    tpls = _rotation_set()
    f = _scenes(tpls, 1, seed=40)[0]
    params, extra = dict(ROT), {}
    if variant == "subpixel":
        params["sub_pixel"] = True
    elif variant == "mfc":
        extra["setMfcCompat"] = True
    elif variant == "stop_layer1":
        extra["setStopLayer1"] = True
    elif variant == "bitwise_not":
        extra["setBitwiseNot"] = True
    elif variant == "tol_range":
        extra["setToleranceRange"] = (-90, 30, 60, 150)
    elif variant == "no_simd":
        params["use_simd"] = False
    elif variant == "small_workspace":
        extra["setWorkspaceMB"] = 0.25
    ref = _matcher(params, extra)
    ref.learnPatternSet(tpls)
    hs = _ranks(3, params, tpls, extra)
    try:
        _check_virtual(hs, f, ref.matchSet(f), {0.3: ref.matchSetMerged(f, 0.3)})
    finally:
        _close(hs + [ref])


# ---- edge cases ---------------------------------------------------------------------------------------------------
def test_nothing_found_and_small_sources():
    from fastest_image_pattern_matching_b200.matcher import match_set_sharded_virtual
    tpls = _rotation_set()
    plain = [t for i, t in enumerate(tpls) if i != 6]        # a flat template scores 1 wherever its NCC is degenerate
    f = synth.background(420, 300, 50)                      # nothing planted
    ref = _matcher(dict(ROT, score=0.999))
    ref.learnPatternSet(plain)
    hs = _ranks(3, dict(ROT, score=0.999), plain)
    try:
        want = ref.matchSet(f)
        assert all(x == [] for x in want)
        _check_virtual(hs, f, want, {0.3: []})
    finally:
        _close(hs + [ref])
    # 100 x 100: the 40 x 130 group does not fit (its lists are empty), the others run; 8 x 8: nothing fits
    ref = _matcher(ROT)
    ref.learnPatternSet(tpls)
    hs = _ranks(3, ROT, tpls)
    try:
        small = np.ascontiguousarray(_scenes(tpls[5:6], 1, w=100, h=100, seed=51)[0])
        want = ref.matchSet(small)
        assert want[8] == [] and want[9] == []
        _check_virtual(hs, small, want, {0.3: ref.matchSetMerged(small, 0.3)})
        tiny = np.zeros((8, 8), np.uint8)
        per_rank = match_set_sharded_virtual(hs, tiny)
        assert all(all(x == [] for x in got) for got in per_rank)
        assert all(got == [] for got in match_set_sharded_virtual(hs, tiny, max_overlap=0.3))
    finally:
        _close(hs + [ref])


@pytest.mark.parametrize("cap", [0, 1])
def test_small_capacity_keeps_totals(cap):
    from fastest_image_pattern_matching_b200 import _lib as L
    tpls = _rotation_set()
    f = np.ascontiguousarray(_scenes(tpls, 1, seed=60)[0])
    T, world = len(tpls), 3
    ref = _matcher(ROT, cap=cap)
    ref.learnPatternSet(tpls)
    res, counts = ref.matchSetBatchRaw(f.ctypes.data, 1, f.shape[1], f.shape[0], f.shape[1], f.size, False)
    want_counts = list(counts)
    _, _, mcount, mset = ref.matchSetBatchMergedRaw(f.ctypes.data, 1, f.shape[1], f.shape[0], f.shape[1], f.size, False, 0.3)
    assert sum(want_counts) > world
    hs = _ranks(world, ROT, tpls, cap=cap)
    try:
        lib = hs[0]._lib
        arr = (C.c_void_p * world)(*[m._h for m in hs])
        out = (L.fpm_result * max(cap * world * T, 1))()
        cnt = (C.c_int * (world * T))()
        assert lib.fpm_match_set_sharded_virtual(arr, world, f.ctypes.data, f.shape[1], f.shape[0], f.shape[1], out, cap, cnt) == 0
        for r in range(world):
            assert list(cnt[r * T:(r + 1) * T]) == want_counts
            if cap:
                assert _rows(_conv(out, r * T * cap, T * cap)) == _rows(_conv(res, 0, T * cap))
        labels = (C.c_int * max(cap * world, 1))()
        mc = (C.c_int * world)()
        ms = (C.c_int * (world * T))()
        out = (L.fpm_result * max(cap * world, 1))()
        assert lib.fpm_match_set_sharded_merged_virtual(arr, world, f.ctypes.data, f.shape[1], f.shape[0], f.shape[1], 0.3, out,
                                                        labels if cap else None, cap, mc, ms) == 0
        for r in range(world):
            assert mc[r] == mcount[0] and list(ms[r * T:(r + 1) * T]) == list(mset)
    finally:
        _close(hs + [ref])


def _conv(arr, start, n):
    from fastest_image_pattern_matching_b200.matcher import _convert
    return _convert(arr[start:start + n], n)


# ---- one large case: 8192^2 frame, four 1024^2 templates at +-180 degrees, eight ranks -----------------------------
def test_large_frame_world8():
    tpls = [synth.synth_template(1024, 4 + k) for k in range(4)]
    f = synth.background(8192, 8192, 11, 3.0)
    for t, (cx, cy, a) in zip(tpls, [(2000, 2000, 30.0), (6100, 2000, -100.0), (2000, 6100, 150.0), (6100, 6100, -20.0)]):
        synth.paste_rotated(f, t, float(cx), float(cy), a, fast=True)
    params = dict(max_pos=4, score=0.8, tolerance_angle=180, min_reduce_area=256, max_overlap=0.0)
    ref = _matcher(params)
    ref.learnPatternSet(tpls)
    want = ref.matchSet(f)
    assert all(len(x) >= 1 for x in want)                 # the templates share a circle and a bar: each may hit the others too
    hs = _ranks(8, params, tpls)
    try:
        _check_virtual(hs, f, want, {0.3: ref.matchSetMerged(f, 0.3)})
    finally:
        _close(hs + [ref])


# ---- a set of one: the new calls equal fpm_match_sharded_virtual -------------------------------------------------
def test_set_of_one_equals_match_sharded_virtual():
    from fastest_image_pattern_matching_b200.matcher import match_set_sharded_virtual, match_sharded_virtual
    tpl = _tpl(48, 40, 3)
    src = _scenes([tpl, tpl, tpl], 1, w=360, h=280, seed=70)[0]
    params = dict(max_pos=5, score=0.6, tolerance_angle=180, max_overlap=0.3)
    hs = [_matcher(params) for _ in range(4)]
    for m in hs:
        m.learnPattern(tpl)
    try:
        before = [m.collectiveCount() for m in hs]
        old = match_sharded_virtual(hs, src)
        assert [m.collectiveCount() for m in hs] == before      # the one-template call does not count its block copies
        new = match_set_sharded_virtual(hs, src)
        merged = match_set_sharded_virtual(hs, src, max_overlap=0.3)
        assert len(old[0]) > 0
        for r in range(4):
            assert _rows(new[r][0]) == _rows(old[r])
            assert _merged_rows(merged[r]) == [(0,) + x for x in _rows(old[r])]
    finally:
        _close(hs)


# ---- NCCL with one rank: host and device frames ------------------------------------------------------------------
def test_nccl_single_rank(ocr_case):
    import torch
    from fastest_image_pattern_matching_b200.matcher import comm_available, comm_unique_id
    assert comm_available()
    tpls = _rotation_set()
    f = np.ascontiguousarray(_scenes(tpls, 1, seed=80)[0])
    m = _matcher(ROT)
    m.learnPatternSet(tpls)
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
        # M12 on the same communicator
        src = get_image(ocr_case["src"])
        params = dict(ocr_case["params"], score=0.7)
        g = _matcher(params)
        g.learnPatternSet(_glyphs())
        want12, want12_m = g.matchSet(src), g.matchSetMerged(src, 0.3)
        g.close()
        configure(m, params)
        m.learnPatternSet(_glyphs())
        assert [_rows(x) for x in m.matchSetSharded(src)] == [_rows(x) for x in want12]
        assert _merged_rows(m.matchSetShardedMerged(src, 0.3)) == _merged_rows(want12_m)
    finally:
        m.commDestroy()
        m.close()


# ---- refusals ----------------------------------------------------------------------------------------------------
def test_refusals():
    from fastest_image_pattern_matching_b200 import FpmError, TemplateMatcher
    from fastest_image_pattern_matching_b200 import _lib as L
    from fastest_image_pattern_matching_b200.matcher import comm_unique_id, match_set_sharded_virtual
    tpls = _rotation_set()[:5]
    f = np.ascontiguousarray(_scenes(tpls, 1, w=200, h=160, seed=90)[0])
    m = _matcher(ROT)
    m.learnPatternSet(tpls)
    m.setTrace(True)
    with pytest.raises(FpmError, match="TRACE"):
        m.matchSetSharded(f)
    with pytest.raises(FpmError, match="TRACE"):
        m.matchSetShardedMerged(f, 0.3)
    m.setTrace(False)
    for bad in (float("nan"), float("inf"), -math.inf):
        with pytest.raises(FpmError, match="max_overlap"):
            m.matchSetShardedMerged(f, bad)
    lib, h = m._lib, m._h
    out = (L.fpm_result * 64)()
    cnt = (C.c_int * 8)()
    assert lib.fpm_match_set_sharded(h, f.ctypes.data, f.shape[1], f.shape[0], f.shape[1], 0, out, 8, None) == L_ERR_INVALID
    assert lib.fpm_match_set_sharded(h, f.ctypes.data, f.shape[1], f.shape[0], f.shape[1], 0, None, 8, cnt) == L_ERR_INVALID
    assert lib.fpm_match_set_sharded_merged(h, f.ctypes.data, f.shape[1], f.shape[0], f.shape[1], 0, 0.3, out, None, 8, cnt,
                                            None) == L_ERR_INVALID
    assert "labels" in lib.fpm_last_error(h).decode()
    # the single-template sharded call still refuses a set
    n = C.c_int()
    assert lib.fpm_match_sharded(h, f.ctypes.data, f.shape[1], f.shape[0], f.shape[1], 0, out, 8, C.byref(n)) == L_ERR_INVALID
    # virtual ranks: set sizes differ (the message names the rank), a handle with a communicator
    other = _matcher(ROT)
    other.learnPatternSet(tpls[:3])
    with pytest.raises(FpmError, match="rank 1"):
        match_set_sharded_virtual([m, other], f)
    with pytest.raises(FpmError, match="rank 1"):
        match_set_sharded_virtual([m, other], f, max_overlap=0.3)
    other.learnPatternSet(tpls)
    other.commInit(1, 0, comm_unique_id())
    with pytest.raises(FpmError, match="communicator"):
        match_set_sharded_virtual([m, other], f)
    other.commDestroy()
    assert len(match_set_sharded_virtual([m, other], f)) == 2
    # nothing learned: empty lists
    empty = TemplateMatcher(0, result_capacity=16)
    assert empty.matchSetSharded(f) == [[]]
    assert empty.matchSetShardedMerged(f, 0.3) == []
    _close([m, other, empty])


L_ERR_INVALID = -1
