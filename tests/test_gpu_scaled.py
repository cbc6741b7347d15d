"""Scale-tolerant matching on the GPU (FPM_PARAM_SCALE_MIN / MAX) against tests/scaled_oracle.py.

- [1, 1] set explicitly, also after other ranges on the same handle, and fpm_match_scaled at [1, 1] are bit-identical to a fresh
  handle's fpm_match_batch(_device) (the plan cache); every scale returned is exactly 1.0.
- Scale ranges and fixed scales 0.5 .. 2 on seeded scenes match ScaledOracleMatcher in tensor-core modes 0-4 (and 6), with the
  scales equal to the oracle's doubles; every eval's 7x7 scores equal the oracle's bit for bit under FPM_PARAM_TRACE.
- On a cfg1-size frame [0.8, 1.25] finds instances at 0.85, 1.0 and 1.2, and [1, 1] only the one at 1.0.
- Host, pinned, device and split batches, async descent on and off and ingested frames equal per-frame fpm_match; a masked
  template, sub-pixel, MFC compat, stop layer 1, bitwise-not and the tolerance range match the oracle.
- fpm_dbg_warp_affine reproduces cv2.warpAffine for getRotationMatrix2D(c, angle, 1/s), tiles beyond the staged box included.
- Refusals: values out of [0.5, 2] or NaN (a refused setScaleRange leaves the range unchanged), min > max, sets of more than
  one template, the angle-sharded calls and fpm_stage_* at any range other than [1, 1].
"""
import ctypes as C
import math

import cv2
import numpy as np
import pytest

from fastest_image_pattern_matching_b200 import FpmError, TemplateMatcher
from fastest_image_pattern_matching_b200 import _lib as L
from tests.helpers import assert_results_match, configure, get_image
from tests.masked_oracle import MaskedOracleMatcher, disc_mask
from tests.scaled_oracle import ScaledOracleMatcher, scaled_scene

pytestmark = pytest.mark.gpu

GOLDEN = ["src8", "src9", "test4_src3", "src4", "src9_subpix", "cfg3_src6"]
PARAMS = dict(max_pos=10, score=0.8, tolerance_angle=25, max_overlap=0.2)


def _key(r):
    return (r.dMatchScore, r.dMatchedAngle, r.ptCenter, r.ptLT, r.ptRT, r.ptRB, r.ptLB)


def _scene(s, seed=31):
    """640 x 480 frame with two instances of a 96 x 72 template at scale s (plus one at scale 1 when s != 1)"""
    poses = [(170.0, 140.0, 11.0, s), (450.0, 330.0, -17.0, s)]
    if s != 1.0:
        poses.append((470.0, 110.0, 4.0, 1.0) if s < 1.2 else (130.0, 400.0, 4.0, 1.0))
    if s >= 1.5:                       # the instances grow: keep them apart and inside the frame
        poses = [(190.0, 160.0, 11.0, s), (460.0, 330.0, -17.0, s)]
    return scaled_scene(640, 480, 96, 72, poses, seed)


class ScaledMaskedOracle(ScaledOracleMatcher, MaskedOracleMatcher):
    pass


def _oracle(params, s, tpl, mask=None, **extra):
    om = configure(ScaledMaskedOracle() if mask is not None else ScaledOracleMatcher(), params)
    om.scale_min, om.scale_max = s if isinstance(s, tuple) else (s, s)
    for k, v in extra.items():
        setattr(om, k, v)
    assert om.learn_pattern(tpl, mask) if mask is not None else om.learn_pattern(tpl)
    return om


@pytest.fixture(scope="module")
def gm(fpm_built):
    m = TemplateMatcher(0)
    yield m
    m.close()


def _gpu(m, params, s, tpl, mode=1, mask=None):
    configure(m, params)
    m.setTensorCores(mode)
    m.setScaleRange(*(s if isinstance(s, tuple) else (s, s)))
    assert m.learnPattern(tpl) if mask is None else m.learnPattern(tpl, mask)
    return m


# ---------------- 1. [1, 1] is the unscaled matcher, also after another scale on the same handle ----------------
@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("name", GOLDEN)
def test_unit_range_bit_identical(gm, golden_cases, name, mode):
    c = golden_cases[name]
    tpl, src, params = get_image(c["tpl"]), get_image(c["src"]), c["params"]
    fresh = TemplateMatcher(0)
    try:
        configure(fresh, params)
        fresh.setTensorCores(mode)
        assert fresh.learnPattern(tpl)
        want = fresh.match(src)
        want_b = fresh.matchBatch(np.stack([src, src]))
    finally:
        fresh.close()
    _gpu(gm, params, 1.25, tpl, mode)
    gm.match(src)                                   # a cached plan at scale 1.25
    gm.setScaleRange(1.0, 1.0)
    assert gm.getScaleRange() == (1.0, 1.0)
    assert [_key(r) for r in gm.match(src)] == [_key(r) for r in want]
    assert [[_key(r) for r in f] for f in gm.matchBatch(np.stack([src, src]))] == [[_key(r) for r in f] for f in want_b]


# ---------------- 2. fixed scales against the oracle ----------------
@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4, 6])
@pytest.mark.parametrize("s", [0.8, 1.25])
def test_fixed_scale_matches_oracle(gm, s, mode):
    tpl, src = _scene(s)
    want = _oracle(PARAMS, s, tpl).match(src)
    assert len(want) >= 2 and all(r.scale == s for r in want)
    got = _gpu(gm, PARAMS, s, tpl, mode).match(src)
    assert_results_match(got, want)


@pytest.mark.parametrize("s", [0.5, 0.7, 1.5, 2.0])
def test_fixed_scale_extremes(gm, s):
    tpl, src = _scene(s, seed=40)
    params = dict(PARAMS, tolerance_angle=20)
    want = _oracle(params, s, tpl).match(src)
    assert len(want) >= 2
    got = _gpu(gm, params, s, tpl).match(src)
    assert_results_match(got, want)
    gm.setScaleRange(1.0, 1.0)
    unscaled = gm.match(src)
    assert len(unscaled) < len(got)


# ---------------- 3. every path equals per-frame fpm_match ----------------
def _device_batch(m, frames):
    import torch
    d = torch.from_numpy(np.ascontiguousarray(frames)).cuda()
    B, H, W = frames.shape
    res, n = m.matchBatchRaw(d.data_ptr(), B, W, H, W, H * W, True)
    from fastest_image_pattern_matching_b200.matcher import _convert
    cap = m.result_capacity
    return [[_key(r) for r in _convert(res[b * cap:(b + 1) * cap], min(n[b], cap))] for b in range(B)]


@pytest.mark.parametrize("async_descent", [0, 1])
def test_paths_equal_per_frame(gm, async_descent):
    s = 0.85
    frames = []
    for k in range(8):
        frames.append(_scene(s, seed=50 + k)[1])
    tpl = _scene(s, seed=50)[0]
    frames = np.stack(frames)
    _gpu(gm, PARAMS, s, tpl)
    gm.setAsyncDescent(async_descent)
    try:
        per = [[_key(r) for r in gm.match(f)] for f in frames]
        assert sum(len(p) for p in per) >= 8
        assert [[_key(r) for r in f] for f in gm.matchBatch(frames)] == per             # pageable host batch
        gm.setSplitBatch(4)
        assert _device_batch(gm, frames) == per                                         # split device batch
        gm.setSplitBatch(0)
        assert _device_batch(gm, frames) == per
        gm.setH2DChunk(3)
        assert [[_key(r) for r in f] for f in gm.matchBatch(frames)] == per             # chunked host batch
    finally:
        gm.setSplitBatch(8)
        gm.setH2DChunk(0)
        gm.setAsyncDescent(-1)


def test_ingested_equal_per_frame(gm):
    s = 1.2
    tpl, src = _scene(s, seed=61)
    _gpu(gm, PARAMS, s, tpl)
    want = [_key(r) for r in gm.match(src)]
    ok, buf = cv2.imencode(".bmp", src)
    gm.ingestImage(buf.tobytes())
    assert [_key(r) for r in gm.matchIngested()] == want
    assert [[_key(r) for r in f] for f in gm.matchIngestedBatch()] == [want]


# ---------------- 4. masked template and the other modes against the oracle ----------------
def test_masked_fixed_scale(gm):
    s = 1.15
    tpl, src = _scene(s, seed=70)
    mask = disc_mask(tpl.shape[1], tpl.shape[0])
    want = _oracle(PARAMS, s, tpl, mask).match(src)
    assert len(want) >= 2
    got = _gpu(gm, PARAMS, s, tpl, 1, mask).match(src)
    assert_results_match(got, want)


@pytest.mark.parametrize("mode", ["sub_pixel", "mfc_compat", "stop_layer1", "bitwise_not", "tolerance_range"])
def test_modes_fixed_scale(gm, mode):
    s = 0.9
    tpl, src = _scene(s, seed=80)
    extra = {}
    if mode == "bitwise_not":
        src = (255 - src).astype(np.uint8)
    if mode == "tolerance_range":
        extra["tolerance_range"] = (-25.0, -5.0, 5.0, 25.0)
    else:
        extra[mode] = True
    want = _oracle(PARAMS, s, tpl, **extra).match(src)
    assert want
    _gpu(gm, PARAMS, s, tpl)
    try:
        if mode == "sub_pixel":
            gm.setSubPixelEstimation(True)
        elif mode == "mfc_compat":
            gm.setMfcCompat(True)
        elif mode == "stop_layer1":
            gm.setStopLayer1(True)
        elif mode == "bitwise_not":
            gm.setBitwiseNot(True)
        else:
            gm.setToleranceRange(extra["tolerance_range"])
        got = gm.match(src)
    finally:
        gm.setSubPixelEstimation(False)
        gm.setMfcCompat(False)
        gm.setStopLayer1(False)
        gm.setBitwiseNot(False)
        gm.setToleranceRange(None)
    assert_results_match(got, want)


# ---------------- 5. the ROI warp at scaled matrices ----------------
@pytest.mark.parametrize("s", [0.5, 0.7, 1.3, 2.0])
def test_warp_affine_scaled_matrix(gm, s):
    rng = np.random.default_rng(int(s * 100))
    src = rng.integers(0, 256, (300, 420), dtype=np.uint8)
    lib = gm._lib
    for ang, (dw, dh) in [(0.0, (140, 70)), (17.0, (200, 150)), (-63.0, (96, 300)), (120.0, (257, 65))]:
        m = cv2.getRotationMatrix2D((209.5, 149.5), ang, 1.0 / s)
        m[0, 2] -= 40.0
        m[1, 2] -= 25.0
        want = cv2.warpAffine(src, m, (dw, dh), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=17)
        got = np.zeros((dh, dw), np.uint8)
        mm = (C.c_double * 6)(*m.ravel().tolist())
        assert lib.fpm_dbg_warp_affine(gm._h, src.ctypes.data, 420, 300, 420, mm, dw, dh, 17, got.ctypes.data) == 0
        assert np.array_equal(got, want), (s, ang, int((got != want).sum()))


# ---------------- 6. refusals ----------------
def test_refusals(fpm_built):
    m = TemplateMatcher(0)
    try:
        for v in (0.49, 2.01, float("nan"), float("inf"), -1.0):
            with pytest.raises(FpmError, match="FPM_PARAM_SCALE_MIN"):
                m.setScaleRange(v, 1.0)
            with pytest.raises(FpmError, match="FPM_PARAM_SCALE_MAX"):
                m.setScaleRange(1.0, v)
        assert m.getScaleRange() == (1.0, 1.0)
        tpl, src = _scene(1.0, seed=90)
        assert m.learnPattern(tpl)
        m.setScaleRange(1.2, 1.1)
        with pytest.raises(FpmError, match="FPM_PARAM_SCALE_MIN .* > FPM_PARAM_SCALE_MAX"):
            m.match(src)
        m.setScaleRange(0.9, 1.1)
        with pytest.raises(FpmError):
            m.setScaleRange(0.95, 2.5)
        assert m.getScaleRange() == (0.9, 1.1)
        assert m.match(src)
        res = (L.fpm_result * 16)()
        n = C.c_int(0)
        assert m._lib.fpm_match_sharded(m._h, src.ctypes.data, 640, 480, 640, 0, res, 16, C.byref(n)) == L_ERR
        assert "fpm_match_sharded" in m._lib.fpm_last_error(m._h).decode()
        picks = np.zeros(64, np.float64)
        assert m._lib.fpm_stage_top(m._h, src.ctypes.data, 640, 480, 640, 0, 0, -1, picks.ctypes.data, 16, C.byref(n)) == L_ERR
        assert "fpm_stage_top" in m._lib.fpm_last_error(m._h).decode()
        assert m.match(src) is not None                                 # the handle keeps working
        assert m.learnPatternSet([tpl, tpl[:60, :80].copy()])
        with pytest.raises(FpmError, match="fpm_match_set_batch"):
            m.matchSet(src)
        m.setScaleRange(1.0, 1.0)
        assert len(m.matchSet(src)) == 2
    finally:
        m.close()


L_ERR = -1


# ---------------- 7. scale ranges ----------------
_RANGE_WANT = {}
RANGE_POSES = [(150.0, 130.0, 12.0, 0.8), (440.0, 150.0, -20.0, 1.0), (300.0, 350.0, 7.0, 1.25)]


def _range_scene(seed=21):
    return scaled_scene(640, 480, 96, 72, RANGE_POSES, seed)


def _scaled_call(m, frames, on_device):
    """fpm_match_scaled: [(key, scale)] per frame"""
    f = np.ascontiguousarray(frames)
    B, H, W = f.shape
    cap = m.result_capacity
    res = (L.fpm_result * (cap * B))()
    sc = (C.c_double * (cap * B))()
    n = (C.c_int * B)()
    keep = None
    if on_device:
        import torch
        keep = torch.from_numpy(f).cuda()
        ptr = keep.data_ptr()
    else:
        ptr = f.ctypes.data
    assert m._lib.fpm_match_scaled(m._h, ptr, int(on_device), B, W, H, W, H * W, res, sc, cap, n) == 0, \
        m._lib.fpm_last_error(m._h).decode()
    from fastest_image_pattern_matching_b200.matcher import _convert
    return [[(_key(r), r.dScale) for r in _convert(res[b * cap:(b + 1) * cap], min(n[b], cap), sc[b * cap:(b + 1) * cap])]
            for b in range(B)]


@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("name", GOLDEN)
def test_match_scaled_unit_range_bit_identical(gm, golden_cases, name, mode):
    c = golden_cases[name]
    tpl, src, params = get_image(c["tpl"]), get_image(c["src"]), c["params"]
    _gpu(gm, params, (0.9, 1.1), tpl, mode)
    gm.match(src)                                   # a cached plan of another range
    gm.setScaleRange(1.0, 1.0)
    frames = np.stack([src, src])
    want = [[_key(r) for r in f] for f in gm.matchBatch(frames)]
    res = (L.fpm_result * (gm.result_capacity * 2))()
    n = (C.c_int * 2)()
    assert gm._lib.fpm_match_batch(gm._h, frames.ctypes.data, 2, src.shape[1], src.shape[0], src.shape[1],
                                   src.shape[0] * src.shape[1], res, gm.result_capacity, n) == 0
    from fastest_image_pattern_matching_b200.matcher import _convert
    plain = [[_key(r) for r in _convert(res[b * gm.result_capacity:], min(n[b], gm.result_capacity))] for b in range(2)]
    assert plain == want
    for on_device in (False, True):
        got = _scaled_call(gm, frames, on_device)
        assert [[k for k, _ in f] for f in got] == want
        assert all(s == 1.0 for f in got for _, s in f)


@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("rng", [(0.8, 1.25), (0.9, 1.1), (0.75, 0.75)])
def test_range_matches_oracle(gm, rng, mode):
    tpl, src = _range_scene()
    if rng not in _RANGE_WANT:                                       # the oracle runs on the CPU: once per range
        _RANGE_WANT[rng] = _oracle(PARAMS, rng, tpl).match(src)
    want = _RANGE_WANT[rng]
    assert want
    _gpu(gm, PARAMS, rng, tpl, mode)
    got = _scaled_call(gm, src[None], False)[0]
    assert_results_match([r for r in gm.match(src)], want)
    assert [s for _, s in got] == [r.scale for r in want]          # the oracle's doubles, exactly
    assert [r.dScale for r in gm.match(src)] == [r.scale for r in want]


def test_range_finds_every_size(gm):
    tpl, src = _range_scene()
    _gpu(gm, PARAMS, (0.8, 1.25), tpl)
    got = gm.match(src)
    assert len(got) == 3
    for cx, cy, a, s in RANGE_POSES:
        assert any(math.hypot(r.ptCenter[0] - cx, r.ptCenter[1] - cy) <= 1.0 and abs(r.dMatchedAngle + a) <= 1.2 and
                   abs(r.dScale / s - 1) <= 2.0 / 96 for r in got), (cx, cy, a, s)
    gm.setScaleRange(1.0, 1.0)
    assert len(gm.match(src)) == 1


@pytest.mark.parametrize("mode", [0, 1, 4])
def test_range_eval_cells_match_oracle(gm, mode):
    tpl, src = _range_scene()
    params = dict(PARAMS, max_pos=3)
    om = _oracle(params, (0.8, 1.25), tpl)
    om.trace = {}
    om.match(src)
    want = {}
    for e in om.trace["refine"]:
        want[(e["layer"], e["cand"], e["j"])] = (e["scale"], e["score"].astype(np.float32))
    _gpu(gm, params, (0.8, 1.25), tpl, mode)
    gm.setTrace(True)
    try:
        gm.match(src)
        got = {}
        for layer in range(len(gm.templateLevels()) - 1):
            rows, scores = gm.traceEvals(layer), gm.traceEvalScores(layer)
            seen = {}
            for i, r in enumerate(rows):
                cid = int(r[0])
                j = seen.get(cid, 0)
                seen[cid] = j + 1
                got[(layer, cid, j)] = scores[i].reshape(7, 7)
    finally:
        gm.setTrace(False)
    assert set(got) == set(want) and len(want) > 9
    assert max(j for (_, _, j) in want) == 8                         # 3 scales x 3 angles per candidate
    bad = [k for k in sorted(want) if not np.array_equal(got[k], want[k][1])]
    assert not bad, (len(bad), bad[:5])


def test_range_paths_equal_per_frame(gm):
    import fpm_workloads as synth
    from tests.scaled_oracle import paste_scaled
    tpl = _range_scene()[0]
    frames = []
    for k in range(8):                                               # one template, its three sizes moved about per frame
        f = synth.background(640, 480, 200 + k, 3.0)
        for cx, cy, a, s in RANGE_POSES:
            paste_scaled(f, tpl, cx + 3 * k, cy - 2 * k, a + 5 * k, s)
        frames.append(f)
    frames = np.stack(frames)
    _gpu(gm, PARAMS, (0.8, 1.25), tpl)
    per = [[(_key(r), r.dScale) for r in gm.match(f)] for f in frames]
    assert sum(len(p) for p in per) >= 16
    try:
        for ad in (0, 1):
            gm.setAsyncDescent(ad)
            assert _scaled_call(gm, frames, False) == per
            gm.setSplitBatch(4)
            assert _scaled_call(gm, frames, True) == per                # split device batch
            gm.setSplitBatch(0)
            assert _scaled_call(gm, frames, True) == per
    finally:
        gm.setSplitBatch(8)
        gm.setAsyncDescent(-1)
    ok, buf = cv2.imencode(".bmp", frames[0])
    gm.ingestImage(buf.tobytes())
    assert [(_key(r), r.dScale) for r in gm.matchIngested()] == per[0]


@pytest.mark.parametrize("mode", ["sub_pixel", "mfc_compat", "stop_layer1", "masked"])
def test_range_modes_match_oracle(gm, mode):
    tpl, src = _range_scene()
    rng = (0.8, 1.25)
    mask = disc_mask(tpl.shape[1], tpl.shape[0]) if mode == "masked" else None
    extra = {} if mode == "masked" else {mode: True}
    want = _oracle(PARAMS, rng, tpl, mask, **extra).match(src)
    assert want
    _gpu(gm, PARAMS, rng, tpl, 1, mask)
    try:
        gm.setSubPixelEstimation(mode == "sub_pixel")
        gm.setMfcCompat(mode == "mfc_compat")
        gm.setStopLayer1(mode == "stop_layer1")
        got = gm.match(src)
    finally:
        gm.setSubPixelEstimation(False)
        gm.setMfcCompat(False)
        gm.setStopLayer1(False)
    assert_results_match(got, want)
    assert [r.dScale for r in got] == [r.scale for r in want]


def test_plan_cache_across_ranges(gm):
    tpl, src = _range_scene()
    fresh = {}
    for rng in [(0.8, 1.25), (1.0, 1.0), (0.9, 1.1), (1.1, 1.1)]:
        m = TemplateMatcher(0)
        try:
            _gpu(m, PARAMS, rng, tpl)
            fresh[rng] = [(_key(r), r.dScale) for r in m.match(src)]
        finally:
            m.close()
    _gpu(gm, PARAMS, (1.0, 1.0), tpl)
    for rng in [(0.8, 1.25), (1.0, 1.0), (0.9, 1.1), (1.1, 1.1), (0.8, 1.25)]:
        gm.setScaleRange(*rng)
        assert [(_key(r), r.dScale) for r in gm.match(src)] == fresh[rng], rng


def test_cfg1_demonstration(gm):
    import fpm_workloads as synth
    from tests.scaled_oracle import paste_scaled
    tpl = synth.load_fixture("Dst7")
    src = synth.background(4024, 3036, 7, 3.0)
    poses = [(900.0, 800.0, 10.0, 0.85), (2600.0, 900.0, -35.0, 1.0), (1900.0, 2200.0, 120.0, 1.2)]
    for cx, cy, a, s in poses:
        paste_scaled(src, tpl, cx, cy, a, s)
    configure(gm, dict(max_pos=3, score=0.8, tolerance_angle=180))
    gm.setTensorCores(1)
    assert gm.learnPattern(tpl)
    gm.setScaleRange(0.8, 1.25)
    got = gm.match(src)
    assert len(got) == 3, [(r.ptCenter, r.dScale, r.dMatchScore) for r in got]
    for cx, cy, a, s in poses:
        assert any(math.hypot(r.ptCenter[0] - cx, r.ptCenter[1] - cy) <= 2.0 and abs(r.dScale / s - 1) <= 0.03 for r in got), \
            (cx, cy, s, [(r.ptCenter, r.dScale) for r in got])
    gm.setScaleRange(1.0, 1.0)
    got1 = gm.match(src)
    assert len(got1) == 1 and math.hypot(got1[0].ptCenter[0] - 2600, got1[0].ptCenter[1] - 900) <= 2.0
