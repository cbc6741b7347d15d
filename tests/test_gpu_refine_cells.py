"""Refinement, cell by cell: all 49 float32 scores of every (layer, candidate, angle) eval of the pyramid descent against
the CPU oracle's trace, bit for bit, on every correlation path (FPM_PARAM_TENSOR_CORES 0, 1, 2, 3, 4, 6 and the exact
numerator of use_simd = 0), together with the rotated ROI patch each eval correlated.

Bit-equality is what the code implies: the same template-row-order float32 chain over exact integer row dots, exact
integer window sums, and the fp64 CCOEFF_NORMED epilogue in the reference's operation order (-fmad=false).  A score that
differs while its ROI matches points at the correlation kernel or the finalize kernel; a differing ROI at the warp.

The scenes are the golden cases plus synthetic ones built here, chosen so that the descent reaches the places kernels go
wrong: the path switches at template widths 16 and 64, the K-chunk at 128 ROI bytes, every width mod 4, template heights
below 6 (the window bookkeeping's edge rows overlap), several dp4a evals per CTA with a partial last CTA, several
workspace waves per layer, and each branch of the epilogue.  test_refine_cell_coverage asserts that they still do.

The top-score kernel's u32 / u64 accumulator boundary (template area 66000) is pinned at the end of the file.
"""
import numpy as np
import pytest

import fpm_workloads as synth
from oracle import oracle as O
from tests.helpers import configure, get_image

pytestmark = pytest.mark.gpu

GOLDEN = ["src8", "src9", "test4_src3", "cfg3_src6", "cfg1_synth", "src4", "cfg2_synth", "src9_subpix"]
MODES = (0, 1, 2, 3, 4, 6)
CORR_KERNELS = ("fpm_corr_rows_kernel", "fpm_corr_mma_kernel", "fpm_corr_fused_kernel", "fpm_corr_warp_kernel")
SMALL_WORKSPACE_MB = 0.25          # src4 and cfg2_synth then refine every layer in several waves
CR_MAX_THREADS = 256               # fpm_corr_rows_kernel: threads per CTA, one per ROI row (fpm_kernels.cuh)
BRANCH_NAMES = {O.BRANCH_FLAT: "den=0", O.BRANCH_CLAMP: "+-1 clamp", O.BRANCH_QUOTIENT: "quotient",
                O.BRANCH_ZERO: "|num|>=1.125den", O.BRANCH_EQUAL1: "flat template"}


# ---------------- synthetic scenes ----------------
def _texture(w, h, seed, lo=0, hi=255, sigma=1.5):
    t = synth.background(w, h, seed, sigma).astype(np.float64)
    t = (t - t.min()) / max(t.max() - t.min(), 1.0)
    return np.round(lo + t * (hi - lo)).astype(np.uint8)


def _scene_exact(tol):
    """a bright template (200..255: the row dots are large enough for the float chain to round) pasted unrotated at
    integer positions that are multiples of the pyramid step: cells at or next to 1.0, and the +-1 clamp"""
    tpl = _texture(64, 48, 31, 200, 255, 1.2)
    src = synth.background(420, 330, 32, 2.0)
    for (x, y) in ((16, 16), (200, 40), (96, 200), (304, 256)):
        src[y:y + 48, x:x + 64] = tpl
    return tpl, src, dict(max_pos=5, score=0.5, tolerance_angle=tol, min_reduce_area=256)


def _scene_flat():
    """Score = 0 on a constant source with one textured patch: the candidates in the flat area have den = 0 at every layer"""
    tpl = _texture(40, 32, 41)
    src = np.full((260, 320), 117, np.uint8)
    src[150:182, 200:240] = tpl
    return tpl, src, dict(max_pos=5, score=0.0, tolerance_angle=20, min_reduce_area=64)


def _scene_border():
    """targets centred less than half a template from the frame edges: the ROIs hang over the border at every layer"""
    tpl = _texture(60, 44, 51)
    src = synth.background(380, 290, 52, 2.5)
    for (cx, cy, a) in ((18.0, 14.0, 12.0), (366.0, 280.0, -150.0), (10.0, 270.0, 95.0), (371.0, 9.0, -33.0)):
        synth.paste_rotated(src, tpl, cx, cy, a)
    return tpl, src, dict(max_pos=6, score=0.5, tolerance_angle=180, min_reduce_area=256)


def _scene_shape(tw, th, mra, seed):
    """a template whose refinement levels have the widths / heights the scene is named after, three rotated copies"""
    tpl = _texture(tw, th, seed, 0, 255, 1.0)
    W, H = max(4 * tw, 300), max(6 * th, 260)
    src = synth.background(W, H, seed + 1, 2.0)
    for k, a in enumerate((0.0, 41.0, -127.0)):
        synth.paste_rotated(src, tpl, W * (k + 1) / 4.0, H * (0.3 + 0.2 * k), a)
    return tpl, src, dict(max_pos=3, score=0.5, tolerance_angle=180, min_reduce_area=mra)


SYNTH = {
    "exact_tol0": lambda: _scene_exact(0),
    "exact_tol180": lambda: _scene_exact(180),
    "flat_den0": _scene_flat,
    "border": _scene_border,
    "w120_h10_5_3": lambda: _scene_shape(120, 10, 64, 61),    # refines at 120x10, 60x5, 30x3
    "w123_62_31_16": lambda: _scene_shape(123, 36, 64, 62),   # 123x36, 62x18, 31x9, 16x5
    "w65_33_17": lambda: _scene_shape(65, 44, 64, 63),        # 65x44, 33x22, 17x11
    "w63_32_16": lambda: _scene_shape(63, 40, 64, 64),        # 63x40, 32x20, 16x10
    "w122_61": lambda: _scene_shape(122, 30, 256, 65),        # 122x30, 61x15
    "w128_64_32_16": lambda: _scene_shape(128, 60, 64, 66),   # 128x60, 64x30, 32x15, 16x8
    "w30_15": lambda: _scene_shape(30, 60, 64, 67),           # 30x60, 15x30, 8x15
}

_scenes = {}


def _scene(name, golden_cases):
    if name not in _scenes:
        if name in SYNTH:
            _scenes[name] = SYNTH[name]()
        else:
            c = golden_cases[name]
            _scenes[name] = (get_image(c["tpl"]), get_image(c["src"]), c["params"])
    return _scenes[name]


# ---------------- the oracle, once per scene ----------------
class _BranchOracle(O.OracleMatcher):
    """the oracle, also recording which epilogue branch every refinement cell takes (in the order of trace["refine"])"""

    def _match_template(self, src, layer, use_simd, top=False):
        if top:
            return super()._match_template(src, layer, use_simd, top)
        tpl = self.td.pyramid[layer]
        num = O.match_template_simd(src, tpl) if (self.use_simd and use_simd) else O.ccorr_exact_dense(src, tpl)
        self.branches.append(O.ccoeff_branches(src, self.td, num, layer))
        return O.ccoeff_denominator(src, self.td, num, layer)


_oracles = {}


def _oracle(name, use_simd, golden_cases):
    """{(layer, cand, j): trace record + "branch"}, template level shapes [(w, h)]"""
    key = (name, use_simd)
    if key not in _oracles:
        tpl, src, params = _scene(name, golden_cases)
        om = configure(_BranchOracle(), dict(params, use_simd=use_simd))
        om.branches, om.trace = [], {}
        om.learn_pattern(tpl)
        om.match(src)
        ref = om.trace["refine"]
        assert len(ref) == len(om.branches)
        evals = {}
        for e, b in zip(ref, om.branches):
            assert e["score"].shape == (7, 7)
            evals[(e["layer"], e["cand"], e["j"])] = dict(e, branch=b)
        _oracles[key] = (evals, [(p.shape[1], p.shape[0]) for p in om.td.pyramid])
    return _oracles[key]


# ---------------- the GPU, once per (scene, mode, use_simd, workspace) ----------------
def _corr_path(mode, use_simd, tw, n_ang):
    """the correlation kernel(s) run_refine picks for a level (fpm_host.cu: corr_warp_usable, mma_usable,
    mma_narrow_fused, fused_pays); for failure messages"""
    if mode == 6 and n_ang == 3 and tw >= 64:
        return "fpm_corr_warp_kernel"
    mma = mode in (2, 4) or (mode != 0 and tw >= 64)
    narrow = mode in (1, 6) and use_simd and 16 <= tw < 64
    if narrow or (mma and use_simd and mode != 3):
        if mode == 4:
            return "fpm_corr_fused_kernel"
        return "fpm_corr_fused_kernel or " + ("fpm_corr_mma_kernel" if mma else "fpm_corr_rows_kernel")
    return "fpm_corr_mma_kernel" if mma else "fpm_corr_rows_kernel"


_gpu_runs = {}


def _gpu(matcher, name, mode, use_simd, workspace_mb, golden_cases):
    key = (name, mode, use_simd, workspace_mb)
    if key in _gpu_runs:
        return _gpu_runs[key]
    from fastest_image_pattern_matching_b200 import _lib as L
    tpl, src, params = _scene(name, golden_cases)
    tc0, ws0 = matcher._get(L.PARAM_TENSOR_CORES), matcher._get(L.PARAM_WORKSPACE_MB)
    configure(matcher, dict(params, use_simd=use_simd))
    matcher.setTensorCores(mode)
    matcher.setWorkspaceMB(workspace_mb)
    try:
        assert matcher.learnPattern(tpl)
        matcher.setTrace(True)
        matcher.setProfile(True)
        matcher.profileReset()
        matcher.match(src)
        prof = matcher.profile()
        levels = len(matcher.templateLevels())
        evals = {}
        for layer in range(levels - 1):
            rows = matcher.traceEvals(layer)
            scores = matcher.traceEvalScores(layer)
            rois = matcher.traceEvalRois(layer)
            assert rois is None or len(rois) == len(rows)
            seen = {}
            for i, r in enumerate(rows):                 # rows: cand id, angle, score, locx, locy; n_ang per candidate, in order
                cid = int(r[0])
                j = seen.get(cid, 0)
                seen[cid] = j + 1
                evals[(layer, cid, j)] = dict(angle=float(r[1]), val=np.float32(r[2]), loc=(int(r[3]), int(r[4])),
                                              score=scores[i], roi=None if rois is None else rois[i])
    finally:
        matcher.setTrace(False)
        matcher.setProfile(False)
        matcher.setTensorCores(tc0)
        matcher.setWorkspaceMB(ws0)
        matcher.setUseSIMD(True)
    run = dict(evals=evals, kernels={k for k in CORR_KERNELS if prof[k][1] > 0},
               finalize_launches=prof["fpm_refine_finalize_kernel"][1])
    _gpu_runs[key] = run
    return run


def _compare(matcher, golden_cases, name, mode, use_simd=True, workspace_mb=4096):
    want, shapes = _oracle(name, use_simd, golden_cases)
    run = _gpu(matcher, name, mode, use_simd, workspace_mb, golden_cases)
    got = run["evals"]
    tag = "%s TENSOR_CORES=%d use_simd=%d workspace=%g MB" % (name, mode, use_simd, workspace_mb)
    missing, extra = sorted(set(want) - set(got)), sorted(set(got) - set(want))
    assert not missing and not extra, "%s: different (layer, cand, j) eval sets; only in the oracle %s, only on the GPU %s" % (
        tag, missing[:8], extra[:8])
    bad = []
    n_ang = {}
    for (layer, cand, j) in want:
        n_ang[(layer, cand)] = max(n_ang.get((layer, cand), 0), j + 1)
    for k in sorted(want):
        w, g = want[k], got[k]
        layer, cand, j = k
        tw, th = shapes[layer]
        where = "%s: layer %d (%dx%d) cand %d angle %d" % (tag, layer, tw, th, cand, j)
        path = _corr_path(mode, use_simd, tw, n_ang[(layer, cand)])
        roi_note = "ROI not kept (warped inside %s)" % path
        if g["roi"] is not None:
            roi = g["roi"]
            if not np.array_equal(roi[:, :tw + 6], w["roi"]):
                d = np.argwhere(roi[:, :tw + 6] != w["roi"])
                bad.append("%s: ROI differs at %d pixels, first (y, x) %s: got %d want %d (warp)" % (
                    where, len(d), tuple(d[0]), roi[tuple(d[0])], w["roi"][tuple(d[0])]))
                continue
            if roi[:, tw + 6:].any():
                bad.append("%s: pitch padding columns of the ROI are not zero" % where)
                continue
            roi_note = "ROI equal (correlation / finalize: %s)" % path
        if g["angle"] != w["angle"]:
            bad.append("%s: angle got %r want %r" % (where, g["angle"], w["angle"]))
            continue
        gs, ws = np.asarray(g["score"], np.float32), np.asarray(w["score"], np.float32)
        if not np.isfinite(gs).all():
            r, c = np.argwhere(~np.isfinite(gs))[0]
            bad.append("%s: cell (%d, %d) not finite: got %r; %s" % (where, r, c, gs[r, c], roi_note))
            continue
        diff = gs.view(np.uint32) != ws.view(np.uint32)
        if diff.any():
            cells = np.argwhere(diff)
            r, c = cells[0]
            bad.append("%s: %d of 49 cells differ, first (row %d, col %d): got %r want %r (%s branch); %s" % (
                where, len(cells), r, c, float(gs[r, c]), float(ws[r, c]), BRANCH_NAMES[int(w["branch"][r, c])], roi_note))
            continue
        if (g["loc"], g["val"]) != (tuple(w["loc"]), np.float32(w["val"])):
            bad.append("%s: best cell got %s %r want %s %r (7x7 argmax / best-of-3)" % (where, g["loc"], g["val"], w["loc"], w["val"]))
    assert not bad, "%d of %d evals differ:\n" % (len(bad), len(want)) + "\n".join(bad[:12])
    return run


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", GOLDEN + list(SYNTH))
def test_refine_cells_bit_equal_oracle(matcher, golden_cases, oracle_lib, name, mode):
    _compare(matcher, golden_cases, name, mode)


@pytest.mark.parametrize("mode", (0, 1, 2))
@pytest.mark.parametrize("name", ["src8", "cfg2_synth", "w120_h10_5_3"])
def test_refine_cells_exact_numerator(matcher, golden_cases, oracle_lib, name, mode):
    """use_simd = 0: the exact s64 numerator instead of the float chain (cv::matchTemplate in the reference)"""
    _compare(matcher, golden_cases, name, mode, use_simd=False)


@pytest.mark.parametrize("mode", (0, 1, 4))
@pytest.mark.parametrize("name", ["src4", "cfg2_synth"])
def test_refine_cells_in_workspace_waves(matcher, golden_cases, oracle_lib, name, mode):
    """a workspace that holds a few candidates: every layer in several waves, each wave's scores at its own offset"""
    run = _compare(matcher, golden_cases, name, mode, workspace_mb=SMALL_WORKSPACE_MB)
    layers = {k[0] for k in run["evals"]}
    assert run["finalize_launches"] >= 3 * len(layers), (run["finalize_launches"], sorted(layers))


def test_refine_cell_coverage(matcher, golden_cases, oracle_lib):
    """the scenes above reach every correlation kernel, every epilogue branch and the shapes where kernels go wrong"""
    names = GOLDEN + list(SYNTH)
    kernels = {}
    for name in names:
        for mode in MODES:
            for k in _gpu(matcher, name, mode, True, 4096, golden_cases)["kernels"]:
                kernels.setdefault(k, set()).add((name, mode))
    assert set(CORR_KERNELS) <= set(kernels), "correlation kernels never run: %s" % (set(CORR_KERNELS) - set(kernels))
    assert {m for (_, m) in kernels["fpm_corr_warp_kernel"]} == {6}
    for name in names:
        assert _gpu(matcher, name, 0, True, 4096, golden_cases)["kernels"] <= {"fpm_corr_rows_kernel"}, name
    branches = {}
    widths, heights, rows_grids = set(), set(), []
    for name in names:
        evals, shapes = _oracle(name, True, golden_cases)
        per_layer = {}
        for (layer, _, _), e in evals.items():
            per_layer[layer] = per_layer.get(layer, 0) + 1
            for b, n in zip(*np.unique(e["branch"], return_counts=True)):
                branches[int(b)] = branches.get(int(b), 0) + int(n)
        for layer, ne in per_layer.items():
            tw, th = shapes[layer]
            widths.add(tw)
            heights.add(th)
            epc = CR_MAX_THREADS // (th + 6) if th + 6 <= 128 else 1
            rows_grids.append((name, layer, ne, epc))
    for b in (O.BRANCH_FLAT, O.BRANCH_CLAMP, O.BRANCH_QUOTIENT):
        assert branches.get(b, 0) > 0, "no refinement cell takes the %s branch: %s" % (BRANCH_NAMES[b], branches)
    assert {15, 16, 17, 63, 64, 65, 122, 123} <= widths, sorted(widths)
    assert {w % 4 for w in widths} == {0, 1, 2, 3}
    assert any(h < 6 for h in heights), sorted(heights)
    assert any(h >= 32 and h % 8 for h in heights), sorted(heights)
    # TENSOR_CORES = 0 runs every level on fpm_corr_rows_kernel: one level has several evals per CTA and a partial last CTA
    assert any(epc > 1 and ne % epc for (_, _, ne, epc) in rows_grids), rows_grids


# ---------------- top layer: the u32 / u64 accumulator boundary of fpm_top_score_kernel ----------------
@pytest.mark.parametrize("th", [33, 34])
def test_top_score_accumulator_boundary(matcher, th):
    """2000x33 (area 66000, the largest u32 accumulator: 66000 * 255^2 < 2^32) and 2000x34 (u64) top-layer templates on
    images with saturated regions, random texture and one exact copy: bit-equal to the exact integer map"""
    tw = 2000
    rng = np.random.default_rng(th)
    tpl = np.full((th, tw), 255, np.uint8)                  # mostly saturated: the window sums approach 2^32
    tpl[:, 700:760] = rng.integers(0, 256, (th, 60), dtype=np.uint8)
    tpl[th // 2, ::7] = 0
    img = rng.integers(0, 256, (th + 70, tw + 90), dtype=np.uint8)
    img[:th + 20, :tw + 40] = 255                            # saturated region larger than the template
    img[5:th + 5, 30:40] = rng.integers(0, 256, (th, 10), dtype=np.uint8)
    img[th + 30:2 * th + 30, 60:60 + tw] = tpl                # the exact copy
    mra = 261 * 261                                           # int(sqrt(MinReduceArea))^2 >= 68000: the template is its own top layer
    configure(matcher, dict(min_reduce_area=mra))
    try:
        assert matcher.learnPattern(tpl)
        lv = matcher.templateLevels()
        assert len(lv) == 1 and (lv[0]["w"], lv[0]["h"]) == (tw, th)
        got = matcher.dbgTopScore(img)
    finally:
        matcher.setMinReduceArea(256)
    om = configure(O.OracleMatcher(), dict(min_reduce_area=mra))
    om.learn_pattern(tpl)
    want = O.ccoeff_denominator(img, om.td, O.ccorr_exact_dense(img, tpl), 0)
    assert got.shape == want.shape
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), float(np.abs(got - want).max())
    assert want[th + 30, 60] > 0.999
