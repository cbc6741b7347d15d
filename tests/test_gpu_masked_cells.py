"""Masked templates (fpm_learn_masked), cell by cell: all 49 float32 scores and the ROI of every refinement eval against the
masked CPU oracle (tests/masked_oracle.py), bit for bit, on every correlation path; the masked top-layer score map against
the exact fp64 masked map; and the production (async) descent against the synchronous one.

Masks add device code that unmasked matching never runs: the masked build of fpm_top_score_kernel (row prefix sums from a
warp scan, then walks over each template row's runs of kept pixels), fpm_mask_window_kernel (the 49 window sums of every
refinement eval from the ROI patch) and the finalize kernel's masked window sums.  A mistake there gives slightly wrong
scores, not a crash, so every comparison here is bit-exact.

The scenes are the synthetic shape scenes of tests/test_gpu_refine_cells.py (refinement widths 15/16/17, 63/64/65, 122/123,
every width mod 4, heights below 6, flat windows, exact copies, targets on the border), each under one blob mask and one
edge mask.  The edge masks (tests/masked_oracle.py EDGE_MASKS) give the run tables the blobs never do: rows of many runs
and runs of one pixel (comb), whole empty rows (banded), runs at x = 0 and x = w (frame), and few kept pixels (sparse).
test_masked_cell_coverage asserts that the runs reach all of this.
"""
import numpy as np
import pytest

import fpm_workloads as synth
from oracle import oracle as O
from tests import test_gpu_refine_cells as RC
from tests.helpers import assert_results_match, configure
from tests.masked_oracle import (EDGE_MASKS, MASKS, MaskedOracleMatcher, ccoeff_branches_masked, ccoeff_denominator_masked,
                                 mask_runs)

pytestmark = pytest.mark.gpu

SCENES = ["w120_h10_5_3", "w123_62_31_16", "w65_33_17", "w63_32_16", "w122_61", "w128_64_32_16", "w30_15", "flat_den0",
          "exact_tol180", "border"]
ALL_MASKS = dict(MASKS, **EDGE_MASKS)
BLOB_ORDER = ["disc", "ring", "holed", "blob", "corner_cut"]
EDGE_ORDER = ["comb", "banded", "frame", "sparse"]
# every scene under one blob mask and one edge mask, the masks taken in turn
# (exact copies under the sparse mask: cells whose float chain rounds past the denominator, the +-1 clamp)
PAIRS = [(s, BLOB_ORDER[i % len(BLOB_ORDER)]) for i, s in enumerate(SCENES)] + \
        [(s, EDGE_ORDER[i % len(EDGE_ORDER)]) for i, s in enumerate(SCENES)] + [("exact_tol180", "sparse")]
MODES = (0, 1, 2, 3, 4, 6)
MASK_KERNELS = ("fpm_mask_window_kernel", "fpm_top_score_kernel(masked)")
RUN_KERNELS = ("fpm_corr_rows_kernel", "fpm_corr_mma_kernel", "fpm_corr_fused_kernel")


def _scene(name):
    return RC._scene(name, None)


# ---------------- the masked oracle with the epilogue branch of every refinement cell ----------------
class _MaskedBranchOracle(MaskedOracleMatcher):
    """the masked oracle, also recording which epilogue branch every refinement cell takes (in the order of trace["refine"])"""

    def _match_template(self, src, layer, use_simd, top=False):
        if top:
            return super()._match_template(src, layer, use_simd, top)
        tpl = self.masked_pyr[layer]
        num = O.match_template_simd(src, tpl) if (self.use_simd and use_simd) else O.ccorr_exact_dense(src, tpl)
        self.branches.append(ccoeff_branches_masked(src, self.td, self.masks[layer], num, layer))
        return ccoeff_denominator_masked(src, self.td, self.masks[layer], num, layer)


_oracles = {}


def _oracle(name, mask_name, use_simd=True):
    """({(layer, cand, j): trace record + "branch"}, level shapes [(w, h)], level masks, result list)"""
    key = (name, mask_name, use_simd)
    if key not in _oracles:
        tpl, src, params = _scene(name)
        m = ALL_MASKS[mask_name](tpl.shape[1], tpl.shape[0])
        om = configure(_MaskedBranchOracle(), dict(params, use_simd=use_simd))
        om.branches, om.trace = [], {}
        assert om.learn_pattern(tpl, m)
        res = om.match(src)
        ref = om.trace["refine"]
        assert len(ref) == len(om.branches)
        evals = {(e["layer"], e["cand"], e["j"]): dict(e, branch=b) for e, b in zip(ref, om.branches)}
        _oracles[key] = (evals, [(p.shape[1], p.shape[0]) for p in om.td.pyramid], om.masks, res)
    return _oracles[key]


# ---------------- the GPU, traced, once per (scene, mask, mode, use_simd, workspace) ----------------
_gpu_runs = {}


def _gpu(matcher, name, mask_name, mode, use_simd=True, workspace_mb=4096):
    key = (name, mask_name, mode, use_simd, workspace_mb)
    if key in _gpu_runs:
        return _gpu_runs[key]
    from fastest_image_pattern_matching_b200 import _lib as L
    tpl, src, params = _scene(name)
    m = ALL_MASKS[mask_name](tpl.shape[1], tpl.shape[0])
    tc0, ws0 = matcher._get(L.PARAM_TENSOR_CORES), matcher._get(L.PARAM_WORKSPACE_MB)
    configure(matcher, dict(params, use_simd=use_simd))
    matcher.setTensorCores(mode)
    matcher.setWorkspaceMB(workspace_mb)
    try:
        assert matcher.learnPattern(tpl, m)
        matcher.setTrace(True)
        matcher.setProfile(True)
        matcher.profileReset()
        matcher.match(src)
        prof = matcher.profile()
        levels = matcher.templateLevels()
        evals = {}
        for layer in range(len(levels) - 1):
            rows = matcher.traceEvals(layer)
            scores = matcher.traceEvalScores(layer)
            rois = matcher.traceEvalRois(layer)
            assert rois is None or len(rois) == len(rows)
            seen = {}
            for i, r in enumerate(rows):
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
    run = dict(evals=evals, kernels={k for k in RC.CORR_KERNELS + MASK_KERNELS if prof[k][1] > 0},
               launches={k: prof[k][1] for k in ("fpm_refine_finalize_kernel",) + MASK_KERNELS},
               masks=[lv["mask"] for lv in levels])
    _gpu_runs[key] = run
    return run


def _compare(matcher, name, mask_name, mode, use_simd=True, workspace_mb=4096):
    want, shapes, masks, _ = _oracle(name, mask_name, use_simd)
    run = _gpu(matcher, name, mask_name, mode, use_simd, workspace_mb)
    got = run["evals"]
    tag = "%s mask %s TENSOR_CORES=%d use_simd=%d workspace=%g MB" % (name, mask_name, mode, use_simd, workspace_mb)
    assert len(run["masks"]) == len(masks) and all(np.array_equal(a, b) for a, b in zip(run["masks"], masks)), \
        "%s: level masks differ from M_{L+1} = pyrDown(255 M_L) >= 128" % tag
    missing, extra = sorted(set(want) - set(got)), sorted(set(got) - set(want))
    sets_note = "%s: different (layer, cand, j) eval sets; only in the oracle %s, only on the GPU %s" % (
        tag, missing[:8], extra[:8])
    n_ang = {}
    for (layer, cand, j) in want:
        n_ang[(layer, cand)] = max(n_ang.get((layer, cand), 0), j + 1)
    bad = []
    # the evals both ran, from the layer the descent starts at down: the first difference is where the scores part
    for k in sorted(set(want) & set(got), key=lambda k: (-k[0], k[1], k[2])):
        w, g = want[k], got[k]
        layer, cand, j = k
        tw, th = shapes[layer]
        where = "%s: layer %d (%dx%d, %d kept, %d runs) cand %d angle %d" % (
            tag, layer, tw, th, int(masks[layer].sum()), sum(len(r) for r in mask_runs(masks[layer])), cand, j)
        path = RC._corr_path(mode, use_simd, tw, n_ang[(layer, cand)])
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
            roi_note = "ROI equal: numerator of M_L*T_L from %s, window sums from fpm_mask_window_kernel, epilogue in " \
                       "fpm_refine_finalize_kernel" % path
        if g["angle"] != w["angle"]:
            bad.append("%s: angle got %r want %r" % (where, g["angle"], w["angle"]))
            continue
        gs, ws = np.asarray(g["score"], np.float32).reshape(7, 7), np.asarray(w["score"], np.float32)
        if not np.isfinite(gs).all():
            r, c = np.argwhere(~np.isfinite(gs))[0]
            bad.append("%s: cell (%d, %d) not finite: got %r; %s" % (where, r, c, gs[r, c], roi_note))
            continue
        diff = gs.view(np.uint32) != ws.view(np.uint32)
        if diff.any():
            cells = np.argwhere(diff)
            r, c = cells[0]
            bad.append("%s: %d of 49 cells differ, first (row %d, col %d): got %r want %r (%s branch); %s" % (
                where, len(cells), r, c, float(gs[r, c]), float(ws[r, c]), RC.BRANCH_NAMES[int(w["branch"][r, c])], roi_note))
            continue
        if (g["loc"], g["val"]) != (tuple(w["loc"]), np.float32(w["val"])):
            bad.append("%s: best cell got %s %r want %s %r (7x7 argmax / best-of-3)" % (where, g["loc"], g["val"], w["loc"], w["val"]))
    assert not bad, "%d of %d evals differ:\n" % (len(bad), len(want)) + "\n".join(bad[:12]) + (
        "\n" + sets_note if missing or extra else "")
    assert not missing and not extra, sets_note
    return run


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name,mask_name", PAIRS)
def test_masked_refine_cells_bit_equal_oracle(matcher, oracle_lib, name, mask_name, mode):
    _compare(matcher, name, mask_name, mode)


@pytest.mark.parametrize("mode", (0, 1, 2))
@pytest.mark.parametrize("name,mask_name", [("w120_h10_5_3", "comb"), ("w65_33_17", "frame"), ("border", "ring")])
def test_masked_refine_cells_exact_numerator(matcher, oracle_lib, name, mask_name, mode):
    """use_simd = 0: the exact s64 numerator instead of the float chain"""
    _compare(matcher, name, mask_name, mode, use_simd=False)


@pytest.mark.parametrize("mode", (0, 1, 4))
@pytest.mark.parametrize("name,mask_name", [("border", "banded"), ("w128_64_32_16", "blob")])
def test_masked_refine_cells_in_workspace_waves(matcher, oracle_lib, name, mask_name, mode):
    """a workspace that holds a few candidates: every layer in several waves, each wave's masked window sums next to its
    own finalize"""
    run = _compare(matcher, name, mask_name, mode, workspace_mb=RC.SMALL_WORKSPACE_MB)
    layers = {k[0] for k in run["evals"]}
    n = run["launches"]
    assert n["fpm_refine_finalize_kernel"] >= 3 * len(layers), (n, sorted(layers))
    assert n["fpm_mask_window_kernel"] >= 3 * len(layers), (n, sorted(layers))


def test_masked_cell_coverage(matcher, oracle_lib):
    """the masked runs above reach every correlation kernel, both mask kernels, the shapes and epilogue branches of the
    unmasked coverage test, and the run-table cases of the edge masks at a refined level"""
    kernels = {}
    for name, mask_name in PAIRS:
        for mode in MODES:
            for k in _gpu(matcher, name, mask_name, mode)["kernels"]:
                kernels.setdefault(k, set()).add((name, mask_name, mode))
    missing = set(RUN_KERNELS + MASK_KERNELS) - set(kernels)
    assert not missing, "kernels never run on a masked template: %s" % missing
    assert "fpm_corr_warp_kernel" not in kernels                  # a masked template takes the mode-1 route in mode 6
    branches = {}
    widths, heights = set(), set()
    empty_row = many_runs = run_of_1 = both_edges = False
    for name, mask_name in PAIRS:
        evals, shapes, _, _ = _oracle(name, mask_name)
        refined = {layer for (layer, _, _) in evals}
        for e in evals.values():
            for b, n in zip(*np.unique(e["branch"], return_counts=True)):
                branches[int(b)] = branches.get(int(b), 0) + int(n)
        levels = _gpu(matcher, name, mask_name, 1)["masks"]
        for layer in refined:
            tw, th = shapes[layer]
            widths.add(tw)
            heights.add(th)
            runs = mask_runs(levels[layer])
            empty_row |= any(not r for r in runs)
            many_runs |= any(len(r) >= 8 for r in runs)
            run_of_1 |= any(e - b == 1 for r in runs for b, e in r)
            both_edges |= any(len(r) >= 2 and r[0][0] == 0 and r[-1][1] == tw for r in runs)
    for b in (O.BRANCH_FLAT, O.BRANCH_CLAMP, O.BRANCH_QUOTIENT):
        assert branches.get(b, 0) > 0, "no masked refinement cell takes the %s branch: %s" % (RC.BRANCH_NAMES[b], branches)
    assert {15, 16, 17, 63, 64, 65, 122, 123} <= widths, sorted(widths)
    assert {w % 4 for w in widths} == {0, 1, 2, 3}
    assert any(h < 6 for h in heights), sorted(heights)
    assert any(h >= 32 and h % 8 for h in heights), sorted(heights)
    assert empty_row and many_runs and run_of_1 and both_edges, dict(
        empty_row=empty_row, row_of_8_runs=many_runs, run_of_1=run_of_1, runs_at_both_edges=both_edges)


# ---------------- the production single-frame descent (no trace) ----------------
def _key(r):
    return (r.dMatchScore, r.dMatchedAngle, r.ptCenter, r.ptLT, r.ptRT, r.ptRB, r.ptLB)


_frame_oracles = {}


def _frame_oracle(name, mask_name, k, frame):
    key = (name, mask_name, k)
    if key not in _frame_oracles:
        tpl, _, params = _scene(name)
        om = configure(MaskedOracleMatcher(), params)
        assert om.learn_pattern(tpl, ALL_MASKS[mask_name](tpl.shape[1], tpl.shape[0]))
        _frame_oracles[key] = om.match(frame)
    return _frame_oracles[key]


@pytest.mark.parametrize("mode", (1, 2, 4))
@pytest.mark.parametrize("name,mask_name", [("w65_33_17", "comb"), ("w30_15", "frame"), ("w120_h10_5_3", "disc")])
def test_masked_async_descent_equals_synchronous(matcher, oracle_lib, name, mask_name, mode):
    """FPM_PARAM_ASYNC_DESCENT 1 (every layer enqueued at once, live counts read on the device, fused correlation only in
    mode 4) gives the lists of the synchronous descent, on one frame and a batch of three, and both are the oracle's"""
    tpl, src, params = _scene(name)
    frames = [src, np.ascontiguousarray(src[:, ::-1]), np.ascontiguousarray(src[::-1])]
    configure(matcher, params)
    matcher.setTensorCores(mode)
    try:
        assert matcher.learnPattern(tpl, ALL_MASKS[mask_name](tpl.shape[1], tpl.shape[0]))
        got = {}
        for a in (0, 1):
            matcher.setAsyncDescent(a)
            got[a] = [matcher.match(src)] + matcher.matchBatch(np.stack(frames))
    finally:
        matcher.setAsyncDescent(-1)
        matcher.setTensorCores(1)
    tag = "%s mask %s TENSOR_CORES=%d" % (name, mask_name, mode)
    assert got[0][0], tag
    for i, what in enumerate(["single frame", "batch frame 0", "batch frame 1", "batch frame 2"]):
        assert [_key(r) for r in got[1][i]] == [_key(r) for r in got[0][i]], "%s, %s: async descent differs from synchronous" % (
            tag, what)
        k = max(i - 1, 0)
        want = _oracle(name, mask_name)[3] if k == 0 else _frame_oracle(name, mask_name, k, frames[k])
        assert_results_match(got[0][i], want, ordered=False)


# ---------------- top layer: fpm_top_score_kernel<false, true> against the exact fp64 masked map ----------------
def top_score_smem_masked(tw, th):
    """top_score_smem(tw, th, masked = true) of fpm_host.cu: template words, patch words, and two rows of TS_TW + tw
    prefix entries per patch row (TS_TW = 64, TS_TH = 16)"""
    nwt = (tw + 3) // 4
    pww = 64 // 4 + nwt + 1
    return 4 * (th * nwt + (16 + th - 1) * (pww + 2 * (64 + tw))) + 16


SMEM_LIMIT = 200 * 1024


def _own_top_layer(matcher, tpl, mask, mra=None):
    """learn at MinReduceArea mra, by default one at which the template is its own top layer; returns the oracle of that
    learn"""
    h, w = tpl.shape
    if mra is None:
        d = int(np.ceil(np.sqrt(w * h))) + 1
        mra = d * d
    configure(matcher, dict(min_reduce_area=mra))
    assert matcher.learnPattern(tpl, mask)
    om = configure(MaskedOracleMatcher(), dict(min_reduce_area=mra))
    assert om.learn_pattern(tpl, mask)
    lv = matcher.templateLevels()
    assert len(lv) == len(om.td.pyramid) and (lv[-1]["w"], lv[-1]["h"]) == om.td.pyramid[-1].shape[::-1]
    return om


def _top_map_compare(matcher, tpl, mask, img, what, mra=None):
    om = _own_top_layer(matcher, tpl, mask, mra)
    try:
        got = matcher.dbgTopScore(img)
    finally:
        matcher.setMinReduceArea(256)
    top = len(om.td.pyramid) - 1
    num = O.ccorr_exact_dense(img, om.masked_pyr[top])
    want = ccoeff_denominator_masked(img, om.td, om.masks[top], num, top)
    assert got.shape == want.shape, what
    diff = got.view(np.uint32) != want.view(np.uint32)
    if diff.any():
        r, c = np.argwhere(diff)[0]
        unmasked = ccoeff_denominator_masked(img, om.td, om.masks[top], O.ccorr_exact_dense(img, om.td.pyramid[top]), top)
        cause = ("the map is that of the unmasked T_L: the device template of level %d is not M_L*T_L (the learn's masked "
                 "upload)" % top) if np.array_equal(got.view(np.uint32), unmasked.view(np.uint32)) else \
            "prefix scan / run walk of fpm_top_score_kernel(masked)"
        raise AssertionError("%s: top level %d, fpm_top_score_kernel(masked) map differs at %d of %d cells, first (%d, %d): "
                             "got %r want %r; %s" % (what, top, int(diff.sum()), diff.size, r, c, float(got[r, c]),
                                                     float(want[r, c]), cause))
    return want


@pytest.mark.parametrize("mask_name", ["comb", "frame", "disc"])
@pytest.mark.parametrize("top", [1, 2])
def test_masked_top_score_map_at_a_reduced_level(matcher, top, mask_name):
    """a top layer that is level 1 or 2 of the pyramid: the score kernel correlates the uploaded M_L*T_L of that level"""
    tw, th = 72, 52
    tpl = synth.background(tw, th, 17, 1.2)
    d = {1: 40, 2: 20}[top]                                  # (tw*th) >> 2*top <= d^2 < (tw*th) >> 2*(top-1)
    rng = np.random.default_rng(top)
    img = rng.integers(0, 256, ((th >> top) + 30, (tw >> top) + 70), dtype=np.uint8)
    img[:12, :40] = 255
    _top_map_compare(matcher, tpl, ALL_MASKS[mask_name](tw, th), img, "%dx%d template, mask %s" % (tw, th, mask_name), mra=d * d)


@pytest.mark.parametrize("mask_name", ["comb", "banded", "frame", "sparse", "ring"])
@pytest.mark.parametrize("rw,rh", [(1, 1), (63, 17), (65, 15), (130, 1), (130, 17)])
@pytest.mark.parametrize("tw,th", [(37, 9), (50, 11), (67, 10), (100, 13)])
def test_masked_top_score_map_shapes(matcher, tw, th, rw, rh, mask_name):
    """template widths of every residue mod 4 (67 and 100: TS_TW + tw > 128, the prefix scan's second 32-word pass and its
    carry), map widths 1 / 63 / 65 / 130 and heights 1 / 15 / 17, on random texture with saturated and dark patches"""
    rng = np.random.default_rng(tw * 1000 + rw * 10 + rh)
    tpl = synth.background(tw, th, tw + th, 1.2)
    img = rng.integers(0, 256, (th + rh - 1, tw + rw - 1), dtype=np.uint8)
    img[: (th + rh) // 2, : (tw + rw) // 3] = 255
    img[-2:, -5:] = 0
    _top_map_compare(matcher, tpl, EDGE_MASKS[mask_name](tw, th) if mask_name in EDGE_MASKS else MASKS[mask_name](tw, th),
                     img, "%dx%d template, %dx%d map, mask %s" % (tw, th, rw, rh, mask_name))


def _largest_fitting_width(th):
    tw = 64
    while top_score_smem_masked(tw + 1, th) <= SMEM_LIMIT:
        tw += 1
    return tw


@pytest.mark.parametrize("th", [8, 24])
def test_masked_top_score_at_the_shared_memory_limit(matcher, th):
    """the widest masked top level whose score kernel fits 200 KB of dynamic shared memory, on mostly saturated images
    (the u32 prefix sums at their largest), bit-equal to the exact map with one exact copy scoring 1; one pixel wider
    is refused by the score kernel and the handle keeps working"""
    from fastest_image_pattern_matching_b200.matcher import FpmError
    tw = _largest_fitting_width(th)
    rng = np.random.default_rng(th)
    tpl = np.full((th, tw), 255, np.uint8)
    tpl[:, tw // 3:tw // 3 + 40] = rng.integers(0, 256, (th, 40), dtype=np.uint8)
    mask = EDGE_MASKS["comb"](tw, th)
    img = rng.integers(0, 256, (2 * th + 40, tw + 70), dtype=np.uint8)
    img[:th + 10, :tw + 30] = 255
    img[th + 20:2 * th + 20, 50:50 + tw] = tpl
    want = _top_map_compare(matcher, tpl, mask, img, "%dx%d masked top level (%d B of shared memory)" % (
        tw, th, top_score_smem_masked(tw, th)))
    assert want[th + 20, 50] > 0.999
    wide = np.full((th, tw + 1), 255, np.uint8)
    wide[:, :tw] = tpl
    _own_top_layer(matcher, wide, EDGE_MASKS["comb"](tw + 1, th))
    try:
        assert top_score_smem_masked(tw + 1, th) > SMEM_LIMIT
        with pytest.raises(FpmError, match="score kernel"):
            matcher.dbgTopScore(img)
        with pytest.raises(FpmError, match="score kernel"):
            matcher.match(img)
    finally:
        matcher.setMinReduceArea(256)
    tpl2, src2, params2 = _scene("w65_33_17")
    configure(matcher, params2)
    assert matcher.learnPattern(tpl2, MASKS["disc"](tpl2.shape[1], tpl2.shape[0]))
    assert_results_match(matcher.match(src2), _oracle("w65_33_17", "disc")[3], ordered=False)


def test_masked_top_score_u64_accumulators_unreachable(matcher):
    """the u32 / u64 accumulator boundary of the top-score kernel (template area 66000) lies beyond the masked shared-memory
    limit: the two prefix rows per patch row alone take 8 * (15 + th) * (64 + tw) > 8 * area bytes, so no masked top level
    above area 25600 fits; a masked 2000x33 top level (area 66000) is refused by the score kernel"""
    from fastest_image_pattern_matching_b200.matcher import FpmError
    assert 8 * 25600 == SMEM_LIMIT and top_score_smem_masked(2000, 33) > SMEM_LIMIT
    tpl = synth.background(2000, 33, 5, 1.5)
    _own_top_layer(matcher, tpl, EDGE_MASKS["frame"](2000, 33))
    try:
        with pytest.raises(FpmError, match="score kernel"):
            matcher.dbgTopScore(np.zeros((40, 2010), np.uint8))
    finally:
        matcher.setMinReduceArea(256)


# ---------------- wide masked levels: fpm_mask_window_kernel with one warp per CTA ----------------
@pytest.mark.parametrize("mode", (0, 1))
@pytest.mark.parametrize("tw,mask_name", [(5000, "frame"), (6400, "comb")])
def test_masked_wide_levels(matcher, oracle_lib, tw, mask_name, mode):
    """a thin wide masked template refined at widths 1250-6400: fpm_mask_window_kernel runs one warp per CTA from width
    4090 and needs more than 48 KB of shared memory from 6138; its 800x8 (625x8) top level fits the masked score kernel"""
    th = 64
    name = "wide%d_%s" % (tw, mask_name)
    if name not in RC._scenes:
        tpl = RC._texture(tw, th, tw, 0, 255, 1.0)
        src = synth.background(tw + 160, 200, tw + 1, 2.0)
        src[90:90 + th, 70:70 + tw] = tpl
        RC._scenes[name] = (tpl, src, dict(max_pos=1, score=0.5, tolerance_angle=0, min_reduce_area=100 * 100))
    _, shapes, _, want = _oracle(name, mask_name)
    assert shapes[0] == (tw, th) and len(shapes) == 4 and top_score_smem_masked(*shapes[-1]) <= SMEM_LIMIT, shapes
    run = _compare(matcher, name, mask_name, mode)
    assert {k[0] for k in run["evals"]} == {0, 1, 2}
    assert run["launches"]["fpm_mask_window_kernel"] >= 3
    tpl, src, params = _scene(name)
    configure(matcher, params)
    matcher.setTensorCores(mode)
    try:
        assert matcher.learnPattern(tpl, EDGE_MASKS[mask_name](tw, th))
        got = matcher.match(src)
    finally:
        matcher.setTensorCores(1)
        matcher.setMinReduceArea(256)
    assert len(want) == 1 and want[0].score > 0.99
    assert_results_match(got, want, ordered=False)
