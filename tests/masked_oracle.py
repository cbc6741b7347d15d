"""CPU oracle of masked templates (fpm_learn_masked) -- TEST INFRASTRUCTURE ONLY.

`MaskedOracleMatcher` is `oracle.oracle.OracleMatcher` with `learn_pattern(tpl, mask=None)`.  With a mask:

- M_0 = (mask != 0), M_{L+1} = (cv2.pyrDown(255 * M_L) >= 128); the template pyramid T_L is the unmasked one;
- per level n_L = sum M_L, inv_area = 1 / n_L, and mean / norm / result_equal1 from the exact integer sums
  sum M_L*T_L and sum M_L*T_L^2 in the operation order of the cv::meanStdDev model (mean = S/N, var = Q/N - mean^2);
- the border colour is (kept mean of level 0) < 128 ? 255 : 0;
- every placement scores the numerator of the template M_L*T_L with the window sums t = sum M_L*S and t2 = sum M_L*S^2
  (exact integers) in the unchanged CCOEFF_NORMED epilogue.

Everything else (angle schedule, peaks, descent, NMS, sub-pixel fit, MFC conventions) is the unmasked oracle's.
"""
from __future__ import annotations

import math

import cv2
import numpy as np

from oracle import oracle as O


def mask_pyramid(mask0, top):
    """[M_0 .. M_top] as 0/1 uint8 arrays."""
    ms = [(np.asarray(mask0) != 0).astype(np.uint8)]
    for _ in range(top):
        ms.append((cv2.pyrDown(ms[-1] * np.uint8(255)) >= 128).astype(np.uint8))
    return ms


def masked_level_stats(tpl, m):
    """(mean, norm, inv_area, result_equal1, n) of one level from the exact sums over the kept pixels."""
    t = tpl.astype(np.int64)
    mk = m.astype(np.int64)
    S, Q, n = int((t * mk).sum()), int((t * t * mk).sum()), int(mk.sum())
    scale = 1.0 / float(n)
    mean = float(S) * scale
    var = max(float(Q) * scale - mean * mean, 0.0)
    sdv = math.sqrt(var)
    inv_area = 1.0 / float(n)
    norm = sdv * sdv
    equal1 = norm < O.DBL_EPSILON
    norm = math.sqrt(norm)
    norm /= math.sqrt(inv_area)
    return mean, norm, inv_area, equal1, n


def mask_runs(m):
    """per row the [b, e) column ranges of kept pixels"""
    out = []
    for row in np.asarray(m, np.uint8):
        d = np.diff(np.concatenate(([0], row.astype(np.int8), [0])))
        out.append(list(zip(np.nonzero(d == 1)[0].tolist(), np.nonzero(d == -1)[0].tolist())))
    return out


def masked_window_sums(src, m):
    """exact t[r, c] = sum M*S and t2[r, c] = sum M*S^2 over every placement of the mask on src (int64)"""
    th, tw = m.shape
    R, C = src.shape[0] - th + 1, src.shape[1] - tw + 1
    s = src.astype(np.int64)
    ps = np.zeros((s.shape[0], s.shape[1] + 1), np.int64)
    pq = np.zeros_like(ps)
    ps[:, 1:] = np.cumsum(s, axis=1)
    pq[:, 1:] = np.cumsum(s * s, axis=1)
    t = np.zeros((R, C), np.int64)
    t2 = np.zeros((R, C), np.int64)
    cols = np.arange(C)
    for i, runs in enumerate(mask_runs(m)):
        if not runs:
            continue
        b, e = (np.asarray(v)[:, None] + cols for v in zip(*runs))     # [run][c]: all runs of the row in one gather
        t += (ps[i:i + R, e] - ps[i:i + R, b]).sum(axis=1)
        t2 += (pq[i:i + R, e] - pq[i:i + R, b]).sum(axis=1)
    return t, t2


def ccoeff_num_den_masked(src, td, m, result, layer):
    """ccoeff_num_den with the masked window sums (float64, same operation order)"""
    ti, t2i = masked_window_sums(src, m)
    t = ti.astype(np.float64)
    num = result.astype(np.float64)
    wnd_mean2 = (t * t) * td.inv_area[layer]
    num = num - t * td.templ_mean[layer]
    wnd_sum2 = t2i.astype(np.float64)
    diff2 = np.maximum(wnd_sum2 - wnd_mean2, 0.0)
    den = np.where(diff2 <= np.minimum(0.5, 10 * O.FLT_EPSILON * wnd_sum2), 0.0,
                   np.sqrt(diff2) * td.templ_norm[layer])
    return num, den


def ccoeff_denominator_masked(src, td, m, result, layer):
    if td.result_equal1[layer]:
        result[:] = 1
        return result
    num, den = ccoeff_num_den_masked(src, td, m, result, layer)
    absn = np.abs(num)
    with np.errstate(divide="ignore", invalid="ignore"):
        out = np.where(absn < den, num / den,
                       np.where(absn < den * 1.125, np.where(num > 0, 1.0, -1.0), 0.0))
    result[:] = out.astype(O.f32)
    return result


class MaskedOracleMatcher(O.OracleMatcher):
    def __init__(self):
        super().__init__()
        self.masks = None            # [M_L] (0/1) when a mask was learned
        self.masked_pyr = None       # [M_L * T_L]

    def learn_pattern(self, tpl, mask=None):
        self.masks = self.masked_pyr = None
        if mask is None:
            return super().learn_pattern(tpl)
        if tpl is None or tpl.size == 0:
            return False
        if np.asarray(mask).shape != tpl.shape:
            raise ValueError("mask shape differs from the template's")
        if not np.any(mask):
            raise ValueError("the mask keeps no pixel")
        td = O.TemplData()
        top = O.get_top_layer(tpl.shape[1], tpl.shape[0], int(math.sqrt(float(self.min_reduce_area))))
        td.pyramid = O.build_pyramid(np.ascontiguousarray(tpl), top)
        masks = mask_pyramid(mask, top)
        for l, m in enumerate(masks):
            if not m.any():
                raise ValueError("the mask keeps no pixel at pyramid level %d" % l)
        for lvl, m in zip(td.pyramid, masks):
            mean, norm, inv_area, equal1, _ = masked_level_stats(lvl, m)
            td.templ_mean.append(mean)
            td.templ_norm.append(norm)
            td.inv_area.append(inv_area)
            td.result_equal1.append(equal1)
        t0, m0 = td.pyramid[0].astype(np.int64), masks[0].astype(np.int64)
        td.border_color = 255 if float(int((t0 * m0).sum())) / float(int(m0.sum())) < 128 else 0
        td.learned = True
        self.td = td
        self.masks = masks
        self.masked_pyr = [(t * m).astype(np.uint8) for t, m in zip(td.pyramid, masks)]
        return True

    def _match_template(self, src, layer, use_simd, top=False):
        if self.masks is None:
            return super()._match_template(src, layer, use_simd, top)
        tpl = self.masked_pyr[layer]
        if self.use_simd and use_simd:
            result = O.match_template_simd(src, tpl)
        elif self.top_numerator == "cv":
            result = cv2.matchTemplate(src, tpl, cv2.TM_CCORR)
        else:
            result = O.ccorr_exact_dense(src, tpl)
        return ccoeff_denominator_masked(src, self.td, self.masks[layer], result, layer)


# ---------------- masks used by the tests ----------------
def disc_mask(w, h, frac=1.0):
    yy, xx = np.mgrid[0:h, 0:w]
    cx, cy = (w - 1) / 2.0, (h - 1) / 2.0
    r = frac * min(w, h) / 2.0
    return (((xx - cx) ** 2 + (yy - cy) ** 2) <= r * r).astype(np.uint8)


def ring_mask(w, h):
    return disc_mask(w, h) - disc_mask(w, h, 0.45)


def holed_mask(w, h):
    m = np.ones((h, w), np.uint8)
    m[h // 3:h // 3 + max(h // 4, 1), w // 4:w // 4 + max(w // 3, 1)] = 0
    m[(2 * h) // 3:(2 * h) // 3 + max(h // 8, 1), (3 * w) // 5:(3 * w) // 5 + max(w // 6, 1)] = 0
    return m


def blob_mask(w, h, seed=7):
    rng = np.random.default_rng(seed)
    f = cv2.GaussianBlur(rng.random((h, w)).astype(np.float32), (0, 0), max(min(w, h) / 8.0, 1.0))
    m = (f > np.median(f)).astype(np.uint8)
    m[h // 2 - h // 8:h // 2 + h // 8 + 1, w // 2 - w // 8:w // 2 + w // 8 + 1] = 1    # keeps every level non-empty
    return m


def corner_cut_mask(w, h):
    yy, xx = np.mgrid[0:h, 0:w]
    c = min(w, h) // 3
    m = np.ones((h, w), np.uint8)
    m[(xx + yy) < c] = 0
    m[((w - 1 - xx) + (h - 1 - yy)) < c] = 0
    m[((w - 1 - xx) + yy) < c] = 0
    return m


MASKS = {"disc": disc_mask, "ring": ring_mask, "holed": holed_mask, "blob": blob_mask, "corner_cut": corner_cut_mask}


def ccoeff_branches_masked(src, td, m, result, layer):
    """ccoeff_branches with the masked window sums: which epilogue branch every cell takes (oracle.BRANCH_*)"""
    if td.result_equal1[layer]:
        return np.full(result.shape, O.BRANCH_EQUAL1, np.int8)
    num, den = ccoeff_num_den_masked(src, td, m, result, layer)
    absn = np.abs(num)
    return np.where(den == 0, O.BRANCH_FLAT, np.where(absn < den, O.BRANCH_QUOTIENT,
                    np.where(absn < den * 1.125, O.BRANCH_CLAMP, O.BRANCH_ZERO))).astype(np.int8)


# ---------------- edge masks: the run-table cases the blobs above never produce ----------------
# Thin structures vanish down the pyramid (M_{L+1} = pyrDown(255 M_L) >= 128), so each of these keeps a solid part that is
# grown until every level of the deepest pyramid the tests use (MinReduceArea 64) keeps 4 pixels (one kept pixel is a
# flat template, which scores 1 everywhere).
EDGE_MIN_DST = 8


def _survives(m):
    top = O.get_top_layer(m.shape[1], m.shape[0], EDGE_MIN_DST)
    return all(l.sum() >= 4 for l in mask_pyramid(m, top))


def comb_mask(w, h):
    """many runs per row: columns x % 4 != 3 (runs of 3), and every third row single pixels x % 2 == 0 (runs of 1)"""
    xx = np.arange(w)[None, :]
    yy = np.arange(h)[:, None]
    return np.where(yy % 3 == 1, xx % 2 == 0, xx % 4 != 3).astype(np.uint8)


def banded_mask(w, h):
    """whole empty rows: bands of 6 empty rows (empty rows at level 1 too) between bands of kept rows, under the fewest
    kept first rows that keep every level non-empty"""
    yy = np.arange(h)
    for k in range(4, h + 1):
        m = np.repeat(((yy < k) | (yy % 12 < 4) | (yy % 12 >= 10))[:, None], w, axis=1).astype(np.uint8)
        if _survives(m):
            return m
    return np.ones((h, w), np.uint8)


def frame_mask(w, h):
    """runs at x = 0 and x = w: a frame whose sides are as thin as the pyramid allows, its middle rows two runs each"""
    for k in range(1, max(w, h)):
        m = np.ones((h, w), np.uint8)
        m[k:h - k, k:w - k] = 0
        if _survives(m):
            return m
    return np.ones((h, w), np.uint8)


def sparse_mask(w, h):
    """a sparse lattice of single pixels, plus the smallest centred block that keeps every pyramid level non-empty"""
    m = np.zeros((h, w), np.uint8)
    m[1::4, ::5] = 1
    for s in range(1, max(w, h)):
        b = m.copy()
        y0, x0 = max(h // 2 - s // 2, 0), max(w // 2 - s, 0)
        b[y0:y0 + s, x0:x0 + 2 * s] = 1
        if _survives(b):
            return b
    return np.ones((h, w), np.uint8)


EDGE_MASKS = {"comb": comb_mask, "banded": banded_mask, "frame": frame_mask, "sparse": sparse_mask}
