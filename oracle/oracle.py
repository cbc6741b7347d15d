"""CPU ORACLE -- TEST INFRASTRUCTURE ONLY.  Never imported by the product path.

A line-by-line CPU restatement of the reference's hot path
`TemplateMatcher::learnPattern` / `TemplateMatcher::match`
(/root/reference/src/TemplateMatcher.cpp, /root/reference/include/DataStructures.h).

Every OpenCV call of the reference is made through the same library (`cv2`, 4.13.0 in
this image) so the third-party arithmetic is the reference's own; the reference's one
hand-written SIMD routine (`IM_Conv_SIMD`, src/TemplateMatcher.cpp:461-483, plus the
row-ordered float accumulation of `MatchTemplate`, :496-510) is restated either in
numpy (exact int row sums + strict float32 chain) or by `oracle/ncc_rowdot.c` (SSE2).

Parity status: the reference ships no tests/golden vectors (SURVEY.md section 4), so this
oracle is pinned against (a) the README/Result-image known answers
(Src6/Dst6 -> 15 targets, Src3/Dst3 -> 36, Src8/Dst8 -> 3), (b) the reference's own
`IM_Conv_SIMD` source compiled from /root/reference into oracle/_ref (see
oracle/build_ref.sh) and (c) cv2 itself for every OpenCV model in oracle/models.py.
The full `match()` cannot be compiled here (needs OpenCV C++ and Qt headers, absent).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg
may import this module.
"""
from __future__ import annotations

import ctypes
import math
import os
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np

try:  # cv2 is the reference's own third-party dependency (OpenCV)
    import cv2
except Exception as e:  # pragma: no cover
    cv2 = None
    _cv2_err = e

VISION_TOLERANCE = 0.0000001           # DataStructures.h:10
D2R = math.pi / 180.0                  # DataStructures.h:11
R2D = 180.0 / math.pi                  # DataStructures.h:12
MATCH_CANDIDATE_NUM = 5                # DataStructures.h:13
DBL_EPSILON = 2.220446049250313e-16
FLT_EPSILON = 1.1920928955078125e-07

f32 = np.float32


# --------------------------------------------------------------------------------------
# optional C helper (SSE2 restatement of IM_Conv_SIMD + the MatchTemplate SIMD loop)
# --------------------------------------------------------------------------------------
_HERE = os.path.dirname(os.path.abspath(__file__))
_rowdot_lib = None


def _load_rowdot():
    global _rowdot_lib
    if _rowdot_lib is not None:
        return _rowdot_lib
    path = os.path.join(_HERE, "libncc_rowdot.so")
    if os.path.exists(path):
        lib = ctypes.CDLL(path)
        lib.oracle_match_template_simd.argtypes = [
            ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
            ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        lib.oracle_match_template_simd.restype = None
        _rowdot_lib = lib
    else:
        _rowdot_lib = False
    return _rowdot_lib


# --------------------------------------------------------------------------------------
# data records (DataStructures.h:16-115)
# --------------------------------------------------------------------------------------
@dataclass
class TemplData:                      # s_TemplData, DataStructures.h:16-55
    pyramid: List[np.ndarray] = field(default_factory=list)
    templ_mean: List[float] = field(default_factory=list)
    templ_norm: List[float] = field(default_factory=list)
    inv_area: List[float] = field(default_factory=list)
    result_equal1: List[bool] = field(default_factory=list)
    learned: bool = False
    border_color: int = 0


@dataclass
class MatchParameter:                 # s_MatchParameter, DataStructures.h:58-94
    pt: tuple = (0.0, 0.0)            # cv::Point2d
    score: float = 0.0
    angle: float = 0.0
    angle_start: float = 0.0
    angle_end: float = 0.0
    rect: object = None               # cv::RotatedRect -> ((cx,cy),(w,h),angle)
    deleted: bool = False
    vec_result: Optional[np.ndarray] = None   # [3][3] indexed [x+1][y+1]
    pos_on_border: bool = False
    cand_id: int = -1                 # oracle-only: index in the sorted top-layer list


@dataclass
class SingleTargetMatch:              # s_SingleTargetMatch, DataStructures.h:97-115
    ptLT: tuple
    ptRT: tuple
    ptRB: tuple
    ptLB: tuple
    ptCenter: tuple
    angle: float
    score: float


# --------------------------------------------------------------------------------------
# small helpers that mirror C++ float/double semantics
# --------------------------------------------------------------------------------------
def pt_rotate_pt2f(pt, org, angle_rad):
    """ptRotatePt2f, src/TemplateMatcher.cpp:971-982.  pt/org are float32 pairs."""
    px, py = float(f32(pt[0])), float(f32(pt[1]))
    ox, oy = float(f32(org[0])), float(f32(org[1]))
    d_height = float(f32(oy * 2))          # float * int -> float, then widened
    dy1 = d_height - py
    dy2 = d_height - oy
    c, s = math.cos(angle_rad), math.sin(angle_rad)
    dx = (px - ox) * c - (dy1 - oy) * s + ox
    dy = (px - ox) * s + (dy1 - oy) * c + dy2
    dy = -dy + d_height
    return (f32(dx), f32(dy))


def get_top_layer(w, h, min_dst_length):
    """getTopLayer, src/TemplateMatcher.cpp:445-455."""
    top = 0
    min_area = min_dst_length * min_dst_length
    area = w * h
    while area > min_area:
        area //= 4
        top += 1
    return top


def build_pyramid(img, maxlevel):
    """cv::buildPyramid (src/TemplateMatcher.cpp:55,124): level 0 = img, then pyrDown chain."""
    out = [img]
    for _ in range(maxlevel):
        out.append(cv2.pyrDown(out[-1]))
    return out


def get_best_rotation_size(size_src, size_dst, angle_deg):
    """getBestRotationSize, src/TemplateMatcher.cpp:901-969.  sizes are (w, h)."""
    sw, sh = size_src
    dw, dh = size_dst
    a_rad = angle_deg * D2R
    center = (f32(f32(sw - 1) / f32(2.0)), f32(f32(sh - 1) / f32(2.0)))
    pts = [(0, 0), (0, sh - 1), (sw - 1, sh - 1), (sw - 1, 0)]
    rot = [pt_rotate_pt2f((f32(p[0]), f32(p[1])), center, a_rad) for p in pts]
    top_y = max(r[1] for r in rot)
    bottom_y = min(r[1] for r in rot)
    right_x = max(r[0] for r in rot)
    left_x = min(r[0] for r in rot)

    ang = angle_deg
    if ang > 360:
        ang -= 360
    elif ang < 0:
        ang += 360
    if abs(abs(ang) - 90) < VISION_TOLERANCE or abs(abs(ang) - 270) < VISION_TOLERANCE:
        return (sh, sw)
    if abs(ang) < VISION_TOLERANCE or abs(abs(ang) - 180) < VISION_TOLERANCE:
        return (sw, sh)
    d = ang
    if 0 < d < 90:
        pass
    elif 90 < d < 180:
        d -= 90
    elif 180 < d < 270:
        d -= 180
    elif 270 < d < 360:
        d -= 270
    # else: "Unkown" branch -- falls through with d unchanged (:948-952)
    fh1 = f32(dw * math.sin(d * D2R) * math.cos(d * D2R))
    fh2 = f32(dh * math.sin(d * D2R) * math.cos(d * D2R))
    half_h = int(math.ceil(f32(f32(top_y - center[1]) - fh1)))
    half_w = int(math.ceil(f32(f32(right_x - center[0]) - fh2)))
    rw, rh = half_w * 2, half_h * 2
    wrong = (dw < rw and dh > rh) or (dw > rw and dh < rh) or (dw * dh > rw * rh)
    if wrong:
        rw = int(float(f32(right_x - left_x)) + 0.5)
        rh = int(float(f32(top_y - bottom_y)) + 0.5)
    return (rw, rh)


def ccorr_exact_rows(src, tpl):
    """Exact per-template-row s32 dot products for every result cell.

    Returns int64 array [R, C, th] with rows[r, c, tr] = sum_tc T[tr,tc]*S[r+tr, c+tc]
    (== IM_Conv_SIMD(T row tr, S row r+tr at col c, tw), src/TemplateMatcher.cpp:461-483)."""
    th, tw = tpl.shape
    R = src.shape[0] - th + 1
    C = src.shape[1] - tw + 1
    t = tpl.astype(np.int64)
    out = np.empty((R, C, th), np.int64)
    s = src.astype(np.int64)
    for r in range(R):
        for c in range(C):
            out[r, c, :] = (t * s[r:r + th, c:c + tw]).sum(axis=1)
    return out


def match_template_simd_numpy(src, tpl):
    """The SIMD branch of MatchTemplate (src/TemplateMatcher.cpp:487-512): per result cell a
    float32 accumulator that receives the exact int row sums in template-row order."""
    rows = ccorr_exact_rows(src, tpl)
    R, C, th = rows.shape
    acc = np.zeros((R, C), f32)
    rows_f = rows.astype(f32)          # int -> float conversion of each row sum (rounds >= 2^24)
    for tr in range(th):
        acc = (acc + rows_f[:, :, tr]).astype(f32)
    return acc


def match_template_simd(src, tpl):
    lib = _load_rowdot()
    if lib:
        src = np.ascontiguousarray(src)
        tpl = np.ascontiguousarray(tpl)
        R = src.shape[0] - tpl.shape[0] + 1
        C = src.shape[1] - tpl.shape[1] + 1
        out = np.zeros((R, C), f32)
        lib.oracle_match_template_simd(src.ctypes.data, src.shape[1], src.shape[0],
                                       tpl.ctypes.data, tpl.shape[1], tpl.shape[0],
                                       out.ctypes.data)
        return out
    return match_template_simd_numpy(src, tpl)


def ccorr_exact_dense(src, tpl):
    """Exact integer TM_CCORR map (sum over the whole template), cast to float32.
    Used for the top layer when top_numerator == 'exact' (SURVEY.md section 7.4)."""
    th, tw = tpl.shape
    R = src.shape[0] - th + 1
    C = src.shape[1] - tw + 1
    s = src.astype(np.int64)
    acc = np.zeros((R, C), np.int64)
    for i in range(th):
        for j in range(tw):
            t = int(tpl[i, j])
            if t:
                acc += t * s[i:i + R, j:j + C]
    return acc.astype(f32)


def ccoeff_num_den(src, td: TemplData, result, layer):
    """The centred numerator and the denominator of every cell of CCOEFF_Denominator (float64, same op order);
    den == 0 where the window is flat."""
    tpl = td.pyramid[layer]
    th, tw = tpl.shape
    s, q = cv2.integral2(src, sdepth=cv2.CV_64F, sqdepth=cv2.CV_64F)
    R, C = result.shape
    t = s[0:R, 0:C] - s[0:R, tw:tw + C] - s[th:th + R, 0:C] + s[th:th + R, tw:tw + C]
    num = result.astype(np.float64)
    wnd_mean2 = (t * t) * td.inv_area[layer]
    num = num - t * td.templ_mean[layer]
    t2 = q[0:R, 0:C] - q[0:R, tw:tw + C] - q[th:th + R, 0:C] + q[th:th + R, tw:tw + C]
    wnd_sum2 = t2
    diff2 = np.maximum(wnd_sum2 - wnd_mean2, 0.0)
    den = np.where(diff2 <= np.minimum(0.5, 10 * FLT_EPSILON * wnd_sum2), 0.0,
                   np.sqrt(diff2) * td.templ_norm[layer])
    return num, den


# outcomes of the CCOEFF_NORMED epilogue per cell (ccoeff_branches)
BRANCH_FLAT, BRANCH_CLAMP, BRANCH_QUOTIENT, BRANCH_ZERO, BRANCH_EQUAL1 = range(5)


def ccoeff_branches(src, td: TemplData, result, layer):
    """Which branch of the epilogue every cell takes: den == 0 (score 0), den <= |num| < 1.125 den (score +-1),
    |num| < den (num / den), |num| >= 1.125 den > 0 (score 0), or a flat template (score 1)."""
    if td.result_equal1[layer]:
        return np.full(result.shape, BRANCH_EQUAL1, np.int8)
    num, den = ccoeff_num_den(src, td, result, layer)
    absn = np.abs(num)
    return np.where(den == 0, BRANCH_FLAT, np.where(absn < den, BRANCH_QUOTIENT,
                    np.where(absn < den * 1.125, BRANCH_CLAMP, BRANCH_ZERO))).astype(np.int8)


def ccoeff_denominator(src, td: TemplData, result, layer):
    """CCOEFF_Denominator, src/TemplateMatcher.cpp:527-598 (vectorised, same op order)."""
    if td.result_equal1[layer]:
        result[:] = 1
        return result
    num, den = ccoeff_num_den(src, td, result, layer)
    absn = np.abs(num)
    with np.errstate(divide="ignore", invalid="ignore"):
        out = np.where(absn < den, num / den,
                       np.where(absn < den * 1.125, np.where(num > 0, 1.0, -1.0), 0.0))
    result[:] = out.astype(f32)
    return result


# ----------------------------------------------------------------------------------
# s_BlockMax (Qt flavour), DataStructures.h:118-245
# ----------------------------------------------------------------------------------
def _min_max_loc(mat):
    """cv::minMaxLoc max: value + first location in row-major scan order -> (val, (x, y))."""
    idx = int(np.argmax(mat))          # numpy argmax returns the first maximum (row-major)
    y, x = divmod(idx, mat.shape[1])
    return float(mat[y, x]), (x, y)


class BlockMax:
    def __init__(self, mat, size_tpl):
        self.mat = mat
        bw, bh = size_tpl
        rows, cols = mat.shape
        ncol, nrow = cols // bw, rows // bh
        self.blocks = []               # [x, y, w, h, max, (px, py)]

        def add(x, y, w, h):
            v, (mx, my) = _min_max_loc(mat[y:y + h, x:x + w])
            self.blocks.append([x, y, w, h, v, (x + mx, y + my)])

        for y in range(nrow):
            for x in range(ncol):
                add(x * bw, y * bh, bw, bh)
        if ncol * bw < cols:
            add(ncol * bw, 0, cols - ncol * bw, rows)
        if nrow * bh < rows:
            if ncol * bw > 0:           # an empty cv::Mat ROI would throw in minMaxLoc
                add(0, nrow * bh, ncol * bw, rows - nrow * bh)
        if ncol * bw < cols and nrow * bh < rows:
            add(ncol * bw, nrow * bh, cols - ncol * bw, rows - nrow * bh)

    def update_max(self, rx, ry, rw, rh):
        for b in self.blocks:
            x0, y0 = max(b[0], rx), max(b[1], ry)
            x1, y1 = min(b[0] + b[2], rx + rw), min(b[1] + b[3], ry + rh)
            if x1 > x0 and y1 > y0:    # (block.rect & rectIgnore).area() > 0
                v, (mx, my) = _min_max_loc(self.mat[b[1]:b[1] + b[3], b[0]:b[0] + b[2]])
                b[4], b[5] = v, (b[0] + mx, b[1] + my)

    def get_max(self):
        if not self.blocks:
            return -1.0, (-1, -1)
        best = self.blocks[0]
        for b in self.blocks[1:]:      # std::max_element: first maximum
            if best[4] < b[4]:
                best = b
        return best[4], best[5]


class BlockMaxMFC(BlockMax):
    """s_BlockMax of the upstream MFC dialog (MatchTool/MatchToolDlg.h:89-213): blocks of 2x the template size,
    right strip when the width leaves a residue, bottom strip over the regular columns when both dimensions do and
    over the full width otherwise, no corner block; GetMaxValueLoc keeps the LAST maximal block (>=, :206) and an
    empty table (less than one block in a dimension) searches the whole map (:196-200)."""

    def __init__(self, mat, size_tpl):
        self.mat = mat
        bw, bh = 2 * size_tpl[0], 2 * size_tpl[1]
        rows, cols = mat.shape
        ncol, nrow = cols // bw, rows // bh
        self.blocks = []
        if ncol == 0 or nrow == 0:
            return

        def add(x, y, w, h):
            v, (mx, my) = _min_max_loc(mat[y:y + h, x:x + w])
            self.blocks.append([x, y, w, h, v, (x + mx, y + my)])

        for y in range(nrow):
            for x in range(ncol):
                add(x * bw, y * bh, bw, bh)
        hres, vres = cols % bw != 0, rows % bh != 0
        if hres and vres:
            add(ncol * bw, 0, cols - ncol * bw, rows)
            add(0, nrow * bh, ncol * bw, rows - nrow * bh)
        elif hres:
            add(ncol * bw, 0, cols - ncol * bw, rows)
        elif vres:                      # upstream's else-branch; with no residue at all it would scan an empty Mat
            add(0, nrow * bh, cols, rows - nrow * bh)

    def get_max(self):
        if not self.blocks:
            return _min_max_loc(self.mat)
        best = self.blocks[0]
        for b in self.blocks[1:]:
            if b[4] >= best[4]:
                best = b
        return best[4], best[5]


def _trunc(v):
    return int(v)                       # C++ double -> int truncation toward zero


def _paint(mat, x, y, w, h):
    """cv::rectangle(mat, Rect(x,y,w,h), -1, FILLED): fills [x, x+w) x [y, y+h) clipped to
    the image; an empty Rect (w<=0 or h<=0) paints nothing (pinned in tests/test_oracle_models.py)."""
    cv2.rectangle(mat, (x, y, w, h), -1.0, cv2.FILLED)


# --------------------------------------------------------------------------------------
# the matcher
# --------------------------------------------------------------------------------------
class OracleMatcher:
    """Restatement of TemplateMatcher (include/TemplateMatcher.h:9-90)."""

    def __init__(self):                                   # src/TemplateMatcher.cpp:28-39
        self.max_pos = 70
        self.max_overlap = 0.0
        self.score = 0.7
        self.tolerance_angle = 0.0
        self.min_reduce_area = 256
        self.use_simd = True
        self.sub_pixel = False
        self.last_time = 0.0
        self.td = TemplData()
        # MFC-only modes of the upstream dialog (MatchTool/MatchToolDlg.cpp), off in the Qt port
        self.tolerance_range = None       # (t1, t2, t3, t4): two angle ranges, :805-816
        self.stop_layer1 = False          # m_bStopLayer1: stop the descent at layer 1, :936
        self.bitwise_not = False          # m_ckBitwiseNot: match on 255 - src, :788-794
        self.mfc_compat = False           # result convention of :1085-1116 (angle sign/wrap, TargetNum truncation)
        # oracle-only switches
        self.top_numerator = "exact"      # "exact" (integer) | "cv" (cv2.matchTemplate)
        self.trace = None                 # dict filled with intermediates when not None

    # -- learnPattern, src/TemplateMatcher.cpp:45-95 ---------------------------------
    def learn_pattern(self, tpl):
        if tpl is None or tpl.size == 0:
            return False
        self.td = TemplData()
        top = get_top_layer(tpl.shape[1], tpl.shape[0], int(math.sqrt(float(self.min_reduce_area))))
        self.td.pyramid = build_pyramid(np.ascontiguousarray(tpl), top)
        mean_color = cv2.mean(tpl)[0]
        self.td.border_color = 255 if mean_color < 128 else 0
        for lvl in self.td.pyramid:
            inv_area = 1.0 / (float(lvl.shape[0]) * lvl.shape[1])
            mean, sdv = cv2.meanStdDev(lvl)
            m, s = float(mean[0, 0]), float(sdv[0, 0])
            norm = s * s
            self.td.result_equal1.append(norm < DBL_EPSILON)
            norm = math.sqrt(norm)
            norm /= math.sqrt(inv_area)
            self.td.inv_area.append(inv_area)
            self.td.templ_mean.append(m)
            self.td.templ_norm.append(norm)
        self.td.learned = True
        return True

    # -- MatchTemplate, src/TemplateMatcher.cpp:485-525 ------------------------------
    def _match_template(self, src, layer, use_simd, top=False):
        tpl = self.td.pyramid[layer]
        if self.use_simd and use_simd:
            result = match_template_simd(src, tpl)
        else:
            if self.top_numerator == "cv":
                result = cv2.matchTemplate(src, tpl, cv2.TM_CCORR)
            else:
                result = ccorr_exact_dense(src, tpl)
        return ccoeff_denominator(src, self.td, result, layer)

    # -- getRotatedROI, src/TemplateMatcher.cpp:1074-1090 ----------------------------
    @staticmethod
    def _get_rotated_roi(src, size, pt_lt, angle):
        a_rad = angle * D2R
        ptc = (f32(f32(src.shape[1] - 1) / f32(2.0)), f32(f32(src.shape[0] - 1) / f32(2.0)))
        lt_rot = pt_rotate_pt2f(pt_lt, ptc, a_rad)
        m = cv2.getRotationMatrix2D((float(ptc[0]), float(ptc[1])), angle, 1)
        m[0, 2] -= float(f32(lt_rot[0] - f32(3)))
        m[1, 2] -= float(f32(lt_rot[1] - f32(3)))
        return cv2.warpAffine(src, m, (size[0] + 6, size[1] + 6))

    # -- getNextMaxLoc (plain), src/TemplateMatcher.cpp:1196-1206 --------------------
    def _next_max_loc(self, result, pt, size_tpl):
        ov = self.max_overlap
        sx = _trunc(pt[0] - size_tpl[0] * (1 - ov))
        sy = _trunc(pt[1] - size_tpl[1] * (1 - ov))
        _paint(result, sx, sy, _trunc(2 * size_tpl[0] * (1 - ov)), _trunc(2 * size_tpl[1] * (1 - ov)))
        return _min_max_loc(result)

    # -- getNextMaxLoc (block), src/TemplateMatcher.cpp:1208-1221 --------------------
    def _next_max_loc_block(self, result, pt, size_tpl, bm: BlockMax):
        ov = self.max_overlap
        sx = _trunc(pt[0] - size_tpl[0] * (1 - ov))
        sy = _trunc(pt[1] - size_tpl[1] * (1 - ov))
        rw = _trunc(2 * size_tpl[0] * (1 - ov))
        rh = _trunc(2 * size_tpl[1] * (1 - ov))
        _paint(result, sx, sy, rw, rh)
        bm.update_max(sx, sy, rw, rh)
        return bm.get_max()

    # -- greedy peak list of one top-layer score map, src/TemplateMatcher.cpp:179-210 --------
    def top_picks(self, result, size_pat, thresh, cal_by_block):
        """Returns [((x, y), value), ...]; `result` is painted in place like the reference does."""
        picks = []
        if cal_by_block:
            bm = BlockMaxMFC(result, size_pat) if self.mfc_compat else BlockMax(result, size_pat)
            val, loc = bm.get_max()
            if val < thresh:
                return picks
            picks.append((loc, val))
            for _ in range(self.max_pos + MATCH_CANDIDATE_NUM - 1):
                val, loc = self._next_max_loc_block(result, loc, size_pat, bm)
                if val < thresh:
                    break
                picks.append((loc, val))
        else:
            val, loc = _min_max_loc(result)
            if val < thresh:
                return picks
            picks.append((loc, val))
            for _ in range(self.max_pos + MATCH_CANDIDATE_NUM - 1):
                val, loc = self._next_max_loc(result, loc, size_pat)
                if val < thresh:
                    break
                picks.append((loc, val))
        return picks

    def top_angles(self, top):
        """angle schedule, src/TemplateMatcher.cpp:130-144."""
        tp = self.td.pyramid[top]
        step = math.atan(2.0 / max(tp.shape[1], tp.shape[0])) * R2D
        angles = []
        if self.tolerance_range is not None:                       # MatchToolDlg.cpp:805-816
            t1, t2, t3, t4 = self.tolerance_range
            a = t1
            while a < t2 + step:
                angles.append(a)
                a += step
            a = t3
            while a < t4 + step:
                angles.append(a)
                a += step
        elif self.tolerance_angle < VISION_TOLERANCE:
            angles.append(0.0)
        else:
            a = 0.0
            while a < self.tolerance_angle + step:
                angles.append(a)
                a += step
            a = -step
            while a > -self.tolerance_angle - step:
                angles.append(a)
                a -= step
        return step, angles

    # -- match, src/TemplateMatcher.cpp:97-437 ---------------------------------------
    def match(self, src) -> List[SingleTargetMatch]:
        td = self.td
        tr = self.trace
        if src is None or src.size == 0 or not td.learned:
            return []
        t0w, t0h = td.pyramid[0].shape[1], td.pyramid[0].shape[0]
        sw, sh = src.shape[1], src.shape[0]
        if (t0w < sw and t0h > sh) or (t0w > sw and t0h < sh):
            return []
        if t0w * t0h > sw * sh:
            return []
        top = get_top_layer(t0w, t0h, int(math.sqrt(float(self.min_reduce_area))))
        if top >= len(td.pyramid):
            raise RuntimeError("MinReduceArea changed after learnPattern (reference would index out of range)")
        if self.tolerance_range is not None and (self.tolerance_range[0] >= self.tolerance_range[1] or
                                                 self.tolerance_range[2] >= self.tolerance_range[3]):
            return []                                              # "left value must be smaller", :807-811
        if self.bitwise_not:
            src = 255 - src
        src_pyr = build_pyramid(np.ascontiguousarray(src), top)
        if tr is not None:
            tr["src_pyr"] = src_pyr

        step, angles = self.top_angles(top)
        top_src = src_pyr[top]
        tsw, tsh = top_src.shape[1], top_src.shape[0]
        center = (f32(f32(tsw - 1) / f32(2.0)), f32(f32(tsh - 1) / f32(2.0)))
        layer_score = [self.score]
        for _ in range(top):
            layer_score.append(layer_score[-1] * 0.9)
        tp = td.pyramid[top]
        size_pat = (tp.shape[1], tp.shape[0])
        cal_by_block = ((tsw * tsh) // (size_pat[0] * size_pat[1]) > 500) and self.max_pos > 10

        cands: List[MatchParameter] = []
        if tr is not None:
            tr["angles"] = angles
            tr["top"] = []
        for ang in angles:
            m = cv2.getRotationMatrix2D((float(center[0]), float(center[1])), ang, 1)
            size_best = get_best_rotation_size((tsw, tsh), size_pat, ang)
            ftx = f32(f32(size_best[0] - 1) / f32(2.0)) - center[0]
            fty = f32(f32(size_best[1] - 1) / f32(2.0)) - center[1]
            ftx, fty = f32(ftx), f32(fty)
            m[0, 2] += float(ftx)
            m[1, 2] += float(fty)
            rot = cv2.warpAffine(top_src, m, size_best, flags=cv2.INTER_LINEAR,
                                 borderMode=cv2.BORDER_CONSTANT, borderValue=(td.border_color,))
            result = self._match_template(rot, top, False, top=True)
            if tr is not None:
                tr["top"].append(dict(angle=ang, size=size_best, rot=rot.copy(), score=result.copy(),
                                      M=m.copy(), picks=[]))
            picks = self.top_picks(result, size_pat, layer_score[top], cal_by_block)
            for loc, val in picks:
                pt = (f32(f32(loc[0]) - ftx), f32(f32(loc[1]) - fty))
                cands.append(MatchParameter(pt=(float(pt[0]), float(pt[1])), score=val, angle=ang))
            if tr is not None:
                tr["top"][-1]["picks"] = picks

        # std::sort by score desc (:214) -- unstable in C++; the oracle uses a stable sort
        cands.sort(key=lambda c: -c.score)
        for i, c in enumerate(cands):
            c.cand_id = i
        if tr is not None:
            tr["cands"] = [(c.pt, c.score, c.angle) for c in cands]
            tr["refine"] = []

        dst_w, dst_h = size_pat
        stop_layer = 1 if self.stop_layer1 else 0
        all_res: List[MatchParameter] = []
        for ci, cand in enumerate(cands):
            r_angle = -cand.angle * D2R
            pt_lt = pt_rotate_pt2f((f32(cand.pt[0]), f32(cand.pt[1])), center, r_angle)
            a_step = math.atan(2.0 / max(dst_w, dst_h)) * R2D
            cand.angle_start = cand.angle - a_step
            cand.angle_end = cand.angle + a_step
            if top <= stop_layer:
                k = 1 if top == 0 else 2
                cand.pt = (float(f32(pt_lt[0] * k)), float(f32(pt_lt[1] * k)))
                all_res.append(cand)
                continue
            for layer in range(top - 1, stop_layer - 1, -1):
                tpl_l = td.pyramid[layer]
                a_step = math.atan(2.0 / max(tpl_l.shape[1], tpl_l.shape[0])) * R2D
                matched = cand.angle
                if self.tolerance_range is None and self.tolerance_angle < VISION_TOLERANCE:
                    l_angles = [0.0]
                else:
                    l_angles = [matched + a_step * i for i in (-1, 0, 1)]
                src_l = src_pyr[layer]
                src_center = (f32(f32(src_l.shape[1] - 1) / f32(2.0)), f32(f32(src_l.shape[0] - 1) / f32(2.0)))
                new = []
                best_idx, big = 0, -1.0
                pt_lt2 = (f32(pt_lt[0] * 2), f32(pt_lt[1] * 2))
                for j, la in enumerate(l_angles):
                    roi = self._get_rotated_roi(src_l, (tpl_l.shape[1], tpl_l.shape[0]), pt_lt2, la)
                    result = self._match_template(roi, layer, True)
                    val, loc = _min_max_loc(result)
                    p = MatchParameter(pt=(float(loc[0]), float(loc[1])), score=val, angle=la)
                    if p.score > big:
                        best_idx, big = j, p.score
                    if loc[0] == 0 or loc[1] == 0 or loc[0] == result.shape[1] - 1 or loc[1] == result.shape[0] - 1:
                        p.pos_on_border = True
                    if not p.pos_on_border:
                        vr = np.zeros((3, 3))
                        for y in (-1, 0, 1):
                            for x in (-1, 0, 1):
                                vr[x + 1][y + 1] = result[loc[1] + y, loc[0] + x]
                        p.vec_result = vr
                    new.append(p)
                    if tr is not None:
                        tr["refine"].append(dict(cand=ci, layer=layer, j=j, angle=la, roi=roi,
                                                 score=result.copy(), loc=loc, val=val,
                                                 pt_lt2=(float(pt_lt2[0]), float(pt_lt2[1]))))
                if new[best_idx].score < layer_score[layer]:
                    break
                if (self.sub_pixel and layer == 0 and not new[best_idx].pos_on_border
                        and best_idx != 0 and best_idx != 2):
                    nx, ny, na = self._sub_pix_estimation(new, a_step, best_idx)
                    new[best_idx].pt = (nx, ny)
                    new[best_idx].angle = na
                new_angle = new[best_idx].angle
                padding = pt_rotate_pt2f(pt_lt2, src_center, new_angle * D2R)
                padding = (f32(padding[0] - f32(3)), f32(padding[1] - f32(3)))
                pt = (f32(new[best_idx].pt[0] + float(padding[0])), f32(new[best_idx].pt[1] + float(padding[1])))
                pt = pt_rotate_pt2f(pt, src_center, -new_angle * D2R)
                if layer == stop_layer:
                    k = 1 if stop_layer == 0 else 2
                    new[best_idx].pt = (float(f32(pt[0] * k)), float(f32(pt[1] * k)))
                    new[best_idx].cand_id = cand.cand_id
                    all_res.append(new[best_idx])
                else:
                    cand.angle = new_angle
                    cand.angle_start = cand.angle - a_step / 2
                    cand.angle_end = cand.angle + a_step / 2
                    pt_lt = pt

        if tr is not None:
            tr["all_res"] = [(r.pt, r.score, r.angle, r.cand_id) for r in all_res]
        # filterWithScore, :984-1000
        all_res.sort(key=lambda c: -c.score)
        for i, r in enumerate(all_res):
            if r.score < self.score:
                all_res = all_res[:i]
                break

        dst_w = td.pyramid[stop_layer].shape[1] * (1 if stop_layer == 0 else 2)
        dst_h = td.pyramid[stop_layer].shape[0] * (1 if stop_layer == 0 else 2)
        for r in all_res:
            lt, rt, lb, rb = self._corners(r, dst_w, dst_h)
            r.rect = cv2.RotatedRect((float(lt[0]), float(lt[1])), (float(rt[0]), float(rt[1])),
                                     (float(rb[0]), float(rb[1])))
        all_res = self._filter_with_rotated_rect(all_res, self.max_overlap)
        all_res.sort(key=lambda c: -c.score)
        if not all_res:
            return []
        iw, ih = td.pyramid[0].shape[1], td.pyramid[0].shape[0]
        out = []
        if self.mfc_compat:                                        # MatchToolDlg.cpp:1085-1116
            for i, r in enumerate(all_res):
                a = -r.angle * D2R
                ltx, lty = float(f32(r.pt[0])), float(f32(r.pt[1]))   # pt holds float values
                rt = (ltx + iw * math.cos(a), lty - iw * math.sin(a))
                lb = (ltx + ih * math.sin(a), lty + ih * math.cos(a))
                rb = (rt[0] + ih * math.sin(a), rt[1] + ih * math.cos(a))
                ang = -r.angle
                if ang < -180:
                    ang += 360
                if ang > 180:
                    ang -= 360
                out.append(SingleTargetMatch(ptLT=(ltx, lty), ptRT=rt, ptRB=rb, ptLB=lb,
                                             ptCenter=((ltx + rt[0] + rb[0] + lb[0]) / 4, (lty + rt[1] + rb[1] + lb[1]) / 4),
                                             angle=ang, score=r.score))
                if i + 1 == self.max_pos:
                    break
            return out
        for r in all_res:
            lt, rt, lb, rb = self._corners(r, iw, ih)
            four = f32(4.0)
            cx = f32(f32(f32(f32(lt[0] + rt[0]) + lb[0]) + rb[0]) / four)
            cy = f32(f32(f32(f32(lt[1] + rt[1]) + lb[1]) + rb[1]) / four)
            out.append(SingleTargetMatch(
                ptLT=(float(lt[0]), float(lt[1])), ptRT=(float(rt[0]), float(rt[1])),
                ptRB=(float(rb[0]), float(rb[1])), ptLB=(float(lb[0]), float(lb[1])),
                ptCenter=(float(cx), float(cy)), angle=r.angle, score=r.score))
        return out

    @staticmethod
    def _corners(r: MatchParameter, w, h):
        """corner construction, src/TemplateMatcher.cpp:380-388 and :412-416 (float math)."""
        ra = -r.angle * D2R
        c, s = f32(math.cos(ra)), f32(math.sin(ra))
        lt = (f32(r.pt[0]), f32(r.pt[1]))
        fw, fh = f32(w), f32(h)
        rt = (f32(lt[0] + f32(fw * c)), f32(lt[1] - f32(fw * s)))
        lb = (f32(lt[0] + f32(fh * s)), f32(lt[1] + f32(fh * c)))
        rb = (f32(rt[0] + f32(fh * s)), f32(rt[1] + f32(fh * c)))
        return lt, rt, lb, rb

    # -- sortPtWithCenter, src/TemplateMatcher.cpp:1093-1131 (quirks kept) ------------
    @staticmethod
    def _sort_pt_with_center(pts):
        n = len(pts)
        cx, cy = f32(0), f32(0)
        for p in pts:
            cx, cy = f32(cx + p[0]), f32(cy + p[1])
        cx, cy = f32(cx / f32(n)), f32(cy / f32(n))
        keyed = []
        for p in pts:
            vx, vy = f32(p[0] - cx), f32(p[1] - cy)
            norm = f32(f32(vx * vx) + f32(vy * vy))      # squared norm (reference quirk :1108)
            dot = vx
            with np.errstate(all="ignore"):
                ratio = float(f32(dot / norm)) if norm != 0 else float("nan")
            if vy < 0:
                key = (math.acos(ratio) if -1 <= ratio <= 1 else float("nan")) * R2D
            elif vy > 0:
                key = 360 - (math.acos(ratio) if -1 <= ratio <= 1 else float("nan")) * R2D
            else:
                key = 0 if f32(vx - cx) > 0 else 180  # reference quirk :1121
            keyed.append((key, p))
        keyed.sort(key=lambda kp: kp[0])
        return [kp[1] for kp in keyed]

    # -- filterWithRotatedRect, src/TemplateMatcher.cpp:1133-1194 ---------------------
    def _filter_with_rotated_rect(self, vec: List[MatchParameter], max_overlap):
        n = len(vec)
        for i in range(n - 1):
            if vec[i].deleted:
                continue
            for j in range(i + 1, n):
                if vec[j].deleted:
                    continue
                r1, r2 = vec[i].rect, vec[j].rect
                typ, inter = cv2.rotatedRectangleIntersection(_rr_tuple(r1), _rr_tuple(r2))
                if typ == cv2.INTERSECT_NONE:
                    continue
                if typ == cv2.INTERSECT_FULL:
                    d = j if vec[i].score >= vec[j].score else i
                    vec[d].deleted = True
                else:
                    if inter is None or len(inter) < 3:
                        continue
                    pts = [(f32(p[0][0]), f32(p[0][1])) for p in inter]
                    pts = self._sort_pt_with_center(pts)
                    area = cv2.contourArea(np.array(pts, f32).reshape(-1, 1, 2))
                    ratio = area / (float(f32(_rr_tuple(r1)[1][0]) * f32(_rr_tuple(r1)[1][1])))
                    if ratio > max_overlap:
                        d = j if vec[i].score >= vec[j].score else i
                        vec[d].deleted = True
        return [v for v in vec if not v.deleted]

    # -- subPixEstimation, src/TemplateMatcher.cpp:1002-1072 -------------------------
    @staticmethod
    def _sub_pix_estimation(new, a_step, best):
        A = np.zeros((27, 10))
        S = np.zeros((27, 1))
        xm, ym, tm = new[best].pt[0], new[best].pt[1], new[best].angle
        row = 0
        for theta in range(3):
            for y in (-1, 0, 1):
                for x in (-1, 0, 1):
                    dx, dy = xm + x, ym + y
                    dt = (tm + (theta - 1) * a_step) * D2R
                    A[row] = [dx * dx, dy * dy, dt * dt, dx * dy, dx * dt, dy * dt, dx, dy, dt, 1.0]
                    vr = new[best + (theta - 1)].vec_result
                    S[row, 0] = vr[x + 1][y + 1] if vr is not None else 0.0
                    row += 1
        ata = cv2.gemm(A, A, 1, None, 0, flags=cv2.GEMM_1_T)
        z = cv2.gemm(cv2.gemm(cv2.invert(ata)[1], A, 1, None, 0, flags=cv2.GEMM_2_T), S, 1, None, 0).ravel()
        k1 = np.array([[2 * z[0], z[3], z[4]], [z[3], 2 * z[1], z[5]], [z[4], z[5], 2 * z[2]]])
        k2 = np.array([[-z[6]], [-z[7]], [-z[8]]])
        # matK1.inv() * matK2 (:1066): OpenCV's MatExpr layer turns inv(A) * B into cv::solve(A, B, DECOMP_LU)
        # (modules/core/src/matop.cpp, MatOp_Invert::matmul), not invert-then-multiply
        ok, d = cv2.solve(k1, k2, flags=cv2.DECOMP_LU)
        if not ok:
            d = np.zeros((3, 1))
        return float(d[0, 0]), float(d[1, 0]), float(d[2, 0]) * R2D


def _rr_tuple(r):
    if isinstance(r, tuple):
        return r
    return ((r.center[0], r.center[1]), (r.size[0], r.size[1]), r.angle)


# --------------------------------------------------------------------------------------
# multi-template "NCC-based OCR" (MatchTool/MatchToolDlg.cpp:718-770; dead code behind an early
# return upstream, README.md:118-122 shows its output)
# --------------------------------------------------------------------------------------
OCR_LETTERS = "0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZ"          # chLetters, :723-725


def ocr_assemble(vec_pos, tol=10.0):
    """vec_pos: [((cx, cy), char), ...] -> text.  Sort by y (:752); every run of neighbours closer than dTol = 10 px
    in y is one line, sorted by x (:756-763); a newline wherever consecutive entries differ by more than dTol (:765-771).
    (std::sort leaves ties unspecified; stable sorts here.)"""
    vec = sorted(vec_pos, key=lambda t: t[0][1])
    if not vec:
        return ""
    start = 0
    for i in range(len(vec) - 1):
        if abs(vec[i + 1][0][1] - vec[i][0][1]) < tol:
            continue
        vec[start:i + 1] = sorted(vec[start:i + 1], key=lambda t: t[0][0])
        start = i + 1
    vec[start:] = sorted(vec[start:], key=lambda t: t[0][0])
    out = []
    pre = vec[0][0]
    for pos, ch in vec:
        if abs(pos[1] - pre[1]) > tol:
            out.append("\n")
        pre = pos
        out.append(ch)
    return "".join(out)


def ocr_read(src, templates, params=None, tol=10.0):
    """templates: {char: u8 image}; one learnPattern + match per glyph in OCR_LETTERS order (:727-750), centres
    collected with their letter, then ocr_assemble.  Returns (text, {char: [SingleTargetMatch, ...]})."""
    vec, per = [], {}
    for ch in OCR_LETTERS:
        if ch not in templates:
            continue
        m = OracleMatcher()
        for k, v in (params or {}).items():
            setattr(m, k, v)
        assert m.learn_pattern(templates[ch])
        res = m.match(src)
        per[ch] = res
        vec.extend((r.ptCenter, ch) for r in res)
    return ocr_assemble(vec, tol), per


# --------------------------------------------------------------------------------------
# image ingest (src/MatchToolDialog.cpp:314, :341, :1557-1575)
# --------------------------------------------------------------------------------------
def ingest_bmp(file_bytes):
    """cv::imread(path, IMREAD_GRAYSCALE) on the file image (same OpenCV decoder through cv2.imdecode)."""
    return cv2.imdecode(np.frombuffer(bytes(file_bytes), np.uint8), cv2.IMREAD_GRAYSCALE)


def ingest_image(file_bytes):
    """cv::imread(path, IMREAD_GRAYSCALE) of a BMP or JPEG file image (src/MatchToolDialog.cpp:314, :341)."""
    return cv2.imdecode(np.frombuffer(bytes(file_bytes), np.uint8), cv2.IMREAD_GRAYSCALE)


def jpeg_idct_islow(coef, quant):
    """libjpeg's accurate integer IDCT (jidctint.c jpeg_idct_islow, the JDCT_ISLOW default behind cv::imread) restated in
    numpy: coef [n, 8, 8] quantised coefficients in natural order, quant [8, 8] -> [n, 8, 8] u8 samples.  Model of the
    device kernel fpm_ingest_jpeg_idct_kernel; pinned against cv2.imdecode in tests/test_ingest.py."""
    def pass1d(x, shift):                                   # x [..., 8] along the last axis
        x = [x[..., k] for k in range(8)]
        z2, z3 = x[2], x[6]
        z1 = (z2 + z3) * 4433
        tmp2 = z1 + z3 * -15137
        tmp3 = z1 + z2 * 6270
        tmp0, tmp1 = (x[0] + x[4]) << 13, (x[0] - x[4]) << 13
        tmp10, tmp13, tmp11, tmp12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
        tmp0, tmp1, tmp2, tmp3 = x[7], x[5], x[3], x[1]
        z1, z2, z3, z4 = tmp0 + tmp3, tmp1 + tmp2, tmp0 + tmp2, tmp1 + tmp3
        z5 = (z3 + z4) * 9633
        tmp0, tmp1, tmp2, tmp3 = tmp0 * 2446, tmp1 * 16819, tmp2 * 25172, tmp3 * 12299
        z1, z2, z3, z4 = z1 * -7373, z2 * -20995, z3 * -16069 + z5, z4 * -3196 + z5
        tmp0, tmp1, tmp2, tmp3 = tmp0 + z1 + z3, tmp1 + z2 + z4, tmp2 + z2 + z3, tmp3 + z1 + z4
        r = 1 << (shift - 1)
        out = [tmp10 + tmp3, tmp11 + tmp2, tmp12 + tmp1, tmp13 + tmp0, tmp13 - tmp0, tmp12 - tmp1, tmp11 - tmp2, tmp10 - tmp3]
        return np.stack([(o + r) >> shift for o in out], axis=-1)

    d = np.asarray(coef, np.int64) * np.asarray(quant, np.int64)[None]
    ws = pass1d(d.transpose(0, 2, 1), 13 - 2).transpose(0, 2, 1)           # pass 1 runs down the columns
    out = pass1d(ws, 13 + 2 + 3) & 1023                                     # pass 2 along the rows; range_limit: 10-bit wrap
    out = np.where(out >= 512, out - 1024, out) + 128
    return np.clip(out, 0, 255).astype(np.uint8)


def ingest_rgb32(pixels):
    """QImage::convertToFormat(Format_Grayscale8) of an RGB32 frame: qGray = (R*11 + G*16 + B*5) / 32 (Qt's documented
    formula; parity unpinned -- there is no Qt in this image to run the real conversion)."""
    p = np.asarray(pixels, np.uint32)
    r, g, b = (p >> 16) & 255, (p >> 8) & 255, p & 255
    return ((r * 11 + g * 16 + b * 5) >> 5).astype(np.uint8)
