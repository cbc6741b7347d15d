"""CPU oracle of scale-tolerant matching (FPM_PARAM_SCALE_MIN / MAX) -- TEST INFRASTRUCTURE ONLY.

`ScaledOracleMatcher` is `oracle.oracle.OracleMatcher` with a scale range [scale_min, scale_max].  An instance s times the
template's size is found with the SAME template pyramid by resampling the source by 1/s around the level centre c:

- schedule (`scale_schedule`): ds = 2 / max(w_top, h_top); {min} when min == max, else n = ceil(log(max/min) / log1p(ds)) + 1
  scales s_k = min * exp(k * log(max/min) / (n - 1)) with s_{n-1} = max exactly;
- top layer, pose slot k * n_angles + a (scale-major): canvas warp getRotationMatrix2D(c, angle, 1/s) plus today's centring
  translation, canvas size getBestRotationSize((cvRound(w/s), cvRound(h/s)), ...); a pick p maps back by c + s * (p - c)
  (double, stored as float) before the inverse rotation; the candidate sort keeps its key (score, then slot, then pick order);
- descent: scales {s / (1 + ds_L), s, s * (1 + ds_L)} for a non-trivial range, else {s}; eval k * n_ang + j; the ROI of
  (angle_j, s_k) warps with getRotationMatrix2D(c_L, angle_j, 1/s_k) shifted by lt' - 3, lt' = c_L + (1/s_k) * (rotated
  anchor - c_L); the best eval is the first strict maximum; sub-pixel uses the three angle evals of the best scale; a point
  maps back through c_L + s * (pt - c_L) before the inverse rotation;
- results: the rectangles of (w * s, h * s) in every convention, so NMS and filterWithScore run unchanged on them.

Every "c + k * (p - c)" step is skipped at s == 1, so [1, 1] is `OracleMatcher` exactly.  The device matches one scale per
call (min == max) today; the range semantics above are what a wider range computes.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import List

import cv2
import numpy as np

from oracle import oracle as O
from oracle.oracle import D2R, R2D, VISION_TOLERANCE, MatchParameter, SingleTargetMatch, f32, pt_rotate_pt2f

SCALE_LO, SCALE_HI = 0.5, 2.0


def scale_step(w, h):
    """relative scale step of a pyramid level: the template's far edge moves by about 2 px (cf. atan(2 / max(w, h)))."""
    return 2.0 / max(w, h)


def scale_schedule(lo, hi, w_top, h_top):
    """the top-layer scales of the range [lo, hi] for a top template level of w_top x h_top."""
    if lo == hi:
        return [float(lo)]
    ds = scale_step(w_top, h_top)
    r = math.log(hi / lo)
    n = int(math.ceil(r / math.log1p(ds))) + 1
    out = [lo * math.exp(k * r / (n - 1)) for k in range(n - 1)]
    out.append(float(hi))
    return out


def scale_about(pt, c, k):
    """c + k * (pt - c) in double, stored as float (pt, c: float32 pairs)."""
    return (f32(float(c[0]) + k * (float(pt[0]) - float(c[0]))), f32(float(c[1]) + k * (float(pt[1]) - float(c[1]))))


@dataclass
class ScaledTargetMatch(SingleTargetMatch):
    scale: float = 1.0


class ScaledOracleMatcher(O.OracleMatcher):
    def __init__(self):
        super().__init__()
        self.scale_min = 1.0
        self.scale_max = 1.0

    def _scaled_roi(self, src, size, pt_lt2, angle, s):
        ptc = (f32(f32(src.shape[1] - 1) / f32(2.0)), f32(f32(src.shape[0] - 1) / f32(2.0)))
        lt = pt_rotate_pt2f(pt_lt2, ptc, angle * D2R)
        if s != 1.0:
            lt = scale_about(lt, ptc, 1.0 / s)
        m = cv2.getRotationMatrix2D((float(ptc[0]), float(ptc[1])), angle, 1.0 / s)
        m[0, 2] -= float(f32(lt[0] - f32(3)))
        m[1, 2] -= float(f32(lt[1] - f32(3)))
        return cv2.warpAffine(src, m, (size[0] + 6, size[1] + 6))

    def match(self, src) -> List[ScaledTargetMatch]:
        if not (SCALE_LO <= self.scale_min <= SCALE_HI and SCALE_LO <= self.scale_max <= SCALE_HI):
            raise ValueError("scale out of [0.5, 2]")
        if self.scale_min > self.scale_max:
            raise ValueError("scale_min > scale_max")
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
        top = O.get_top_layer(t0w, t0h, int(math.sqrt(float(self.min_reduce_area))))
        if self.tolerance_range is not None and (self.tolerance_range[0] >= self.tolerance_range[1] or
                                                 self.tolerance_range[2] >= self.tolerance_range[3]):
            return []
        if self.bitwise_not:
            src = 255 - src
        src_pyr = O.build_pyramid(np.ascontiguousarray(src), top)
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
        ranged = self.scale_min != self.scale_max
        scales = scale_schedule(self.scale_min, self.scale_max, size_pat[0], size_pat[1])

        cands: List[MatchParameter] = []
        if tr is not None:
            tr["angles"] = angles
            tr["scales"] = scales
            tr["top"] = []
        for s in scales:
            rsw, rsh = (tsw, tsh) if s == 1.0 else (int(round(tsw / s)), int(round(tsh / s)))
            for ang in angles:
                m = cv2.getRotationMatrix2D((float(center[0]), float(center[1])), ang, 1.0 / s)
                size_best = O.get_best_rotation_size((rsw, rsh), size_pat, ang)
                ftx = f32(f32(f32(size_best[0] - 1) / f32(2.0)) - center[0])
                fty = f32(f32(f32(size_best[1] - 1) / f32(2.0)) - center[1])
                m[0, 2] += float(ftx)
                m[1, 2] += float(fty)
                rot = cv2.warpAffine(top_src, m, size_best, flags=cv2.INTER_LINEAR,
                                     borderMode=cv2.BORDER_CONSTANT, borderValue=(td.border_color,))
                result = self._match_template(rot, top, False, top=True)
                if tr is not None:
                    tr["top"].append(dict(angle=ang, scale=s, size=size_best, rot=rot.copy(), score=result.copy(),
                                          M=m.copy(), picks=[]))
                picks = self.top_picks(result, size_pat, layer_score[top], cal_by_block)
                for loc, val in picks:
                    pt = (f32(f32(loc[0]) - ftx), f32(f32(loc[1]) - fty))
                    if s != 1.0:
                        pt = scale_about(pt, center, s)
                    c = MatchParameter(pt=(float(pt[0]), float(pt[1])), score=val, angle=ang)
                    c.scale = s
                    cands.append(c)
                if tr is not None:
                    tr["top"][-1]["picks"] = picks

        cands.sort(key=lambda c: -c.score)                           # stable: slot, then pick order
        for i, c in enumerate(cands):
            c.cand_id = i
        if tr is not None:
            tr["cands"] = [(c.pt, c.score, c.angle, c.scale) for c in cands]
            tr["refine"] = []

        stop_layer = 1 if self.stop_layer1 else 0
        all_res: List[MatchParameter] = []
        for ci, cand in enumerate(cands):
            pt_lt = pt_rotate_pt2f((f32(cand.pt[0]), f32(cand.pt[1])), center, -cand.angle * D2R)
            if top <= stop_layer:
                k = 1 if top == 0 else 2
                cand.pt = (float(f32(pt_lt[0] * k)), float(f32(pt_lt[1] * k)))
                all_res.append(cand)
                continue
            for layer in range(top - 1, stop_layer - 1, -1):
                tpl_l = td.pyramid[layer]
                a_step = math.atan(2.0 / max(tpl_l.shape[1], tpl_l.shape[0])) * R2D
                ds = scale_step(tpl_l.shape[1], tpl_l.shape[0])
                if self.tolerance_range is None and self.tolerance_angle < VISION_TOLERANCE:
                    l_angles = [0.0]
                else:
                    l_angles = [cand.angle + a_step * i for i in (-1, 0, 1)]
                l_scales = [cand.scale / (1 + ds), cand.scale, cand.scale * (1 + ds)] if ranged else [cand.scale]
                n_ang = len(l_angles)
                src_l = src_pyr[layer]
                src_center = (f32(f32(src_l.shape[1] - 1) / f32(2.0)), f32(f32(src_l.shape[0] - 1) / f32(2.0)))
                new = []
                best_idx, big = 0, -1.0
                pt_lt2 = (f32(pt_lt[0] * 2), f32(pt_lt[1] * 2))
                for ks, ls in enumerate(l_scales):
                    for j, la in enumerate(l_angles):
                        roi = self._scaled_roi(src_l, (tpl_l.shape[1], tpl_l.shape[0]), pt_lt2, la, ls)
                        result = self._match_template(roi, layer, True)
                        val, loc = O._min_max_loc(result)
                        p = MatchParameter(pt=(float(loc[0]), float(loc[1])), score=val, angle=la)
                        p.scale = ls
                        if p.score > big:
                            best_idx, big = ks * n_ang + j, p.score
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
                            tr["refine"].append(dict(cand=ci, layer=layer, j=ks * n_ang + j, angle=la, scale=ls, roi=roi,
                                                     score=result.copy(), loc=loc, val=val,
                                                     pt_lt2=(float(pt_lt2[0]), float(pt_lt2[1]))))
                best = new[best_idx]
                if best.score < layer_score[layer]:
                    break
                jb = best_idx % n_ang
                if self.sub_pixel and layer == 0 and not best.pos_on_border and n_ang == 3 and jb == 1:
                    row = new[best_idx - jb:best_idx - jb + 3]
                    nx, ny, na = self._sub_pix_estimation(row, a_step, 1)
                    best.pt = (nx, ny)
                    best.angle = na
                new_angle, s = best.angle, best.scale
                padding = pt_rotate_pt2f(pt_lt2, src_center, new_angle * D2R)
                if s != 1.0:
                    padding = scale_about(padding, src_center, 1.0 / s)
                padding = (f32(padding[0] - f32(3)), f32(padding[1] - f32(3)))
                pt = (f32(best.pt[0] + float(padding[0])), f32(best.pt[1] + float(padding[1])))
                if s != 1.0:
                    pt = scale_about(pt, src_center, s)
                pt = pt_rotate_pt2f(pt, src_center, -new_angle * D2R)
                if layer == stop_layer:
                    k = 1 if stop_layer == 0 else 2
                    best.pt = (float(f32(pt[0] * k)), float(f32(pt[1] * k)))
                    best.cand_id = cand.cand_id
                    all_res.append(best)
                else:
                    cand.angle = new_angle
                    cand.scale = s
                    pt_lt = pt

        if tr is not None:
            tr["all_res"] = [(r.pt, r.score, r.angle, r.cand_id, r.scale) for r in all_res]
        all_res.sort(key=lambda c: -c.score)
        for i, r in enumerate(all_res):
            if r.score < self.score:
                all_res = all_res[:i]
                break

        k = 1 if stop_layer == 0 else 2
        for r in all_res:
            lt, rt, lb, rb = self._corners(r, td.pyramid[stop_layer].shape[1] * k * r.scale,
                                           td.pyramid[stop_layer].shape[0] * k * r.scale)
            r.rect = cv2.RotatedRect((float(lt[0]), float(lt[1])), (float(rt[0]), float(rt[1])),
                                     (float(rb[0]), float(rb[1])))
        all_res = self._filter_with_rotated_rect(all_res, self.max_overlap)
        all_res.sort(key=lambda c: -c.score)
        if not all_res:
            return []
        iw, ih = td.pyramid[0].shape[1], td.pyramid[0].shape[0]
        out = []
        if self.mfc_compat:
            for i, r in enumerate(all_res):
                a = -r.angle * D2R
                w, h = iw * r.scale, ih * r.scale
                ltx, lty = float(f32(r.pt[0])), float(f32(r.pt[1]))
                rt = (ltx + w * math.cos(a), lty - w * math.sin(a))
                lb = (ltx + h * math.sin(a), lty + h * math.cos(a))
                rb = (rt[0] + h * math.sin(a), rt[1] + h * math.cos(a))
                ang = -r.angle
                if ang < -180:
                    ang += 360
                if ang > 180:
                    ang -= 360
                out.append(ScaledTargetMatch(ptLT=(ltx, lty), ptRT=rt, ptRB=rb, ptLB=lb,
                                             ptCenter=((ltx + rt[0] + rb[0] + lb[0]) / 4, (lty + rt[1] + rb[1] + lb[1]) / 4),
                                             angle=ang, score=r.score, scale=r.scale))
                if i + 1 == self.max_pos:
                    break
            return out
        for r in all_res:
            lt, rt, lb, rb = self._corners(r, iw * r.scale, ih * r.scale)
            four = f32(4.0)
            cx = f32(f32(f32(f32(lt[0] + rt[0]) + lb[0]) + rb[0]) / four)
            cy = f32(f32(f32(f32(lt[1] + rt[1]) + lb[1]) + rb[1]) / four)
            out.append(ScaledTargetMatch(
                ptLT=(float(lt[0]), float(lt[1])), ptRT=(float(rt[0]), float(rt[1])),
                ptRB=(float(rb[0]), float(rb[1])), ptLB=(float(lb[0]), float(lb[1])),
                ptCenter=(float(cx), float(cy)), angle=r.angle, score=r.score, scale=r.scale))
        return out


def paste_scaled(dst, tpl, cx, cy, angle_deg, scale):
    """fpm_workloads.paste_rotated with a scale: `tpl` scaled by `scale` and rotated by angle_deg (OpenCV sign) with its
    centre at (cx, cy), in place."""
    th, tw = tpl.shape
    m = cv2.getRotationMatrix2D(((tw - 1) / 2.0, (th - 1) / 2.0), angle_deg, scale)
    m[0, 2] += cx - (tw - 1) / 2.0
    m[1, 2] += cy - (th - 1) / 2.0
    size = (dst.shape[1], dst.shape[0])
    warped = cv2.warpAffine(tpl, m, size, flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
    mask = cv2.warpAffine(np.full_like(tpl, 255), m, size, flags=cv2.INTER_NEAREST, borderMode=cv2.BORDER_CONSTANT,
                          borderValue=0)
    dst[mask > 0] = warped[mask > 0]
    return dst


def scaled_scene(w, h, tw, th, poses, seed):
    """a seeded template (tw x th) and frame (w x h) with one instance per (cx, cy, angle, scale) pose"""
    import fpm_workloads as synth
    tpl = synth.synth_template(max(tw, th), seed)[:th, :tw].copy()
    src = synth.background(w, h, seed + 100, 3.0)
    for cx, cy, a, s in poses:
        paste_scaled(src, tpl, cx, cy, a, s)
    return tpl, src
