"""Host-side mirror of the reference's `TemplateMatcher` class
(/root/reference/include/TemplateMatcher.h:9-52), bound to the CUDA library through the C ABI.

Same method names, argument meaning and error behaviour as the reference:
`learnPattern` returns False for an empty template, `match` returns an empty list when nothing
is learned / the source is empty / the template does not fit / nothing is found.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib as L


class FpmError(RuntimeError):
    pass


@dataclass
class SingleTargetMatch:
    """s_SingleTargetMatch (/root/reference/include/DataStructures.h:97-115)."""
    ptLT: Tuple[float, float]
    ptRT: Tuple[float, float]
    ptRB: Tuple[float, float]
    ptLB: Tuple[float, float]
    ptCenter: Tuple[float, float]
    dMatchedAngle: float
    dMatchScore: float
    dScale: float = 1.0             # match scale (setScaleRange): the instance is dScale times the template's size


def _as_u8_2d(img) -> np.ndarray:
    a = np.asarray(img)
    if a.ndim != 2 or a.dtype != np.uint8:
        raise FpmError("images must be single-channel 8-bit (IMREAD_GRAYSCALE), got %s %s" % (a.dtype, a.shape))
    if a.strides[1] != 1:
        a = np.ascontiguousarray(a)
    return a


def _convert(res, n, scales=None) -> List[SingleTargetMatch]:
    out = []
    for i in range(n):
        r = res[i]
        out.append(SingleTargetMatch((r.ltx, r.lty), (r.rtx, r.rty), (r.rbx, r.rby), (r.lbx, r.lby),
                                     (r.cx, r.cy), r.angle, r.score, 1.0 if scales is None else scales[i]))
    return out


class TemplateMatcher:
    def __init__(self, device: int = 0, result_capacity: int = 4096):
        self._lib = L.load()
        self._h = self._lib.fpm_create(device)
        if not self._h:
            raise FpmError("fpm_create(%d) failed: no usable CUDA device (there is no CPU fallback)" % device)
        self.device = device
        self.result_capacity = result_capacity

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._lib.fpm_destroy(self._h)
                self._h = None
        except Exception:
            pass

    close = __del__

    def _check(self, rc):
        if rc != 0:
            raise FpmError("fpm error %d: %s" % (rc, self._lib.fpm_last_error(self._h).decode()))

    # ---- parameters (include/TemplateMatcher.h:22-37) ----
    def _set(self, p, v): self._check(self._lib.fpm_set_param(self._h, p, float(v)))
    def _get(self, p): return self._lib.fpm_get_param(self._h, p)
    def setMaxPositions(self, v: int): self._set(L.PARAM_MAX_POSITIONS, v)
    def setMaxOverlap(self, v: float): self._set(L.PARAM_MAX_OVERLAP, v)
    def setScore(self, v: float): self._set(L.PARAM_SCORE, v)
    def setToleranceAngle(self, v: float): self._set(L.PARAM_TOLERANCE_ANGLE, v)
    def setMinReduceArea(self, v: int): self._set(L.PARAM_MIN_REDUCE_AREA, v)
    def setUseSIMD(self, v: bool): self._set(L.PARAM_USE_SIMD, 1 if v else 0)
    def setSubPixelEstimation(self, v: bool): self._set(L.PARAM_SUBPIXEL, 1 if v else 0)
    def getMaxPositions(self) -> int: return int(self._get(L.PARAM_MAX_POSITIONS))
    def getMaxOverlap(self) -> float: return self._get(L.PARAM_MAX_OVERLAP)
    def getScore(self) -> float: return self._get(L.PARAM_SCORE)
    def getToleranceAngle(self) -> float: return self._get(L.PARAM_TOLERANCE_ANGLE)
    def getMinReduceArea(self) -> int: return int(self._get(L.PARAM_MIN_REDUCE_AREA))
    def getUseSIMD(self) -> bool: return bool(self._get(L.PARAM_USE_SIMD))
    def getSubPixelEstimation(self) -> bool: return bool(self._get(L.PARAM_SUBPIXEL))
    def setTrace(self, v: bool): self._set(L.PARAM_TRACE, 1 if v else 0)
    def setSplitBatch(self, v: int): self._set(L.PARAM_SPLIT_BATCH, int(v))
    def getSplitBatch(self) -> int: return int(self._get(L.PARAM_SPLIT_BATCH))
    def setWorkspaceMB(self, v: float): self._set(L.PARAM_WORKSPACE_MB, v)
    def setH2DChunk(self, v: int): self._set(L.PARAM_H2D_CHUNK, v)
    def setTensorCores(self, v: int): self._set(L.PARAM_TENSOR_CORES, v)
    def setMfcCompat(self, v: bool): self._set(L.PARAM_MFC_COMPAT, 1 if v else 0)
    def setStopLayer1(self, v: bool): self._set(L.PARAM_STOP_LAYER1, 1 if v else 0)
    def setBitwiseNot(self, v: bool): self._set(L.PARAM_BITWISE_NOT, 1 if v else 0)

    def setToleranceRange(self, rng):
        """rng = (t1, t2, t3, t4) enables the MFC two-range sweep, None disables it"""
        if rng is None:
            self._set(L.PARAM_TOLERANCE_RANGE, 0)
            return
        for p, v in zip((L.PARAM_TOLERANCE1, L.PARAM_TOLERANCE2, L.PARAM_TOLERANCE3, L.PARAM_TOLERANCE4), rng):
            self._set(p, v)
        self._set(L.PARAM_TOLERANCE_RANGE, 1)

    def setScaleRange(self, lo: float, hi: float):
        """Match instances lo..hi times the template's size (FPM_PARAM_SCALE_MIN / MAX, each in [0.5, 2]; default 1, 1; a
        match refuses lo > hi).  Result rectangles have the scaled size and dScale reports each one's scale.  Both values are
        checked before either is set, so a refused call leaves the range as it was."""
        for name, v in (("FPM_PARAM_SCALE_MIN", lo), ("FPM_PARAM_SCALE_MAX", hi)):
            if not (math.isfinite(float(v)) and 0.5 <= float(v) <= 2.0):
                raise FpmError("%s must lie in [0.5, 2], got %r" % (name, v))
        self._set(L.PARAM_SCALE_MIN, lo)
        self._set(L.PARAM_SCALE_MAX, hi)

    def getScaleRange(self) -> Tuple[float, float]:
        return self._get(L.PARAM_SCALE_MIN), self._get(L.PARAM_SCALE_MAX)

    def getLastExecutionTime(self) -> float:
        """seconds, like the reference (include/TemplateMatcher.h:40)"""
        return self._lib.fpm_last_time_ms(self._h) / 1000.0

    def isPatternLearned(self) -> bool: return bool(self._lib.fpm_is_learned(self._h))
    def clearPattern(self): self._lib.fpm_clear(self._h)
    def setUserDefinedRect(self, rect: Sequence[int]): self._lib.fpm_set_user_rect(self._h, *[int(v) for v in rect])

    def getUserDefinedRect(self):
        v = [C.c_int() for _ in range(4)]
        self._lib.fpm_get_user_rect(self._h, *[C.byref(x) for x in v])
        return tuple(x.value for x in v)

    def hasUserDefinedRect(self) -> bool:
        return bool(self._lib.fpm_get_user_rect(self._h, None, None, None, None))

    def launchCount(self) -> int: return int(self._lib.fpm_launch_count(self._h))

    # ---- learnPattern (src/TemplateMatcher.cpp:45-95) ----
    def learnPattern(self, templateImage, mask=None) -> bool:
        """mask (optional): a 2-D array of the template's shape, nonzero = kept pixel; the masked pixels do not count
        (fpm_learn_masked).  Without a mask the whole rectangle is matched."""
        if templateImage is None or np.asarray(templateImage).size == 0:
            return False
        t = _as_u8_2d(templateImage)
        self._tpl_keepalive = t
        if mask is None:
            self._check(self._lib.fpm_learn(self._h, t.ctypes.data, t.shape[1], t.shape[0], t.strides[0]))
            return True
        m = np.ascontiguousarray(np.asarray(mask) != 0, dtype=np.uint8)
        if m.shape != t.shape:
            raise ValueError(f"mask shape {m.shape} differs from the template's {t.shape}")
        self._check(self._lib.fpm_learn_masked(self._h, t.ctypes.data, t.shape[1], t.shape[0], t.strides[0],
                                               m.ctypes.data, m.strides[0]))
        return True

    # ---- template sets: n templates in one handle, matched in shared launches (fpm_learn_set) ----
    def learnPatternSet(self, templates, masks=None) -> bool:
        """n templates (2-D uint8 arrays) replace the pattern; all use this matcher's parameters.  masks (optional): a list
        of n entries, each None (unmasked) or an array of its template's shape, nonzero = kept (fpm_learn_set_masked)."""
        ts = [_as_u8_2d(t) for t in templates]
        n = len(ts)
        ptrs = (C.c_void_p * max(n, 1))(*[t.ctypes.data for t in ts])
        ws = (C.c_int * max(n, 1))(*[t.shape[1] for t in ts])
        hs = (C.c_int * max(n, 1))(*[t.shape[0] for t in ts])
        st = (C.c_int * max(n, 1))(*[t.strides[0] for t in ts])
        if masks is None:
            self._tpl_keepalive = ts
            self._check(self._lib.fpm_learn_set(self._h, n, ptrs, ws, hs, st))
            return True
        if len(masks) != n:
            raise ValueError(f"{len(masks)} masks for {n} templates")
        ms = []
        for i, (t, m) in enumerate(zip(ts, masks)):
            if m is not None:
                m = np.ascontiguousarray(np.asarray(m) != 0, dtype=np.uint8)
                if m.shape != t.shape:
                    raise ValueError(f"mask {i}: shape {m.shape} differs from the template's {t.shape}")
            ms.append(m)
        self._tpl_keepalive = (ts, ms)
        mp = (C.c_void_p * max(n, 1))(*[None if m is None else m.ctypes.data for m in ms])
        mst = (C.c_int * max(n, 1))(*[0 if m is None else m.strides[0] for m in ms])
        self._check(self._lib.fpm_learn_set_masked(self._h, n, ptrs, ws, hs, st, mp, mst))
        return True

    def patternSetSize(self) -> int: return int(self._lib.fpm_set_size(self._h))

    # scaled=True on the set methods: the scaled set calls (fpm_match_set_scaled*, fpm_match_ingested_set_scaled*,
    # fpm_match_set_sharded_scaled*), which match at the handle's scale range (setScaleRange) and fill dScale; the default
    # calls match at [1, 1] only and refuse any other range
    def _set_results(self, res, counts, B, T, scales=None):
        cap = self.result_capacity
        return [[_convert(res[(b * T + t) * cap:(b * T + t + 1) * cap], min(counts[b * T + t], cap),
                          None if scales is None else scales[(b * T + t) * cap:(b * T + t + 1) * cap]) for t in range(T)]
                for b in range(B)]

    def matchSetBatchRaw(self, ptr: int, B: int, W: int, H: int, stride: int, frame_stride: int, on_device: bool,
                         res=None, counts=None, scaled: bool = False, scales=None):
        """Pointer-level set match: returns (results ctypes array [B][T][cap], counts [B][T]), and with scaled=True
        (fpm_match_set_scaled) also the scales [B][T][cap] at the indices of the results."""
        cap, T = self.result_capacity, max(self.patternSetSize(), 1)
        if res is None:
            res = (L.fpm_result * (cap * B * T))()
        if counts is None:
            counts = (C.c_int * (B * T))()
        if not scaled:
            self._check(self._lib.fpm_match_set_batch(self._h, ptr, 1 if on_device else 0, B, W, H, stride, frame_stride, res, cap,
                                                      counts))
            return res, counts
        if scales is None:
            scales = (C.c_double * (cap * B * T))()
        self._check(self._lib.fpm_match_set_scaled(self._h, ptr, 1 if on_device else 0, B, W, H, stride, frame_stride, res, scales,
                                                   cap, counts))
        return res, counts, scales

    def matchSetBatch(self, frames: np.ndarray, scaled: bool = False) -> List[List[List[SingleTargetMatch]]]:
        """frames: [B, H, W] uint8 in host memory -> [frame][template][results]."""
        f = np.asarray(frames)
        if f.ndim != 3 or f.dtype != np.uint8 or f.strides[2] != 1:
            raise FpmError("frames must be a [B,H,W] uint8 array with unit pixel stride")
        B, H, W = f.shape
        T = max(self.patternSetSize(), 1)
        out = self.matchSetBatchRaw(f.ctypes.data, B, W, H, f.strides[1], f.strides[0], False, scaled=scaled)
        return self._set_results(out[0], out[1], B, T, out[2] if scaled else None)

    def matchSet(self, sourceImage, scaled: bool = False) -> List[List[SingleTargetMatch]]:
        """one host image -> [template][results]"""
        return self.matchSetBatch(_as_u8_2d(sourceImage)[None], scaled=scaled)[0]

    def matchIngestedSetBatch(self, scaled: bool = False) -> List[List[List[SingleTargetMatch]]]:
        """the frames of the last ingest x the set: [frame][template][results]"""
        B, T, cap = self.ingestedCount(), max(self.patternSetSize(), 1), self.result_capacity
        res = (L.fpm_result * (cap * max(B, 1) * T))()
        counts = (C.c_int * (max(B, 1) * T))()
        if not scaled:
            self._check(self._lib.fpm_match_ingested_set_batch(self._h, res, cap, counts))
            return self._set_results(res, counts, B, T)
        sc = (C.c_double * (cap * max(B, 1) * T))()
        self._check(self._lib.fpm_match_ingested_set_scaled(self._h, res, sc, cap, counts))
        return self._set_results(res, counts, B, T, sc)

    # ---- merged set results: one labelled list per frame, rotated-rectangle NMS across templates ----
    def _merged_results(self, res, labels, counts, B, scales=None):
        cap = self.result_capacity
        out = []
        for b in range(B):
            m = min(counts[b], cap)
            out.append(list(zip(labels[b * cap:b * cap + m],
                                _convert(res[b * cap:(b + 1) * cap], m, None if scales is None else scales[b * cap:(b + 1) * cap]))))
        return out

    def matchSetBatchMergedRaw(self, ptr: int, B: int, W: int, H: int, stride: int, frame_stride: int, on_device: bool,
                               max_overlap: float, res=None, labels=None, counts=None, set_counts=None, scaled: bool = False,
                               scales=None):
        """Pointer-level merged set match (fpm_match_set_batch_merged): returns (results ctypes array [B][cap], labels [B][cap],
        counts [B], set_counts [B][T]: the per-template totals), and with scaled=True (fpm_match_set_scaled_merged) also the
        scales [B][cap]."""
        cap, T = self.result_capacity, max(self.patternSetSize(), 1)
        if res is None:
            res = (L.fpm_result * (cap * B))()
        if labels is None:
            labels = (C.c_int * (cap * B))()
        if counts is None:
            counts = (C.c_int * B)()
        if set_counts is None:
            set_counts = (C.c_int * (B * T))()
        if not scaled:
            self._check(self._lib.fpm_match_set_batch_merged(self._h, ptr, 1 if on_device else 0, B, W, H, stride, frame_stride,
                                                             float(max_overlap), res, labels, cap, counts, set_counts))
            return res, labels, counts, set_counts
        if scales is None:
            scales = (C.c_double * (cap * B))()
        self._check(self._lib.fpm_match_set_scaled_merged(self._h, ptr, 1 if on_device else 0, B, W, H, stride, frame_stride,
                                                          float(max_overlap), res, scales, labels, cap, counts, set_counts))
        return res, labels, counts, set_counts, scales

    def matchSetBatchMerged(self, frames: np.ndarray, max_overlap: float,
                            scaled: bool = False) -> List[List[Tuple[int, SingleTargetMatch]]]:
        """frames: [B, H, W] uint8 in host memory -> per frame one list of (set index, result), score descending, after NMS
        across templates with the overlap threshold max_overlap (the per-template lists keep MaxOverlap)."""
        f = np.asarray(frames)
        if f.ndim != 3 or f.dtype != np.uint8 or f.strides[2] != 1:
            raise FpmError("frames must be a [B,H,W] uint8 array with unit pixel stride")
        B, H, W = f.shape
        out = self.matchSetBatchMergedRaw(f.ctypes.data, B, W, H, f.strides[1], f.strides[0], False, max_overlap, scaled=scaled)
        return self._merged_results(out[0], out[1], out[2], B, out[4] if scaled else None)

    def matchSetMerged(self, sourceImage, max_overlap: float, scaled: bool = False) -> List[Tuple[int, SingleTargetMatch]]:
        """one host image -> [(set index, result)]"""
        return self.matchSetBatchMerged(_as_u8_2d(sourceImage)[None], max_overlap, scaled=scaled)[0]

    def matchIngestedSetBatchMerged(self, max_overlap: float, scaled: bool = False) -> List[List[Tuple[int, SingleTargetMatch]]]:
        """the frames of the last ingest x the set, merged: [frame][(set index, result)]"""
        B, T, cap = self.ingestedCount(), max(self.patternSetSize(), 1), self.result_capacity
        res = (L.fpm_result * (cap * max(B, 1)))()
        labels = (C.c_int * (cap * max(B, 1)))()
        counts = (C.c_int * max(B, 1))()
        if not scaled:
            self._check(self._lib.fpm_match_ingested_set_batch_merged(self._h, float(max_overlap), res, labels, cap, counts, None))
            return self._merged_results(res, labels, counts, B)
        sc = (C.c_double * (cap * max(B, 1)))()
        self._check(self._lib.fpm_match_ingested_set_scaled_merged(self._h, float(max_overlap), res, sc, labels, cap, counts, None))
        return self._merged_results(res, labels, counts, B, sc)

    # ---- match (src/TemplateMatcher.cpp:97-437) ----
    def match(self, sourceImage) -> List[SingleTargetMatch]:
        if sourceImage is None or np.asarray(sourceImage).size == 0:
            return []
        s = _as_u8_2d(sourceImage)
        cap = self.result_capacity
        res = (L.fpm_result * cap)()
        sc = (C.c_double * cap)()
        n = (C.c_int * 1)()
        self._check(self._lib.fpm_match_scaled(self._h, s.ctypes.data, 0, 1, s.shape[1], s.shape[0], s.strides[0],
                                               s.strides[0] * s.shape[0], res, sc, cap, n))
        return _convert(res, min(n[0], cap), sc)

    # ---- image ingest (SURVEY 8f rank 4): decode on the device, match without a pixel copy ----
    def ingestBmp(self, file_bytes) -> tuple:
        """BMP file image (bytes / uint8 array) -> device-resident grayscale frame; returns (width, height)."""
        b = np.frombuffer(bytes(file_bytes), np.uint8) if not isinstance(file_bytes, np.ndarray) else np.ascontiguousarray(file_bytes, np.uint8)
        w, h = C.c_int(0), C.c_int(0)
        self._check(self._lib.fpm_ingest_bmp(self._h, b.ctypes.data, b.size, C.byref(w), C.byref(h)))
        self._ingest_shape = (h.value, w.value)
        return w.value, h.value

    def _ingest_file(self, fn, file_bytes) -> tuple:
        b = np.frombuffer(bytes(file_bytes), np.uint8) if not isinstance(file_bytes, np.ndarray) else np.ascontiguousarray(file_bytes, np.uint8)
        w, h = C.c_int(0), C.c_int(0)
        self._check(fn(self._h, b.ctypes.data, b.size, C.byref(w), C.byref(h)))
        self._ingest_shape = (h.value, w.value)
        return w.value, h.value

    def ingestJpeg(self, file_bytes) -> tuple:
        """baseline JPEG file image -> the grayscale frame cv::imread(IMREAD_GRAYSCALE) returns (luma, ISLOW IDCT on the device)"""
        return self._ingest_file(self._lib.fpm_ingest_jpeg, file_bytes)

    def ingestImage(self, file_bytes) -> tuple:
        """BMP or JPEG by signature, like cv::imread"""
        return self._ingest_file(self._lib.fpm_ingest_image, file_bytes)

    def ingestRgb32(self, pixels) -> None:
        """camera frame: [H, W] uint32 0xAARRGGBB (QImage::Format_RGB32) -> device-resident grayscale frame"""
        p = np.ascontiguousarray(pixels, np.uint32)
        self._check(self._lib.fpm_ingest_rgb32(self._h, p.ctypes.data, p.shape[1], p.shape[0], p.strides[0]))
        self._ingest_shape = p.shape

    def ingestedPixels(self) -> np.ndarray:
        out = np.zeros(self._ingest_shape, np.uint8)
        self._check(self._lib.fpm_ingested_pixels(self._h, out.ctypes.data))
        return out

    def matchIngested(self) -> List[SingleTargetMatch]:
        cap = self.result_capacity
        res = (L.fpm_result * cap)()
        n = C.c_int(0)
        if self.ingestedCount() != 1:                     # fpm_match_ingested's refusal and message
            self._check(self._lib.fpm_match_ingested(self._h, res, cap, C.byref(n)))
        sc = (C.c_double * cap)()
        cnt = (C.c_int * 1)()
        self._check(self._lib.fpm_match_ingested_scaled(self._h, res, sc, cap, cnt))
        return _convert(res, min(cnt[0], cap), sc)

    def learnIngested(self) -> bool:
        self._check(self._lib.fpm_learn_ingested(self._h))
        return True

    def ingestJpegBatch(self, files, offsets=None) -> tuple:
        """n JPEG file images of one frame size -> n device-resident grayscale frames; returns (width, height).
        files: a list of bytes-like objects (packed here into one buffer), or a 1-D uint8 buffer holding the files back to back
        with offsets (n + 1 entries): a numpy array, or the data_ptr() of a pinned torch CPU tensor (no copy, PCIe rate)."""
        if offsets is None:
            parts = [np.frombuffer(bytes(f), np.uint8) for f in files]
            offs = np.zeros(len(parts) + 1, np.uint64)
            offs[1:] = np.cumsum([p.size for p in parts])
            buf = np.concatenate(parts) if parts else np.zeros(0, np.uint8)
            ptr = buf.ctypes.data
        else:
            offs = np.ascontiguousarray(offsets, np.uint64)
            if isinstance(files, int):
                buf, ptr = None, files
            else:
                buf = np.ascontiguousarray(files, np.uint8)
                if buf.ndim != 1:
                    raise FpmError("the packed JPEG buffer must be 1-D uint8")
                if offs.size and int(offs[-1]) > buf.size:
                    raise FpmError("JPEG batch offsets run past the buffer")
                ptr = buf.ctypes.data
        n = max(int(offs.size) - 1, 0)
        w, h = C.c_int(0), C.c_int(0)
        self._check(self._lib.fpm_ingest_jpeg_batch(self._h, ptr, offs.ctypes.data, n, C.byref(w), C.byref(h)))
        self._ingest_shape = (h.value, w.value)
        return w.value, h.value

    def ingestedCount(self) -> int: return int(self._lib.fpm_ingested_count(self._h))

    def ingestedFramePixels(self, index: int) -> np.ndarray:
        out = np.zeros(self._ingest_shape, np.uint8)
        self._check(self._lib.fpm_ingested_frame_pixels(self._h, int(index), out.ctypes.data))
        return out

    def matchIngestedBatch(self) -> List[List[SingleTargetMatch]]:
        """the frames of the last ingest matched as one batch: one result list per frame"""
        B = self.ingestedCount()
        cap = self.result_capacity
        res = (L.fpm_result * (cap * max(B, 1)))()
        n = (C.c_int * max(B, 1))()
        sc = (C.c_double * (cap * max(B, 1)))()
        self._check(self._lib.fpm_match_ingested_scaled(self._h, res, sc, cap, n))
        return [_convert(res[b * cap:(b + 1) * cap], min(n[b], cap), sc[b * cap:(b + 1) * cap]) for b in range(B)]

    def matchBatch(self, frames: np.ndarray) -> List[List[SingleTargetMatch]]:
        """frames: [B, H, W] uint8 in host memory (pinned for full PCIe speed)."""
        f = np.asarray(frames)
        if f.ndim != 3 or f.dtype != np.uint8 or f.strides[2] != 1:
            raise FpmError("frames must be a [B,H,W] uint8 array with unit pixel stride")
        B, H, W = f.shape
        cap = self.result_capacity
        res = (L.fpm_result * (cap * B))()
        sc = (C.c_double * (cap * B))()
        n = (C.c_int * B)()
        self._check(self._lib.fpm_match_scaled(self._h, f.ctypes.data, 0, B, W, H, f.strides[1], f.strides[0], res, sc, cap, n))
        return [_convert(res[b * cap:(b + 1) * cap], min(n[b], cap), sc[b * cap:(b + 1) * cap]) for b in range(B)]

    def matchBatchRaw(self, ptr: int, B: int, W: int, H: int, stride: int, frame_stride: int, on_device: bool,
                      res=None, counts=None):
        """Pointer-level entry used by bench.py (torch tensors): returns (results ctypes array, counts)."""
        cap = self.result_capacity
        if res is None:
            res = (L.fpm_result * (cap * B))()
        if counts is None:
            counts = (C.c_int * B)()
        fn = self._lib.fpm_match_batch_device if on_device else self._lib.fpm_match_batch
        self._check(fn(self._h, ptr, B, W, H, stride, frame_stride, res, cap, counts))
        return res, counts

    # ---- timing / profiling (bench.py) ----
    def setProfile(self, v: bool): self._set(L.PARAM_PROFILE, 1 if v else 0)
    def timerRecord(self, which: int): self._check(self._lib.fpm_timer_record(self._h, which))
    def timerElapsedMs(self) -> float: return self._lib.fpm_timer_elapsed_ms(self._h)
    def profileReset(self): self._lib.fpm_profile_reset(self._h)

    def profile(self):
        """{kernel name: (device ms, launches, algorithmic work)} accumulated since profileReset()."""
        out = {}
        for k in range(self._lib.fpm_profile_num_kernels()):
            ms, n, w = C.c_double(), C.c_longlong(), C.c_double()
            self._check(self._lib.fpm_profile_get(self._h, k, C.byref(ms), C.byref(n), C.byref(w)))
            out[self._lib.fpm_profile_name(k).decode()] = (ms.value, n.value, w.value)
        return out

    # ---- learned-template introspection ----
    def templateLevels(self):
        out = []
        for l in range(self._lib.fpm_tpl_levels(self._h)):
            w, h, eq = C.c_int(), C.c_int(), C.c_int()
            mean, norm, inv = C.c_double(), C.c_double(), C.c_double()
            self._check(self._lib.fpm_tpl_level_info(self._h, l, C.byref(w), C.byref(h), C.byref(mean), C.byref(norm),
                                                     C.byref(inv), C.byref(eq)))
            pix = np.empty((h.value, w.value), np.uint8)
            self._check(self._lib.fpm_tpl_level_pixels(self._h, l, pix.ctypes.data))
            mask = np.empty((h.value, w.value), np.uint8)
            n_kept = self._lib.fpm_tpl_level_mask(self._h, l, mask.ctypes.data)
            self._check(min(n_kept, 0))
            out.append(dict(w=w.value, h=h.value, mean=mean.value, norm=norm.value, inv_area=inv.value,
                            result_equal1=bool(eq.value), pixels=pix, mask=mask, n_kept=n_kept))
        return out

    def borderColor(self) -> int: return self._lib.fpm_tpl_border_color(self._h)

    # ---- traces (FPM_PARAM_TRACE) ----
    def traceCandidates(self) -> np.ndarray:
        n = self._lib.fpm_trace_num_candidates(self._h)
        rows = np.zeros((n, 4), np.float64)
        if n:
            self._check(self._lib.fpm_trace_candidates(self._h, rows.ctypes.data))
        return rows

    def traceEvals(self, level: int) -> np.ndarray:
        n = self._lib.fpm_trace_num_evals(self._h, level)
        rows = np.zeros((n, 5), np.float64)
        if n:
            self._check(self._lib.fpm_trace_evals(self._h, level, rows.ctypes.data))
        return rows

    def traceEvalScores(self, level: int) -> np.ndarray:
        """[n, 7, 7] float32: the score patch of every refinement eval of `level`, rows as in traceEvals(level)"""
        n = self._lib.fpm_trace_num_evals(self._h, level)
        out = np.zeros((n, 7, 7), np.float32)
        if n:
            self._check(self._lib.fpm_trace_eval_scores(self._h, level, out.ctypes.data))
        return out

    def traceEvalRois(self, level: int) -> Optional[np.ndarray]:
        """[n, h, pitch] uint8: the ROI patch of every refinement eval of `level` at the device pitch (the patch is
        [:, :, :w] with w = template width + 6), rows as in traceEvals(level); None where the ROIs are warped inside the
        correlation kernel and never stored"""
        w, h, p = C.c_int(), C.c_int(), C.c_int()
        n = self._lib.fpm_trace_eval_rois(self._h, level, None, C.byref(w), C.byref(h), C.byref(p))
        if n < 0:
            self._check(n)
        if n == 0:
            return None
        out = np.zeros((n, h.value, p.value), np.uint8)
        rc = self._lib.fpm_trace_eval_rois(self._h, level, out.ctypes.data, C.byref(w), C.byref(h), C.byref(p))
        self._check(rc if rc < 0 else 0)
        return out

    def traceLevel(self, level: int) -> Optional[np.ndarray]:
        w, h = C.c_int(), C.c_int()
        if self._lib.fpm_trace_level(self._h, level, None, C.byref(w), C.byref(h)) != 0:
            return None
        out = np.empty((h.value, w.value), np.uint8)
        self._check(self._lib.fpm_trace_level(self._h, level, out.ctypes.data, C.byref(w), C.byref(h)))
        return out

    # ---- stage kernels (parity tests) ----
    def dbgPyrDown(self, img) -> np.ndarray:
        s = _as_u8_2d(img)
        out = np.empty(((s.shape[0] + 1) // 2, (s.shape[1] + 1) // 2), np.uint8)
        self._check(self._lib.fpm_dbg_pyrdown(self._h, s.ctypes.data, s.shape[1], s.shape[0], s.strides[0], out.ctypes.data))
        return out

    def dbgPyrDown2(self, img, misalign=0, two=True):
        """one launch of the pyramid kernel: (pyrDown(img), pyrDown(pyrDown(img))), or the first level only."""
        s = _as_u8_2d(img)
        h1, w1 = (s.shape[0] + 1) // 2, (s.shape[1] + 1) // 2
        o1 = np.empty((h1, w1), np.uint8)
        o2 = np.empty(((h1 + 1) // 2, (w1 + 1) // 2), np.uint8) if two else None
        self._check(self._lib.fpm_dbg_pyrdown2(self._h, s.ctypes.data, s.shape[1], s.shape[0], s.strides[0], int(misalign),
                                               o1.ctypes.data, o2.ctypes.data if two else None))
        return (o1, o2) if two else o1

    def dbgWarpAffine(self, img, M, dsize, border=0) -> np.ndarray:
        s = _as_u8_2d(img)
        m = np.ascontiguousarray(np.asarray(M, np.float64).reshape(6))
        out = np.empty((dsize[1], dsize[0]), np.uint8)
        self._check(self._lib.fpm_dbg_warp_affine(self._h, s.ctypes.data, s.shape[1], s.shape[0], s.strides[0],
                                                  m.ctypes.data, dsize[0], dsize[1], int(border), out.ctypes.data))
        return out

    def dbgCorrRows(self, roi, tpl):
        r = np.ascontiguousarray(_as_u8_2d(roi))
        t = np.ascontiguousarray(_as_u8_2d(tpl))
        th, tw = t.shape
        assert r.shape == (th + 6, tw + 6)
        rowsum = np.zeros((th, 7, 7), np.int32)
        rowS = np.zeros((th + 6, 7), np.int32)
        rowQ = np.zeros((th + 6, 7), np.int32)
        self._check(self._lib.fpm_dbg_corr_rows(self._h, r.ctypes.data, t.ctypes.data, tw, th, rowsum.ctypes.data,
                                                rowS.ctypes.data, rowQ.ctypes.data))
        return rowsum, rowS, rowQ

    def dbgCorrRowsMMA(self, rois, tpl):
        """tensor-core path: rois [ne, th+6, tw+6] u8 -> (rowsum [ne, th, 7, 7], rowS [ne, th+6, 7], rowQ)"""
        r = np.ascontiguousarray(np.asarray(rois, np.uint8))
        t = np.ascontiguousarray(_as_u8_2d(tpl))
        th, tw = t.shape
        ne = r.shape[0]
        assert r.shape == (ne, th + 6, tw + 6)
        rowsum = np.zeros((ne, th, 7, 7), np.int32)
        rowS = np.zeros((ne, th + 6, 7), np.int32)
        rowQ = np.zeros((ne, th + 6, 7), np.int32)
        self._check(self._lib.fpm_dbg_corr_rows_mma(self._h, r.ctypes.data, ne, t.ctypes.data, tw, th, rowsum.ctypes.data,
                                                    rowS.ctypes.data, rowQ.ctypes.data))
        return rowsum, rowS, rowQ

    def dbgCorrFused(self, rois, tpl):
        """fused tensor-core kernel: rois [ne, th+6, tw+6] u8 -> (numer [ne, 7, 7] f32, winS [ne, 7, 7] i64, winQ)"""
        r = np.ascontiguousarray(np.asarray(rois, np.uint8))
        t = np.ascontiguousarray(_as_u8_2d(tpl))
        th, tw = t.shape
        ne = r.shape[0]
        assert r.shape == (ne, th + 6, tw + 6)
        numer = np.zeros((ne, 7, 7), np.float32)
        winS = np.zeros((ne, 7, 7), np.int64)
        winQ = np.zeros((ne, 7, 7), np.int64)
        edge = np.zeros((ne, th + 6, 7), np.int32)
        self._check(self._lib.fpm_dbg_corr_fused(self._h, r.ctypes.data, ne, t.ctypes.data, tw, th, numer.ctypes.data,
                                                 winS.ctypes.data, winQ.ctypes.data, edge.ctypes.data))
        self.last_edge_rows = edge
        return numer, winS, winQ

    def dbgTopScore(self, img) -> np.ndarray:
        s = np.ascontiguousarray(_as_u8_2d(img))
        lv = self.templateLevels()[-1]
        out = np.zeros((s.shape[0] - lv["h"] + 1, s.shape[1] - lv["w"] + 1), np.float32)
        self._check(self._lib.fpm_dbg_top_score(self._h, s.ctypes.data, s.shape[1], s.shape[0], out.ctypes.data))
        return out

    def dbgPeaks(self, score, tw, th, block_mode, thresh, max_overlap, max_picks):
        sc = np.ascontiguousarray(np.asarray(score, np.float32))
        picks = np.zeros((max_picks, 3), np.float64)
        n = C.c_int(0)
        self._check(self._lib.fpm_dbg_peaks(self._h, sc.ctypes.data, sc.shape[1], sc.shape[0], tw, th, int(block_mode),
                                            float(thresh), float(max_overlap), max_picks, picks.ctypes.data, C.byref(n)))
        return picks[:n.value]

    def dbgTopScoreProduction(self, img):
        """the top-layer map exactly as match() computes it; returns (map, reject_below)"""
        s = np.ascontiguousarray(_as_u8_2d(img))
        lv = self.templateLevels()[-1]
        out = np.zeros((s.shape[0] - lv["h"] + 1, s.shape[1] - lv["w"] + 1), np.float32)
        rb = C.c_float(0)
        self._check(self._lib.fpm_dbg_top_score_production(self._h, s.ctypes.data, s.shape[1], s.shape[0], out.ctypes.data, C.byref(rb)))
        return out, rb.value

    # ---- angle-sharded latency mode: one handle per GPU, two NCCL allgathers on device buffers (fpm_match_sharded) ----
    def setShardUpload(self, v: bool): self._set(L.PARAM_SHARD_UPLOAD, 1 if v else 0)
    def setAsyncDescent(self, v: int): self._set(L.PARAM_ASYNC_DESCENT, int(v))
    def setJpegDeviceHuffman(self, on: bool): self._set(L.PARAM_JPEG_DEVICE_HUFFMAN, 1 if on else 0)
    def getJpegPasses(self) -> int: return int(self._lib.fpm_get_param(self._h, L.PARAM_JPEG_PASSES))
    def collectiveCount(self) -> int: return int(self._lib.fpm_collective_count(self._h))

    def commInit(self, nranks: int, rank: int, unique_id: bytes):
        """collective: ncclCommInitRank on this handle's device with the 128-byte id made by comm_unique_id() on rank 0"""
        buf = C.create_string_buffer(bytes(unique_id), 128)
        self._check(self._lib.fpm_comm_init(self._h, nranks, rank, buf))

    def commDestroy(self): self._lib.fpm_comm_destroy(self._h)

    def matchSharded(self, sourceImage=None, ptr=None, shape=None, stride=None, on_device=False) -> List[SingleTargetMatch]:
        """collective over the communicator's ranks: every rank passes the SAME frame and receives the same result list"""
        cap = self.result_capacity
        if not hasattr(self, "_res_buf"):
            self._res_buf = (L.fpm_result * cap)()
        res, n = self._res_buf, C.c_int(0)
        if ptr is None:
            s = _as_u8_2d(sourceImage)
            ptr, shape, stride = s.ctypes.data, s.shape, s.strides[0]
        self._check(self._lib.fpm_match_sharded(self._h, ptr, shape[1], shape[0], stride, 1 if on_device else 0, res, cap, C.byref(n)))
        return _convert(res, min(n.value, cap))

    def matchSetSharded(self, sourceImage=None, ptr=None, shape=None, stride=None, on_device=False,
                        scaled: bool = False) -> List[List[SingleTargetMatch]]:
        """collective, the whole template set against one frame (fpm_match_set_sharded, scaled: fpm_match_set_sharded_scaled):
        every rank passes the SAME frame and receives the same [template][results] lists, equal to matchSet on one GPU"""
        cap, T = self.result_capacity, max(self.patternSetSize(), 1)
        res, counts = (L.fpm_result * (cap * T))(), (C.c_int * T)()
        if ptr is None:
            s = _as_u8_2d(sourceImage)
            ptr, shape, stride = s.ctypes.data, s.shape, s.strides[0]
        if not scaled:
            self._check(self._lib.fpm_match_set_sharded(self._h, ptr, shape[1], shape[0], stride, 1 if on_device else 0, res, cap,
                                                        counts))
            return self._set_results(res, counts, 1, T)[0]
        sc = (C.c_double * (cap * T))()
        self._check(self._lib.fpm_match_set_sharded_scaled(self._h, ptr, shape[1], shape[0], stride, 1 if on_device else 0, res, sc,
                                                           cap, counts))
        return self._set_results(res, counts, 1, T, sc)[0]

    def matchSetShardedMerged(self, sourceImage=None, max_overlap: Optional[float] = None, ptr=None, shape=None, stride=None,
                              on_device=False, scaled: bool = False) -> List[Tuple[int, SingleTargetMatch]]:
        """collective, merged as matchSetMerged (fpm_match_set_sharded_merged, scaled: fpm_match_set_sharded_scaled_merged):
        [(set index, result)] on every rank"""
        if max_overlap is None:
            raise FpmError("matchSetShardedMerged needs max_overlap")
        cap, T = self.result_capacity, max(self.patternSetSize(), 1)
        res, labels, count, set_counts = (L.fpm_result * cap)(), (C.c_int * cap)(), (C.c_int * 1)(), (C.c_int * T)()
        if ptr is None:
            s = _as_u8_2d(sourceImage)
            ptr, shape, stride = s.ctypes.data, s.shape, s.strides[0]
        if not scaled:
            self._check(self._lib.fpm_match_set_sharded_merged(self._h, ptr, shape[1], shape[0], stride, 1 if on_device else 0,
                                                               float(max_overlap), res, labels, cap, count, set_counts))
            return self._merged_results(res, labels, count, 1)[0]
        sc = (C.c_double * cap)()
        self._check(self._lib.fpm_match_set_sharded_scaled_merged(self._h, ptr, shape[1], shape[0], stride, 1 if on_device else 0,
                                                                  float(max_overlap), res, sc, labels, cap, count, set_counts))
        return self._merged_results(res, labels, count, 1, sc)[0]

    # ---- angle-sharded stage API ----
    def stageNumAngles(self, W, H) -> int: return self._lib.fpm_stage_num_angles(self._h, W, H)

    def stageTop(self, src, a0, a1, ptr=None, shape=None, stride=None) -> np.ndarray:
        cap = (self.getMaxPositions() + 5) * max(a1 - a0, 1)
        rows = np.zeros((cap, 5), np.float64)
        n = C.c_int(0)
        if ptr is None:
            s = _as_u8_2d(src)
            self._check(self._lib.fpm_stage_top(self._h, s.ctypes.data, s.shape[1], s.shape[0], s.strides[0], 0, a0, a1,
                                                rows.ctypes.data, cap, C.byref(n)))
        else:
            self._check(self._lib.fpm_stage_top(self._h, ptr, shape[1], shape[0], stride, 1, a0, a1, rows.ctypes.data, cap,
                                                C.byref(n)))
        return rows[:n.value]

    def stageSortCandidates(self, picks: np.ndarray) -> np.ndarray:
        p = np.ascontiguousarray(picks, np.float64).reshape(-1, 5)
        out = np.zeros_like(p)
        self._check(self._lib.fpm_stage_sort_candidates(self._h, p.ctypes.data, p.shape[0], out.ctypes.data))
        return out

    def stageRefine(self, cands: np.ndarray) -> np.ndarray:
        c = np.ascontiguousarray(cands, np.float64).reshape(-1, 5)
        rows = np.zeros((max(c.shape[0], 1), 5), np.float64)
        n = C.c_int(0)
        self._check(self._lib.fpm_stage_refine(self._h, c.ctypes.data, c.shape[0], rows.ctypes.data, rows.shape[0], C.byref(n)))
        return rows[:n.value]

    def stageFinal(self, refined: np.ndarray) -> List[SingleTargetMatch]:
        r = np.ascontiguousarray(refined, np.float64).reshape(-1, 5)
        cap = self.result_capacity
        res = (L.fpm_result * cap)()
        n = C.c_int(0)
        self._check(self._lib.fpm_stage_final(self._h, r.ctypes.data, r.shape[0], res, cap, C.byref(n)))
        return _convert(res, min(n.value, cap))


def rrect_overlap_host(r1, r2, max_overlap=0.0):
    """CPU evaluation of the NMS pair decision (shared host/device geometry code); for tests."""
    lib = L.load()
    a = (C.c_float * 5)(*r1)
    b = (C.c_float * 5)(*r2)
    typ, ratio = C.c_int(), C.c_double()
    d = lib.fpm_dbg_rrect_overlap(a, b, float(max_overlap), C.byref(typ), C.byref(ratio))
    return d, typ.value, ratio.value


def rrect_from3_host(p1, p2, p3):
    lib = L.load()
    pts = (C.c_float * 6)(p1[0], p1[1], p2[0], p2[1], p3[0], p3[1])
    out = (C.c_float * 5)()
    lib.fpm_dbg_rrect_from3(pts, out)
    return tuple(out)


def comm_available() -> bool:
    return bool(L.load().fpm_comm_available())


def comm_unique_id() -> bytes:
    """ncclGetUniqueId through the C ABI (rank 0 calls it and distributes the 128 bytes)"""
    buf = C.create_string_buffer(128)
    rc = L.load().fpm_comm_get_unique_id(buf)
    if rc != 0:
        raise FpmError("fpm_comm_get_unique_id failed (%d): libnccl.so.2 not loadable?" % rc)
    return buf.raw


def shard_angle_range(n_angles: int, nranks: int, rank: int):
    a0, a1 = C.c_int(), C.c_int()
    rc = L.load().fpm_shard_angle_range(n_angles, nranks, rank, C.byref(a0), C.byref(a1))
    if rc != 0:
        raise FpmError("fpm_shard_angle_range: bad arguments")
    return a0.value, a1.value


def match_sharded_virtual(matchers, sourceImage):
    """fpm_match_sharded_virtual: the angle-sharded pipeline with the given handles of ONE device as the ranks;
    returns one result list per rank (they must all be equal)."""
    s = _as_u8_2d(sourceImage)
    lib = matchers[0]._lib
    n = len(matchers)
    cap = min(m.result_capacity for m in matchers)
    hs = (C.c_void_p * n)(*[m._h for m in matchers])
    res = (L.fpm_result * (cap * n))()
    counts = (C.c_int * n)()
    rc = lib.fpm_match_sharded_virtual(hs, n, s.ctypes.data, s.shape[1], s.shape[0], s.strides[0], res, cap, counts)
    if rc != 0:
        errs = [lib.fpm_last_error(m._h).decode() for m in matchers]
        raise FpmError("fpm_match_sharded_virtual error %d: %s" % (rc, "; ".join(e for e in errs if e)))
    return [_convert(res[i * cap:(i + 1) * cap], min(counts[i], cap)) for i in range(n)]


def match_set_sharded_virtual(matchers, sourceImage, max_overlap=None, scaled=False):
    """fpm_match_set_sharded_virtual: the whole template set against one frame, angle-sharded over the given handles of ONE
    device as the ranks.  Returns one result per rank (they must all be equal): [template][results], or with max_overlap
    the merged [(set index, result)] list (fpm_match_set_sharded_merged_virtual).  scaled=True: the _scaled calls, which match
    at the handles' scale range and fill dScale."""
    s = _as_u8_2d(sourceImage)
    lib = matchers[0]._lib
    n = len(matchers)
    cap = min(m.result_capacity for m in matchers)
    T = max(matchers[0].patternSetSize(), 1)
    hs = (C.c_void_p * n)(*[m._h for m in matchers])
    args = (hs, n, s.ctypes.data, s.shape[1], s.shape[0], s.strides[0])
    sc = None
    name = "fpm_match_set_sharded%s%s_virtual" % ("_scaled" if scaled else "", "" if max_overlap is None else "_merged")
    fn = getattr(lib, name)
    if max_overlap is None:
        res, counts = (L.fpm_result * (cap * n * T))(), (C.c_int * (n * T))()
        if scaled:
            sc = (C.c_double * (cap * n * T))()
            rc = fn(*args, res, sc, cap, counts)
        else:
            rc = fn(*args, res, cap, counts)
    else:
        res, labels, counts, set_counts = (L.fpm_result * (cap * n))(), (C.c_int * (cap * n))(), (C.c_int * n)(), (C.c_int * (n * T))()
        if scaled:
            sc = (C.c_double * (cap * n))()
            rc = fn(*args, float(max_overlap), res, sc, labels, cap, counts, set_counts)
        else:
            rc = fn(*args, float(max_overlap), res, labels, cap, counts, set_counts)
    if rc != 0:
        errs = [lib.fpm_last_error(m._h).decode() for m in matchers]
        raise FpmError("%s error %d: %s" % (name, rc, "; ".join(e for e in errs if e)))

    def conv(i, m):
        return _convert(res[i * cap:(i + 1) * cap], m, None if sc is None else sc[i * cap:(i + 1) * cap])
    if max_overlap is None:
        return [[conv(r * T + t, min(counts[r * T + t], cap)) for t in range(T)] for r in range(n)]
    return [list(zip(labels[r * cap:r * cap + min(counts[r], cap)], conv(r, min(counts[r], cap)))) for r in range(n)]


# ---- multi-template matching ("NCC-based OCR", MatchTool/MatchToolDlg.cpp:718-770) --------------------------
OCR_LETTERS = "0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZ"          # chLetters, :723-725


def match_multi(matchers, sourceImage):
    """The same host image matched by several learned TemplateMatcher handles of one device, concurrently
    (fpm_match_multi).  Returns one result list per matcher."""
    if not matchers:
        return []
    s = _as_u8_2d(sourceImage)
    lib = matchers[0]._lib
    n = len(matchers)
    cap = min(m.result_capacity for m in matchers)
    hs = (C.c_void_p * n)(*[m._h for m in matchers])
    res = (L.fpm_result * (cap * n))()
    counts = (C.c_int * n)()
    rc = lib.fpm_match_multi(hs, n, s.ctypes.data, s.shape[1], s.shape[0], s.strides[0], res, cap, counts)
    if rc != 0:
        errs = [lib.fpm_last_error(m._h).decode() for m in matchers]
        raise FpmError("fpm_match_multi error %d: %s" % (rc, "; ".join(e for e in errs if e)))
    return [_convert(res[i * cap:(i + 1) * cap], min(counts[i], cap)) for i in range(n)]


def ocr_assemble(centres, labels, line_tol: float = 10.0) -> str:
    """fpm_ocr_assemble: centres [(cx, cy), ...] + one character each -> text lines (MatchToolDlg.cpp:752-771)."""
    lib = L.load()
    n = len(labels)
    if n == 0:
        return ""
    cx = (C.c_double * n)(*[float(c[0]) for c in centres])
    cy = (C.c_double * n)(*[float(c[1]) for c in centres])
    lab = C.create_string_buffer("".join(labels).encode("ascii"), n + 1)
    out = C.create_string_buffer(2 * n + 2)
    rc = lib.fpm_ocr_assemble(cx, cy, lab, n, float(line_tol), out, len(out))
    if rc < 0:
        raise FpmError("fpm_ocr_assemble error %d" % rc)
    return out.value.decode("ascii")


class GlyphReader:
    """One learned TemplateMatcher per glyph; read(image) = the upstream OCR loop: match every glyph, collect the
    centres with their letter, assemble lines.  readBatch(frames) reads many frames with one handle holding all glyphs as
    a template set (created on first use).  masks (optional): {letter: mask} for glyphs matched under a don't-care mask,
    e.g. their strokes; glyphs without an entry are unmasked.  scale_range=(lo, hi) among the params reads text printed lo..hi
    times the glyphs' size (setScaleRange on every handle; readBatch then uses the scaled set calls)."""

    def __init__(self, templates: dict, masks: Optional[dict] = None, device: int = 0, result_capacity: int = 256, **params):
        self.letters = [ch for ch in OCR_LETTERS if ch in templates] + sorted(k for k in templates if k not in OCR_LETTERS)
        self._templates = [templates[ch] for ch in self.letters]
        masks = masks or {}
        unknown = sorted(set(masks) - set(templates))
        if unknown:
            raise ValueError(f"masks for glyphs without a template: {unknown}")
        self._masks = [masks.get(ch) for ch in self.letters]
        self._device, self._capacity, self._params = device, result_capacity, params
        self._set_matcher = None
        self.matchers = []
        for ch, mk in zip(self.letters, self._masks):
            m = self._new_matcher()
            if not m.learnPattern(templates[ch], mk):
                raise FpmError("learnPattern failed for glyph %r" % ch)
            self.matchers.append(m)

    def _new_matcher(self):
        m = TemplateMatcher(self._device, result_capacity=self._capacity)
        for k, v in self._params.items():
            if k == "scale_range" and v is None:             # no range: the unscaled matcher
                continue
            {"max_pos": m.setMaxPositions, "max_overlap": m.setMaxOverlap, "score": m.setScore,
             "tolerance_angle": m.setToleranceAngle, "min_reduce_area": m.setMinReduceArea, "use_simd": m.setUseSIMD,
             "sub_pixel": m.setSubPixelEstimation, "scale_range": lambda r: m.setScaleRange(*r)}[k](v)
        return m

    def _assemble(self, per, line_tol):
        centres, labels = [], []
        for ch, res in zip(self.letters, per):
            for r in res:
                centres.append(r.ptCenter)
                labels.append(ch)
        return ocr_assemble(centres, labels, line_tol), dict(zip(self.letters, per))

    def readBatch(self, frames, line_tol: float = 10.0, merge_overlap: Optional[float] = None):
        """frames: [B, H, W] uint8 (or a list of equally sized images) -> [(text, {letter: results})] per frame.
        merge_overlap: None reads every glyph's own list; a float merges the glyphs' lists of a frame with NMS across
        glyphs at that overlap threshold (similar glyphs that hit the same cell, O/0/Q or 8/B, keep only the best) and
        {letter: results} holds the survivors."""
        if self._set_matcher is None:
            self._set_matcher = self._new_matcher()
            self._set_matcher.learnPatternSet(self._templates, self._masks if any(m is not None for m in self._masks) else None)
        f = np.ascontiguousarray(np.stack([_as_u8_2d(x) for x in frames]) if isinstance(frames, (list, tuple)) else frames, np.uint8)
        scaled = self._params.get("scale_range") is not None
        if merge_overlap is None:
            return [self._assemble(per, line_tol) for per in self._set_matcher.matchSetBatch(f, scaled=scaled)]
        out = []
        for merged in self._set_matcher.matchSetBatchMerged(f, merge_overlap, scaled=scaled):
            per = [[] for _ in self.letters]
            for t, r in merged:
                per[t].append(r)
            out.append(self._assemble(per, line_tol))
        return out

    def read(self, sourceImage, line_tol: float = 10.0):
        """Returns (text, {letter: [SingleTargetMatch, ...]})."""
        return self._assemble(match_multi(self.matchers, sourceImage), line_tol)
