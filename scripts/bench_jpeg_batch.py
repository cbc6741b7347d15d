"""Batched JPEG ingest: 64-file steps of fpm_ingest_jpeg_batch alone and with fpm_match_ingested_batch, against a loop of
fpm_ingest_jpeg + fpm_match_ingested over the same files and against fpm_match_batch on the decoded frames from pinned memory
(the raw-pixel arm of bench.py on the same frames).  cfg1 (seeded frames from bench.make_frames, Dst7) and cfg3 (Src6, Dst6),
encoded by cv2.imencode at quality 90 and 95 (cfg3 also Src6.jpg as it is), packed into one pinned buffer.  Every timing is a
host clock around calls that end in a device synchronise, after warm-up, over at least 0.5 s.  The results of the timed step
are checked against fpm_match_batch on the cv2.imdecode frames (counts equal, records bit-equal); a separate profiled step gives
where the time goes.  Prints one JSON line.
    python scripts/bench_jpeg_batch.py [--batch 64] [--distinct 8]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
import cv2  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402
import bench  # noqa: E402
from fastest_image_pattern_matching_b200 import TemplateMatcher  # noqa: E402
from fastest_image_pattern_matching_b200 import _lib as L  # noqa: E402


def timed(fn, min_s=0.5, warmup=2):
    """ms per call: host clock around calls that each end in a device synchronise"""
    for _ in range(warmup):
        fn()
    n, t0 = 0, time.perf_counter()
    while True:
        fn()
        n += 1
        el = time.perf_counter() - t0
        if el >= min_s and n >= 3:
            return round(el / n * 1e3, 3)


def records(res, counts, cap, B):
    return [[tuple(getattr(res[b * cap + i], f) for f, _ in L.fpm_result._fields_) for i in range(counts[b])] for b in range(B)]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                               timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                                   # noqa: BLE001
        power = "unknown (%s)" % e
    return name, power


def run_case(m, wl_name, frames, files, B):
    """files: B JPEG file images; frames: their cv2.imdecode frames [B, H, W]"""
    lib, h = m._lib, m._h
    cap = m.result_capacity
    H, W = frames.shape[1:]
    sizes = [len(f) for f in files]
    offs = np.zeros(B + 1, np.uint64)
    offs[1:] = np.cumsum(sizes)
    packed = torch.empty(int(offs[-1]), dtype=torch.uint8).pin_memory()
    packed.numpy()[:] = np.frombuffer(b"".join(files), np.uint8)
    ptr = packed.data_ptr()
    pinned_frames = torch.from_numpy(np.ascontiguousarray(frames)).pin_memory()
    res = (L.fpm_result * (cap * B))()
    counts = (C.c_int * B)()
    w, hh = C.c_int(), C.c_int()

    def ingest():
        m._check(lib.fpm_ingest_jpeg_batch(h, ptr, offs.ctypes.data, B, C.byref(w), C.byref(hh)))

    def ingest_match():
        ingest()
        m._check(lib.fpm_match_ingested_batch(h, res, cap, counts))

    def loop():
        for i in range(B):
            m._check(lib.fpm_ingest_jpeg(h, ptr + int(offs[i]), sizes[i], None, None))
            n = C.c_int()
            m._check(lib.fpm_match_ingested(h, res, cap, C.byref(n)))

    def raw():
        m.matchBatchRaw(pinned_frames.data_ptr(), B, W, H, W, H * W, False, res, counts)

    out = {"mean_file_bytes": int(np.mean(sizes)), "frame_bytes": H * W}
    out["ingest_batch_ms"] = timed(ingest)
    out["passes"] = m.getJpegPasses()
    out["ingest_match_batch_ms"] = timed(ingest_match)
    got = records(res, counts, cap, B)
    out["single_file_loop_ms"] = timed(loop, warmup=1)
    out["match_batch_pinned_pixels_ms"] = timed(raw)
    m.matchBatchRaw(pinned_frames.data_ptr(), B, W, H, W, H * W, False, res, counts)
    want = records(res, counts, cap, B)
    out["results_equal_match_batch"] = got == want
    out["targets_per_frame"] = sorted(set(len(r) for r in got))
    out["ingest_match_images_per_s"] = round(B / out["ingest_match_batch_ms"] * 1e3, 1)
    out["match_batch_pinned_images_per_s"] = round(B / out["match_batch_pinned_pixels_ms"] * 1e3, 1)
    # where the time of one step goes (profiled separately: the events slow the host)
    m.setProfile(True)
    m.profileReset()
    t0 = time.perf_counter()
    ingest_match()
    out["profiled_step_ms"] = round((time.perf_counter() - t0) * 1e3, 3)
    prof = m.profile()
    m.setProfile(False)
    out["profile_ms"] = {k: round(v[0], 3) for k, v in prof.items() if v[1] > 0}
    assert out["results_equal_match_batch"], wl_name
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--distinct", type=int, default=8, help="distinct cfg1 frames, repeated to fill the batch")
    args = ap.parse_args()
    B = args.batch
    name, power = card()
    result = {"bench": "jpeg_batch", "gpu": name, "power_limit": power, "batch": B, "cases": {}}
    m = TemplateMatcher(0, result_capacity=256)
    for wl_name in ("cfg1", "cfg3"):
        wl = bench.WORKLOADS[wl_name]
        tpl, frames = bench.make_frames(args.distinct, 1000, wl_name)
        bench.configure(m, wl)
        assert m.learnPattern(tpl)
        encodings = [("q90", 90), ("q95", 95)]
        if wl_name == "cfg3":
            encodings.append(("Src6.jpg", None))
        for label, q in encodings:
            if q is None:
                data = open(os.path.join(ROOT, "tests", "golden", "jpeg", "Src6.jpg"), "rb").read()
                files = [data] * B
            else:
                enc = [bytes(cv2.imencode(".jpg", f, [cv2.IMWRITE_JPEG_QUALITY, q])[1]) for f in frames]
                files = [enc[i % len(enc)] for i in range(B)]
            dec = np.stack([cv2.imdecode(np.frombuffer(f, np.uint8), cv2.IMREAD_GRAYSCALE) for f in files])
            result["cases"]["%s_%s" % (wl_name, label)] = run_case(m, wl_name, dec, files, B)
            print(json.dumps({"case": "%s_%s" % (wl_name, label), **result["cases"]["%s_%s" % (wl_name, label)]}), file=sys.stderr)
    m.close()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
