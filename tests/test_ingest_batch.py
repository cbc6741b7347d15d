"""Batched JPEG ingest (fpm_ingest_jpeg_batch): the device unstuffing (a stream compaction over the entropy-coded segments of all
files) and the multi-file Huffman decoder, emulated on the CPU against the sequential references, then on the GPU against
cv2.imdecode, the single-file ingest and the batch matcher."""
import ctypes as C
import os

import cv2
import numpy as np
import pytest

from oracle import oracle as O
from tests.helpers import assert_results_match, configure, get_image
from tests.test_ingest import _host_luma, _jpeg_cases

GOLDEN_JPEG = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "jpeg")


def _lib():
    from fastest_image_pattern_matching_b200 import _lib as L
    return L.load()


def _golden(name):
    with open(os.path.join(GOLDEN_JPEG, name + ".jpg"), "rb") as f:
        return f.read()


def _scan_begin(data):
    """offset of the entropy-coded segment: the byte after the SOS segment"""
    i = data.index(b"\xff\xda")
    return i + 2 + (data[i + 2] << 8 | data[i + 3])


def _random_encoding(seed):
    """the generator of test_jpeg_decoders_on_random_encodings"""
    rng = np.random.default_rng(1000 + seed)
    h, w = int(rng.integers(1, 200)), int(rng.integers(1, 260))
    color = bool(rng.integers(0, 2))
    img = rng.integers(0, 256, (h, w, 3) if color else (h, w), dtype=np.uint8)
    if rng.integers(0, 2):
        img = cv2.GaussianBlur(img, (0, 0), float(rng.uniform(0.6, 4.0)))
    params = [cv2.IMWRITE_JPEG_QUALITY, int(rng.integers(5, 101))]
    if color:
        params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, int(rng.choice([cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420,
                                                                     cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440,
                                                                     cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444]))]
    if rng.integers(0, 2):
        params += [cv2.IMWRITE_JPEG_RST_INTERVAL, int(rng.integers(1, 9))]
    if rng.integers(0, 2):
        params += [cv2.IMWRITE_JPEG_OPTIMIZE, 1]
    return bytes(cv2.imencode(".jpg", img, params)[1])


def _damaged_files():
    """the 400 files of test_jpeg_parser_and_decoders_survive_damaged_files"""
    rng = np.random.default_rng(99)
    cases = _jpeg_cases()
    names = sorted(cases)
    out = []
    for it in range(400):
        data = bytearray(cases[names[it % len(names)]])
        if it % 3 == 0:
            for pos in rng.integers(2, min(len(data), 700), int(rng.integers(1, 6))):
                data[pos] = int(rng.integers(0, 256))
        elif it % 3 == 1:
            data = data[:int(rng.integers(2, len(data)))]
        else:
            for pos in rng.integers(2, len(data), int(rng.integers(1, 20))):
                data[pos] = int(rng.integers(0, 256))
        out.append(bytes(data))
    return out


def _with_fill_bytes(data, rng):
    """0xFF fill bytes inserted in front of every RST marker and in front of EOI (allowed by T.81 B.1.1.2)"""
    sb = _scan_begin(data)
    out = bytearray(data[:sb])
    i = sb
    while i < len(data):
        if data[i] == 0xFF and i + 1 < len(data) and (0xD0 <= data[i + 1] <= 0xD7 or data[i + 1] == 0xD9):
            out += b"\xff" * int(rng.integers(1, 4))
        out.append(data[i])
        i += 1
    return bytes(out)


def _unstuff(data, emulated):
    lib = _lib()
    buf = np.frombuffer(data, np.uint8)
    out = np.zeros(len(data) + 64, np.uint8)
    rst_cap = len(data) // 2 + 4
    rst = np.zeros(rst_cap, np.uint32)
    nbits, nint, tile = C.c_uint(), C.c_int(), C.c_int()
    rc = lib.fpm_dbg_jpeg_unstuff(buf.ctypes.data, buf.size, emulated, out.ctypes.data, out.size, rst.ctypes.data, rst_cap,
                                  C.byref(nbits), C.byref(nint), C.byref(tile))
    if rc != 0:
        return rc, None
    nb = nbits.value // 8
    return rc, (out[:nb + 16].tobytes(), rst[:nint.value + 1].tolist(), nbits.value, nint.value, tile.value)


def _unstuff_corpus():
    rng = np.random.default_rng(5)
    files = dict(_jpeg_cases())
    files["Src6"] = _golden("Src6")
    files["Dst10"] = _golden("Dst10")
    for s in range(20):
        files["random_%d" % s] = _random_encoding(s)
    for k, name in enumerate(("gray_restart_7", "gray_restart_1", "color_420_restart_2", "gray_q95", "color_420")):
        files["fill_" + name] = _with_fill_bytes(_jpeg_cases()[name], rng)
    files["last_byte_ff"] = _jpeg_cases()["gray_restart_7"][:-2] + b"\xff"
    files["last_byte_ff_mid_scan"] = _jpeg_cases()["gray_q95"][:len(_jpeg_cases()["gray_q95"]) // 2] + b"\xff"
    for k, d in enumerate(_damaged_files()):
        files["damaged_%03d" % k] = d
    files.update(_straddling(_unstuff(files["gray_q95"], 1)[1][4]))
    return files


def _straddling(tile):
    """an RST marker and an FF 00 pair moved onto a compaction tile boundary by fill bytes in front of an RST marker"""
    rng = np.random.default_rng(8)
    img = rng.integers(0, 256, (256, 256), dtype=np.uint8)
    data = bytes(cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, 100, cv2.IMWRITE_JPEG_RST_INTERVAL, 2])[1])
    sb = _scan_begin(data)
    rsts = [i for i in range(sb, len(data) - 1) if data[i] == 0xFF and 0xD0 <= data[i + 1] <= 0xD7]
    i = next(r for r in rsts if r >= sb + tile)
    pad = (sb + tile - 1 - i) % tile
    on_rst = data[:i] + b"\xff" * pad + data[i:]
    j = next(k for k in range(sb + tile, len(data) - 1) if data[k] == 0xFF and data[k + 1] == 0x00 and any(r < k for r in rsts[1:]))
    r = max(x for x in rsts if x < j)
    pad = (sb + tile - 1 - j) % tile
    on_ff00 = data[:r] + b"\xff" * pad + data[r:]
    return {"rst_on_tile_boundary": on_rst, "ff00_on_tile_boundary": on_ff00}


def test_device_unstuffing_emulated_equals_the_sequential_reference():
    """every byte, restart position, nbits and nint of the stream compaction equal jpeg_unstuff; at least one FF 00 pair and one
    RST marker straddle a compaction tile boundary"""
    straddle_ff00 = straddle_rst = 0
    compared = 0
    for name, data in _unstuff_corpus().items():
        rc0, want = _unstuff(data, 0)
        rc1, got = _unstuff(data, 1)
        assert rc0 == rc1, name
        if rc0 != 0:
            continue
        compared += 1
        assert got[0] == want[0], name
        assert got[1] == want[1], name
        assert got[2:4] == want[2:4], name
        tile = got[4]
        sb = _scan_begin(data)
        for i in range(sb + tile - 1, len(data) - 1, tile):     # the pair's first byte is a tile's last position
            if data[i] == 0xFF and data[i + 1] == 0x00:
                straddle_ff00 += 1
            if data[i] == 0xFF and 0xD0 <= data[i + 1] <= 0xD7:
                straddle_rst += 1
    assert compared > 200, compared
    assert straddle_ff00 >= 1 and straddle_rst >= 1, (straddle_ff00, straddle_rst)


def test_unstuffing_edge_cases():
    """a marker pair on a tile boundary, fill bytes before RST / EOI, 0xFF as the last byte, RSTn without DRI (ends the scan)"""
    base = _jpeg_cases()["gray_restart_1"]
    rc, r = _unstuff(base, 1)
    tile = r[4]
    sb = _scan_begin(base)
    # move an RST marker onto a tile boundary by padding the scan's first interval with fill bytes in front of its marker
    first_rst = next(i for i in range(sb, len(base) - 1) if base[i] == 0xFF and 0xD0 <= base[i + 1] <= 0xD7)
    for target in (tile - 1, tile, tile + 1, 2 * tile - 1):
        pad = (sb + target) - first_rst
        if pad < 0:
            continue
        data = base[:first_rst] + b"\xff" * pad + base[first_rst:]
        assert _unstuff(data, 1) == _unstuff(data, 0)
        assert _unstuff(data, 0)[1][0] == r[0]                     # fill bytes change nothing
    no_dri = _jpeg_cases()["gray_q95"]
    sb = _scan_begin(no_dri)
    p = next(k for k in range(sb + 100, len(no_dri)) if no_dri[k - 1] != 0xFF)
    data = no_dri[:p] + b"\xff\xd3" + no_dri[p:]
    rc, got = _unstuff(data, 1)
    assert got == _unstuff(data, 0)[1] and got[3] == 1
    assert got[2] == _unstuff(no_dri[:p] + b"\xff\xd9", 0)[1][2]


def _coef_shape(data):
    w, h, bw, bh, quant, coef = _host_luma(data)
    return coef


def _batch_emulation(files):
    lib = _lib()
    buf = np.frombuffer(b"".join(files), np.uint8)
    offs = np.zeros(len(files) + 1, np.uint64)
    offs[1:] = np.cumsum([len(f) for f in files])
    wants = [_coef_shape(f) for f in files]
    coffs = np.zeros(len(files) + 1, np.uint64)
    coffs[1:] = np.cumsum([c.size for c in wants])
    coef = np.zeros(int(coffs[-1]), np.int16)
    passes = np.zeros(len(files), np.int32)
    err = C.create_string_buffer(256)
    rc = lib.fpm_dbg_jpeg_luma_parallel_batch(buf.ctypes.data, offs.ctypes.data, len(files), coef.ctypes.data, coffs.ctypes.data,
                                              passes.ctypes.data, err, 256)
    assert rc == 0, err.value
    return [coef[int(coffs[i]):int(coffs[i + 1])].reshape(wants[i].shape) for i in range(len(files))], wants, passes


def _single_emulation_passes(data, shape):
    lib = _lib()
    buf = np.frombuffer(data, np.uint8)
    out = np.zeros(shape, np.int16)
    passes, err = C.c_int(), C.create_string_buffer(256)
    assert lib.fpm_dbg_jpeg_luma_parallel(buf.ctypes.data, buf.size, out.ctypes.data, out.size, C.byref(passes), err, 256) == 0
    return passes.value


@pytest.mark.parametrize("seed", range(4))
def test_batch_emulation_equals_the_single_file_decoders(seed):
    """mixed batches (grayscale, 4:2:0 / 4:2:2 / 4:1:1 / 4:4:4, restart intervals 1-8, optimised tables, quality 5-100, different
    sizes): per file the coefficients of the sequential decoder and the passes of the single-file emulation"""
    rng = np.random.default_rng(300 + seed)
    cases = _jpeg_cases()
    names = sorted(cases)
    files = [cases[names[int(i)]] for i in rng.permutation(len(names))[:6]]
    files += [_random_encoding(int(s)) for s in rng.integers(0, 40, 6)]
    if seed == 0:
        files.append(_golden("Dst10"))
    rng.shuffle(files)
    got, wants, passes = _batch_emulation(files)
    for f, g, w, p in zip(files, got, wants, passes):
        assert np.array_equal(g, w)
        assert p == _single_emulation_passes(f, w.shape)


def test_batch_emulation_of_identical_files_and_of_src6():
    files = [_golden("Src6"), _jpeg_cases()["gray_restart_7"], _golden("Src6")]
    got, wants, passes = _batch_emulation(files)
    for g, w in zip(got, wants):
        assert np.array_equal(g, w)
    assert passes[0] == passes[2] == _single_emulation_passes(files[0], wants[0].shape)


def test_batch_emulation_rejects_with_the_file_index():
    lib = _lib()
    prog = bytes(cv2.imencode(".jpg", np.zeros((16, 16), np.uint8), [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1])
    good = _jpeg_cases()["gray_q95"]
    files = [good, prog, good]
    buf = np.frombuffer(b"".join(files), np.uint8)
    offs = np.array([0, len(good), len(good) + len(prog), len(buf)], np.uint64)
    coef = np.zeros(1 << 20, np.int16)
    coffs = np.array([0, 1 << 18, 1 << 19, 1 << 20], np.uint64)
    err = C.create_string_buffer(256)
    rc = lib.fpm_dbg_jpeg_luma_parallel_batch(buf.ctypes.data, offs.ctypes.data, 3, coef.ctypes.data, coffs.ctypes.data, None, err, 256)
    assert rc != 0 and b"file 1" in err.value and b"progressive" in err.value


# ---------------------------------------------------------------- GPU ----------------------------------------------------------
def _mixed_same_size(n, h=203, w=317, seed=0):
    rng = np.random.default_rng(seed)
    gray = cv2.GaussianBlur(rng.integers(0, 256, (h, w), dtype=np.uint8), (0, 0), 2.0)
    col = cv2.GaussianBlur(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), (0, 0), 1.5)
    Q, SS, RST = cv2.IMWRITE_JPEG_QUALITY, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_RST_INTERVAL
    subs = [cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411,
            cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444]
    files = []
    for i in range(n):
        p = [Q, int(rng.integers(5, 101))]
        if i % 5 == 0:
            img = gray
        else:
            img = col
            p += [SS, subs[i % 4]]
        if i % 3 == 1:
            p += [RST, int(rng.integers(1, 9))]
        if i % 4 == 3:
            p += [cv2.IMWRITE_JPEG_OPTIMIZE, 1]
        files.append(bytes(cv2.imencode(".jpg", img, p)[1]))
    return files


def _decoded(data):
    return cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_GRAYSCALE)


@pytest.mark.gpu
def test_gpu_batch_equals_cv2_and_the_single_file_ingest(matcher):
    files = _mixed_same_size(16)
    for device_huffman in (True, False):
        matcher.setJpegDeviceHuffman(device_huffman)
        w, h = matcher.ingestJpegBatch(files)
        assert (h, w) == (203, 317) and matcher.ingestedCount() == 16
        assert (matcher.getJpegPasses() > 0) == device_huffman
        got = [matcher.ingestedFramePixels(i) for i in range(16)]
        for f, g in zip(files, got):
            assert np.array_equal(g, _decoded(f))
            matcher.ingestJpeg(f)
            assert matcher.ingestedCount() == 1
            assert np.array_equal(matcher.ingestedPixels(), g)
    matcher.setJpegDeviceHuffman(True)


@pytest.mark.gpu
def test_gpu_batch_of_src6_and_its_reencodings(matcher):
    src6 = _golden("Src6")
    fixture = get_image("Src6")
    re = [bytes(cv2.imencode(".jpg", fixture, [cv2.IMWRITE_JPEG_QUALITY, q] + extra)[1])
          for q, extra in ((90, []), (95, [cv2.IMWRITE_JPEG_RST_INTERVAL, 4]), (75, [cv2.IMWRITE_JPEG_OPTIMIZE, 1]))]
    files = [src6] * 8 + re
    matcher.ingestJpegBatch(files)
    for i in range(8):
        assert np.array_equal(matcher.ingestedFramePixels(i), fixture)
    for i, f in enumerate(re):
        assert np.array_equal(matcher.ingestedFramePixels(8 + i), _decoded(f))


@pytest.mark.gpu
def test_gpu_batch_in_waves_equals_one_wave(matcher):
    files = _mixed_same_size(12, 480, 640, seed=3)
    matcher.ingestJpegBatch(files)
    one = [matcher.ingestedFramePixels(i) for i in range(12)]
    matcher.setWorkspaceMB(1.2)                                  # ~0.9 MB of coefficients and states per 640x480 file
    matcher.setProfile(True)
    matcher.profileReset()
    try:
        matcher.ingestJpegBatch(files)
        idct = matcher.profile()["fpm_ingest_jpeg_idct_kernel"][1]
        waves = [matcher.ingestedFramePixels(i) for i in range(12)]
    finally:
        matcher.setWorkspaceMB(4096)
        matcher.setProfile(False)
    assert idct >= 3                                             # one IDCT launch per wave
    for a, b, f in zip(one, waves, files):
        assert np.array_equal(a, b) and np.array_equal(a, _decoded(f))


@pytest.mark.gpu
def test_gpu_match_ingested_batch_equals_match_batch(matcher, golden_cases):
    import bench
    tpl, frames = bench.make_frames(3, 11, "cfg1")
    wl = bench.WORKLOADS["cfg1"]
    bench.configure(matcher, wl)
    assert matcher.learnPattern(tpl)
    files = [bytes(cv2.imencode(".jpg", f, [cv2.IMWRITE_JPEG_QUALITY, 90])[1]) for f in frames]
    matcher.ingestJpegBatch(files)
    got = matcher.matchIngestedBatch()
    want = matcher.matchBatch(np.stack([_decoded(f) for f in files]))
    assert len(got) == 3
    for g, w in zip(got, want):
        assert_results_match(g, w, 0, 0, 0)
    c = golden_cases["cfg3_src6"]
    configure(matcher, c["params"])
    assert matcher.learnPattern(get_image(c["tpl"]))
    src6 = _golden("Src6")
    matcher.ingestJpegBatch([src6] * 4)
    got = matcher.matchIngestedBatch()
    want = matcher.matchBatch(np.stack([_decoded(src6)] * 4))
    for g, w in zip(got, want):
        assert_results_match(g, w, 0, 0, 0)
        assert_results_match(g, c["results"])
    configure(matcher, {})                                       # the session matcher's defaults again


@pytest.mark.gpu
def test_gpu_batch_launches_and_a_missing_restart_marker(matcher):
    from fastest_image_pattern_matching_b200 import FpmError
    src6 = _golden("Src6")
    matcher.ingestJpegBatch([src6])
    n0 = matcher.launchCount()
    matcher.ingestJpegBatch([src6])
    one = matcher.launchCount() - n0
    n0 = matcher.launchCount()
    matcher.ingestJpegBatch([src6] * 16)
    assert matcher.launchCount() - n0 == one                     # identical files need identical passes in one wave
    good = _jpeg_cases()["gray_restart_7"]
    sb = _scan_begin(good)
    k = next(i for i in range(sb, len(good) - 1) if good[i] == 0xFF and 0xD0 <= good[i + 1] <= 0xD7)
    bad = good[:k] + good[k + 2:]                                # one RST marker removed: the host decoder takes the file
    try:
        matcher.ingestJpeg(bad)
        alone = matcher.ingestedPixels()
    except FpmError as e:
        alone = str(e)
    try:
        matcher.ingestJpegBatch([good, bad, good])
        batch = matcher.ingestedFramePixels(1)
        assert np.array_equal(matcher.ingestedFramePixels(0), O.ingest_image(good))
    except FpmError as e:
        batch = str(e).replace("JPEG file 1 of the batch: ", "")
    if isinstance(alone, str):
        assert isinstance(batch, str) and batch == alone
    else:
        assert np.array_equal(batch, alone)


@pytest.mark.gpu
def test_gpu_batch_rejections(matcher):
    from fastest_image_pattern_matching_b200 import FpmError
    files = _mixed_same_size(4)
    img = np.zeros((203, 317), np.uint8)
    png = bytes(cv2.imencode(".png", img)[1])
    prog = bytes(cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1])
    other = bytes(cv2.imencode(".jpg", np.zeros((40, 50), np.uint8))[1])
    lib, h = matcher._lib, matcher._h
    good = np.frombuffer(b"".join(files), np.uint8)
    offs = np.zeros(5, np.uint64)
    offs[1:] = np.cumsum([len(f) for f in files])

    def rejected(call, word=None):
        matcher.ingestJpegBatch(files)                           # a good batch in front: the error must clear it
        assert matcher.ingestedCount() == 4
        with pytest.raises(FpmError) as e:
            call()
        if word:
            assert word in str(e.value), str(e.value)
        assert matcher.ingestedCount() == 0
        with pytest.raises(FpmError):
            matcher.ingestedFramePixels(0)

    rejected(lambda: matcher.ingestJpegBatch([]), "empty")
    rejected(lambda: matcher._check(lib.fpm_ingest_jpeg_batch(h, None, offs.ctypes.data, 4, None, None)))
    bad_offs = offs.copy()
    bad_offs[2] = bad_offs[1] - 1
    rejected(lambda: matcher.ingestJpegBatch(good, bad_offs), "decrease")
    rejected(lambda: matcher.ingestJpegBatch(files[:2] + [png] + files[2:]), "file 2")
    rejected(lambda: matcher.ingestJpegBatch(files[:1] + [prog] + files[1:]), "progressive")
    rejected(lambda: matcher.ingestJpegBatch(files[:3] + [other]), "file 3")
    matcher.ingestJpegBatch(files)
    for i, f in enumerate(files):
        assert np.array_equal(matcher.ingestedFramePixels(i), _decoded(f))
    for call in (matcher.ingestedPixels, matcher.matchIngested, matcher.learnIngested):
        with pytest.raises(FpmError) as e:
            call()
        assert "4 frames" in str(e.value)
    for idx in (-1, 4):
        with pytest.raises(FpmError):
            matcher.ingestedFramePixels(idx)


@pytest.mark.gpu
def test_gpu_batch_survives_damaged_scans(matcher):
    """the damage kinds of test_gpu_jpeg_ingest_survives_damaged_scans inside batches: frames of the right size or an error, and
    the next good batch is bit-exact"""
    from fastest_image_pattern_matching_b200 import FpmError
    rng = np.random.default_rng(23)
    for name in ("gray_q95", "color_420", "gray_restart_7"):
        good = _jpeg_cases()[name]
        want = O.ingest_image(good)
        for trial in range(6):
            bad = bytearray(good)
            lo = len(bad) // 2
            if trial < 4:
                for pos in rng.integers(lo, len(bad) - 2, 12):
                    bad[pos] = int(rng.integers(0, 255))
            else:
                bad = bad[:lo + int(rng.integers(0, len(bad) - lo - 2))]
            try:
                w, h = matcher.ingestJpegBatch([good, bytes(bad), good])
                assert (h, w) == want.shape and matcher.ingestedCount() == 3
                assert matcher.ingestedFramePixels(1).shape == want.shape
                assert np.array_equal(matcher.ingestedFramePixels(2), want)
            except FpmError:
                assert matcher.ingestedCount() == 0
        matcher.ingestJpegBatch([good] * 3)
        for i in range(3):
            assert np.array_equal(matcher.ingestedFramePixels(i), want)
