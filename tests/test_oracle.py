"""CPU tests: the oracle against its pins (known answers, golden vectors, the reference's own
IM_Conv_SIMD build, cv2 for every OpenCV model the CUDA kernels restate)."""
import ctypes
import json
import os

import cv2
import numpy as np
import pytest

from oracle import oracle as O
from oracle import models as M
from tests.helpers import assert_results_match, configure, get_image, imconv_pin_digest, imconv_pin_inputs

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


# ---- known answers of the reference (README / Result Images, SURVEY.md section 4) ----
@pytest.mark.parametrize("case,count", [("test4_src3", 36), ("cfg3_src6", 15), ("src8", 3), ("src9", 1)])
def test_known_answer_counts(golden_cases, oracle_lib, case, count):
    c = golden_cases[case]
    assert len(c["results"]) == count
    m = configure(O.OracleMatcher(), c["params"])
    assert m.learn_pattern(get_image(c["tpl"]))
    res = m.match(get_image(c["src"]))
    assert len(res) == count
    assert_results_match(res, c["results"], 0, 0, 0)      # oracle is deterministic: identical to golden


def test_cfg1_recovers_readme_poses(golden_cases):
    # README.md:47-49 poses (synthetic Src7: Dst7 pasted there); MFC angle sign = -Qt sign
    from fpm_workloads import CFG1_POSES
    res = golden_cases["cfg1_synth"]["results"]
    assert len(res) == 3
    for (cx, cy, a) in CFG1_POSES:
        best = min(res, key=lambda r: abs(r["cx"] - cx) + abs(r["cy"] - cy))
        assert abs(best["cx"] - cx) < 1.0 and abs(best["cy"] - cy) < 1.0
        d = (best["angle"] + a + 180) % 360 - 180
        assert abs(d) < 0.2


def test_numpy_and_sse2_numerators_agree(oracle_lib):
    rng = np.random.default_rng(0)
    for (tw, th) in [(12, 9), (54, 54), (191, 131), (33, 17)]:
        tpl = rng.integers(0, 256, (th, tw), dtype=np.uint8)
        src = rng.integers(0, 256, (th + 6, tw + 6), dtype=np.uint8)
        a = O.match_template_simd_numpy(src, tpl)
        assert O._load_rowdot()
        b = O.match_template_simd(src, tpl)
        assert np.array_equal(a, b)


def test_restated_simd_matches_reference_build(oracle_lib):
    """The oracle's restatements of the reference's IM_Conv_SIMD (SSE2 C and numpy) return the stored values of
    tests/golden/imconv_ref.json; so does oracle/_ref/libimconv_ref.so, the reference's own IM_Conv_SIMD compiled from
    its source (oracle/build_ref.sh), wherever that build is present."""
    with open(os.path.join(ROOT, "tests", "golden", "imconv_ref.json")) as f:
        golden = json.load(f)
    rows, cells = imconv_pin_inputs()
    assert imconv_pin_digest(rows, cells) == golden["inputs_sha256"], "the seeded stream no longer draws the stored inputs"
    lib = O._load_rowdot()
    assert lib, "oracle/libncc_rowdot.so not built"
    lib.oracle_row_dot.restype = ctypes.c_int
    for (k, c), want in zip(rows, golden["row_dot"]):
        assert int((k.astype(np.int64) * c).sum()) == want
        assert lib.oracle_row_dot(k.ctypes.data, c.ctypes.data, k.size) == want
    # bright rows: float accumulation rounds -- restatement must round identically
    for (tpl, src), want in zip(cells, golden["cell"]):
        got = O.match_template_simd(src, tpl)[0, 0]
        assert np.float32(want) == got
        assert O.match_template_simd_numpy(src, tpl)[0, 0] == got
    ref_path = os.path.join(ROOT, "oracle", "_ref", "libimconv_ref.so")
    if os.path.exists(ref_path):
        ref = ctypes.CDLL(ref_path)
        ref.ref_IM_Conv_SIMD.restype = ctypes.c_int
        ref.ref_cell.restype = ctypes.c_float
        for (k, c), want in zip(rows, golden["row_dot"]):
            assert ref.ref_IM_Conv_SIMD(k.ctypes.data, c.ctypes.data, k.size) == want
        for (tpl, src), want in zip(cells, golden["cell"]):
            th, tw = tpl.shape
            assert np.float32(ref.ref_cell(tpl.ctypes.data, tw, th, src.ctypes.data, tw)) == np.float32(want)


# ---- OpenCV models the CUDA kernels restate, pinned against cv2 itself ----
@pytest.mark.parametrize("shape", [(7, 9), (1, 1), (2, 5), (480, 640), (101, 333), (64, 47), (1519, 2013)])
def test_pyrdown_model(shape):
    rng = np.random.default_rng(shape[0] * 7 + shape[1])
    img = rng.integers(0, 256, shape, dtype=np.uint8)
    assert np.array_equal(M.pyrdown(img), cv2.pyrDown(img))


def test_warp_affine_model():
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (190, 253), dtype=np.uint8)
    for ang in [0.0, 9.462, 90.0, -37.3, 180.0, 123.456]:
        for border in (0, 255):
            m = cv2.getRotationMatrix2D((126.0, 94.5), ang, 1)
            m[0, 2] += 13.5
            m[1, 2] -= 7.25
            want = cv2.warpAffine(img, m, (280, 220), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=border)
            got = M.warp_affine(img, m, (280, 220), border)
            assert np.array_equal(got, want), (ang, border)


def test_rotation_matrix_model():
    for ang in [0, 33.3, -120.15, 270]:
        a = cv2.getRotationMatrix2D((100.5, 50.25), ang, 1)
        assert np.array_equal(M.rotation_matrix(100.5, 50.25, ang), a)


def test_mean_stddev_model():
    rng = np.random.default_rng(3)
    for shape in [(521, 762), (9, 12), (54, 54), (131, 191)]:
        img = rng.integers(0, 256, shape, dtype=np.uint8)
        mean, sdv = cv2.meanStdDev(img)
        m2, s2 = M.mean_stddev(img)
        assert mean[0, 0] == m2 and sdv[0, 0] == s2


def test_rectangle_paint_model():
    for rect in [(3, 4, 5, 6), (-3, -2, 6, 5), (18, 17, 10, 10), (5, 5, 0, 3), (5, 5, -2, 3), (0, 0, 1, 1)]:
        a = np.zeros((20, 22), np.float32)
        cv2.rectangle(a, rect, -1.0, cv2.FILLED)
        b = np.zeros((20, 22), np.float32)
        M.paint(b, *rect)
        assert np.array_equal(a, b), rect


def test_minmaxloc_first_in_scan_order():
    a = np.zeros((5, 7), np.float32)
    a[3, 2] = a[1, 6] = a[1, 4] = 2.0
    _, mx, _, loc = cv2.minMaxLoc(a)
    assert mx == 2.0 and loc == (4, 1)
    assert O._min_max_loc(a) == (2.0, (4, 1))


def test_top_numerator_exact_vs_cv(golden_cases):
    """cv::matchTemplate (DFT float) vs the exact integer numerator: identical candidate list (SURVEY 7.4)."""
    c = golden_cases["src8"]
    src, tpl = get_image(c["src"]), get_image(c["tpl"])
    outs = []
    for mode in ("exact", "cv"):
        m = configure(O.OracleMatcher(), c["params"])
        m.top_numerator = mode
        m.trace = {}
        m.learn_pattern(tpl)
        res = m.match(src)
        outs.append((res, m.trace["cands"]))
    assert len(outs[0][0]) == len(outs[1][0])
    assert [(c0[0], c0[2]) for c0 in outs[0][1]] == [(c1[0], c1[2]) for c1 in outs[1][1]]
    assert_results_match(outs[0][0], outs[1][0])


def test_guards_and_edge_cases():
    m = O.OracleMatcher()
    assert m.match(np.zeros((10, 10), np.uint8)) == []          # not learned
    assert not m.learn_pattern(np.zeros((0, 0), np.uint8))
    tpl = np.full((40, 40), 7, np.uint8)
    tpl[10:30, 10:30] = 200
    assert m.learn_pattern(tpl)
    assert m.match(np.zeros((20, 100), np.uint8)) == []         # template taller than source
    assert m.match(np.zeros((30, 30), np.uint8)) == []          # template area larger


@pytest.mark.parametrize("shape", [(211, 300), (216, 288), (90, 301)])
def test_block_max_variants_agree_with_plain_search_without_ties(shape):
    """SURVEY 8a row 9: on a tie-free score map the Qt s_BlockMax, the MFC s_BlockMax and the plain minMaxLoc path
    return the identical ordered pick list (they can differ only on exact float ties)."""
    rng = np.random.default_rng(shape[0])
    n = shape[0] * shape[1]
    score = rng.permutation(np.linspace(-0.2, 0.9, n).astype(np.float32)).reshape(shape)
    assert len(np.unique(score)) == score.size                 # no ties
    om = O.OracleMatcher()
    om.max_pos, om.max_overlap = 25, 0.2
    plain = om.top_picks(score.copy(), (9, 7), 0.3, False)
    qt = om.top_picks(score.copy(), (9, 7), 0.3, True)
    om.mfc_compat = True
    mfc = om.top_picks(score.copy(), (9, 7), 0.3, True)
    assert len(plain) > 5 and plain == qt == mfc


def test_block_max_tie_rules_differ_as_documented():
    """two equal maxima in different blocks: Qt keeps the FIRST maximal block (std::max_element, DataStructures.h:241-245),
    MFC the LAST one (>=, MatchToolDlg.h:206)"""
    score = np.zeros((60, 80), np.float32)
    score[5, 6] = 1.0
    score[50, 70] = 1.0
    om = O.OracleMatcher()
    om.max_pos, om.max_overlap = 1, 0.0
    assert om.top_picks(score.copy(), (9, 7), 0.5, True)[0][0] == (6, 5)
    om.mfc_compat = True
    assert om.top_picks(score.copy(), (9, 7), 0.5, True)[0][0] == (70, 50)


# ---------------- round 2: sub-pixel arithmetic pins (src/TemplateMatcher.cpp:1002-1072) ----------------
def _det3(m):
    return (m[0, 0] * (m[1, 1] * m[2, 2] - m[1, 2] * m[2, 1]) - m[0, 1] * (m[1, 0] * m[2, 2] - m[1, 2] * m[2, 0]) +
            m[0, 2] * (m[1, 0] * m[2, 1] - m[1, 1] * m[2, 0]))


def _solve3_closed_form(S, b):
    """cv::solve(3x3, DECOMP_LU) for doubles -- the arithmetic fpm_subpix uses for K1^-1 K2"""
    d = 1.0 / _det3(S)
    t0 = ((S[1, 1] * S[2, 2] - S[1, 2] * S[2, 1]) * b[0] + (S[0, 2] * S[2, 1] - S[0, 1] * S[2, 2]) * b[1] + (S[0, 1] * S[1, 2] - S[0, 2] * S[1, 1]) * b[2]) * d
    t1 = ((S[1, 2] * S[2, 0] - S[1, 0] * S[2, 2]) * b[0] + (S[0, 0] * S[2, 2] - S[0, 2] * S[2, 0]) * b[1] + (S[0, 2] * S[1, 0] - S[0, 0] * S[1, 2]) * b[2]) * d
    t2 = ((S[1, 0] * S[2, 1] - S[1, 1] * S[2, 0]) * b[0] + (S[0, 1] * S[2, 0] - S[0, 0] * S[2, 1]) * b[1] + (S[0, 0] * S[1, 1] - S[0, 1] * S[1, 0]) * b[2]) * d
    return np.array([t0, t1, t2])


def test_cv_solve_3x3_closed_form_is_bit_exact():
    """`matK1.inv() * matK2` (:1066) is evaluated by OpenCV's MatExpr layer as cv::solve(K1, K2, DECOMP_LU); for a 3x3
    double system that is the adjugate closed form restated in fpm_subpix -- pinned bit for bit against cv2.solve"""
    rng = np.random.default_rng(0)
    for _ in range(2000):
        S = rng.normal(size=(3, 3))
        S = S + S.T
        b = rng.normal(size=3)
        ok, x = cv2.solve(S, b.reshape(3, 1), flags=cv2.DECOMP_LU)
        assert ok and np.array_equal(x.ravel(), _solve3_closed_form(S, b))


def _lu_inverse(Ain):
    """cv::invert(DECOMP_LU) for n > 3: hal::LU64f (LUImpl, partial pivoting, eps = 100*DBL_EPSILON) on [A | I]"""
    A = Ain.copy()
    m = A.shape[0]
    B = np.eye(m)
    eps = np.finfo(float).eps * 100
    for i in range(m):
        k = i
        for j in range(i + 1, m):
            if abs(A[j, i]) > abs(A[k, i]):
                k = j
        if abs(A[k, i]) < eps:
            return np.zeros_like(B)
        if k != i:
            A[[i, k], i:] = A[[k, i], i:]
            B[[i, k]] = B[[k, i]]
        d = -1 / A[i, i]
        for j in range(i + 1, m):
            al = A[j, i] * d
            for kk in range(i + 1, m):
                A[j, kk] += al * A[i, kk]
            for kk in range(m):
                B[j, kk] += al * B[i, kk]
    for i in range(m - 1, -1, -1):
        for j in range(m):
            s = B[i, j]
            for k in range(i + 1, m):
                s -= A[i, k] * B[k, j]
            B[i, j] = s / A[i, i]
    return B


def test_subpixel_fit_is_well_inside_the_tolerance_in_fp64():
    """The 10x10 normal equations mix pixels and radians (cond(AtA) ~ 1e10..1e11): a strictly sequential, FMA-free
    restatement of the chain (= the GPU's fpm_subpix, compiled with -fmad=false) and cv2's own gemm/invert/solve (SIMD
    dispatched, FMA contracted on this host) must agree far inside 0.05 px / 0.01 deg -- so the north_star tolerance
    holds for sub-pixel mode too, whatever the host's OpenCV dispatch does."""
    rng = np.random.default_rng(5)
    worst = 0.0
    for it in range(40):
        xm, ym = float(rng.integers(1, 6)), float(rng.integers(1, 6))
        tm, step = float(rng.uniform(-180, 180)), float(rng.uniform(0.1, 9.0))
        A = np.zeros((27, 10))
        S = np.zeros(27)
        row = 0
        peak = rng.uniform(0.8, 1.0)
        for theta in range(3):
            for y in (-1, 0, 1):
                for x in (-1, 0, 1):
                    dx, dy = xm + x, ym + y
                    dt = (tm + (theta - 1) * step) * O.D2R
                    A[row] = [dx * dx, dy * dy, dt * dt, dx * dy, dx * dt, dy * dt, dx, dy, dt, 1.0]
                    S[row] = np.float32(peak - 0.01 * ((x - 0.2) ** 2 + (y + 0.3) ** 2) - 0.004 * (theta - 1.1) ** 2 + rng.normal(0, 1e-4))
                    row += 1
        # cv2 chain (the oracle's)
        ata = cv2.gemm(A, A, 1, None, 0, flags=cv2.GEMM_1_T)
        zc = cv2.gemm(cv2.gemm(cv2.invert(ata)[1], A, 1, None, 0, flags=cv2.GEMM_2_T), S.reshape(-1, 1), 1, None, 0).ravel()
        # sequential chain (the GPU's)
        AtA = np.zeros((10, 10))
        for i in range(10):
            for j in range(10):
                s = 0.0
                for k in range(27):
                    s += A[k, i] * A[k, j]
                AtA[i, j] = s
        inv = _lu_inverse(AtA)
        P = np.zeros((10, 27))
        for i in range(10):
            for j in range(27):
                s = 0.0
                for k in range(10):
                    s += inv[i, k] * A[j, k]
                P[i, j] = s
        zg = np.array([sum(P[i, k] * S[k] for k in range(27)) for i in range(10)])
        outs = []
        for z in (zc, zg):
            k1 = np.array([[2 * z[0], z[3], z[4]], [z[3], 2 * z[1], z[5]], [z[4], z[5], 2 * z[2]]])
            d = _solve3_closed_form(k1, -z[6:9])
            outs.append((d[0], d[1], d[2] * O.R2D))
        worst = max(worst, abs(outs[0][0] - outs[1][0]), abs(outs[0][1] - outs[1][1]), abs(outs[0][2] - outs[1][2]))
    assert worst < 1e-4, worst


# ---------------- round 2: CPU Baseline A (oracle/cpu_match.cpp) against the Python oracle ----------------
@pytest.mark.parametrize("case", ["test4_src3", "src8", "src9", "src9_subpix", "src4", "cfg1_synth", "cfg2_synth", "cfg3_src6"])
def test_cpp_baseline_equals_python_oracle_results(golden_cases, case):
    """the C++ restatement of match() (reference Release flags incl. -ffast-math, own models of the OpenCV calls) returns the
    Python oracle's accepted set on every golden case, within the north_star tolerances"""
    from oracle.cpu_match import CpuMatcher
    from tests.helpers import get_image
    c = golden_cases[case]
    m = CpuMatcher()
    for k, v in c["params"].items():
        setattr(m, k, v)
    assert m.learn_pattern(get_image(c["tpl"]))
    rows = m.match(get_image(c["src"]))
    want = c["results"]
    assert len(rows) == len(want)
    if len({r["score"] for r in want}) != len(want):          # exact ties: compare as sets by pose
        rows = np.array(sorted(rows.tolist(), key=lambda r: (round(r[2] / 4), round(r[3] / 4))))
        want = sorted(want, key=lambda r: (round(r["cx"] / 4), round(r["cy"] / 4)))
    for r, w in zip(rows, want):
        assert abs(r[0] - w["score"]) <= 1e-4 and abs(r[1] - w["angle"]) <= 0.01
        assert abs(r[2] - w["cx"]) <= 0.05 and abs(r[3] - w["cy"]) <= 0.05
