import hashlib

import numpy as np

import fpm_workloads as synth

# inputs of the IM_Conv_SIMD pin (tests/golden/imconv_ref.json): row lengths around the 16-byte SIMD blocks, and cells of
# bright rows whose float accumulation rounds
IMCONV_ROW_LENGTHS = [1, 7, 15, 16, 17, 54, 762, 1024, 4000]
IMCONV_CELLS = [(762, 521), (1024, 300), (54, 54)]


def imconv_pin_inputs():
    """([(kernel row, source row)], [(template, source) cell]) drawn from one seeded stream, rows first."""
    rng = np.random.default_rng(1)
    rows = [(rng.integers(0, 256, n, dtype=np.uint8), rng.integers(0, 256, n, dtype=np.uint8)) for n in IMCONV_ROW_LENGTHS]
    cells = [(rng.integers(200, 256, (th, tw), dtype=np.uint8), rng.integers(200, 256, (th, tw), dtype=np.uint8))
             for (tw, th) in IMCONV_CELLS]
    return rows, cells


def imconv_pin_digest(rows, cells):
    h = hashlib.sha256()
    for a, b in rows + cells:
        h.update(a.tobytes())
        h.update(b.tobytes())
    return h.hexdigest()


def get_image(name):
    if name == "@cfg1":
        return synth.cfg1_source()
    if name == "@cfg2":
        return synth.cfg2_source()
    return synth.load_fixture(name)


def configure(m, params):
    """Apply an oracle-style params dict to a TemplateMatcher (GPU) or OracleMatcher."""
    from oracle.oracle import OracleMatcher
    if isinstance(m, OracleMatcher):
        m.max_pos, m.score, m.tolerance_angle = 70, 0.7, 0.0
        m.min_reduce_area, m.max_overlap, m.sub_pixel, m.use_simd = 256, 0.0, False, True
        for k, v in params.items():
            setattr(m, k, v)
        return m
    m.setMaxPositions(params.get("max_pos", 70))
    m.setScore(params.get("score", 0.7))
    m.setToleranceAngle(params.get("tolerance_angle", 0.0))
    m.setMinReduceArea(params.get("min_reduce_area", 256))
    m.setMaxOverlap(params.get("max_overlap", 0.0))
    m.setSubPixelEstimation(params.get("sub_pixel", False))
    m.setUseSIMD(params.get("use_simd", True))
    return m


# north_star tolerances
TOL_SCORE = 1e-4
TOL_POS = 0.05
TOL_ANGLE = 0.01


def assert_results_match(got, want, tol_score=TOL_SCORE, tol_pos=TOL_POS, tol_angle=TOL_ANGLE, ordered=True):
    """got: list of SingleTargetMatch (GPU); want: list of dicts (golden) or oracle SingleTargetMatch."""
    def norm(r):
        if isinstance(r, dict):
            return (r["score"], r["angle"], r["cx"], r["cy"], r["lt"], r["rt"], r["rb"], r["lb"])
        if hasattr(r, "dMatchScore"):
            return (r.dMatchScore, r.dMatchedAngle, r.ptCenter[0], r.ptCenter[1], r.ptLT, r.ptRT, r.ptRB, r.ptLB)
        return (r.score, r.angle, r.ptCenter[0], r.ptCenter[1], r.ptLT, r.ptRT, r.ptRB, r.ptLB)
    g = [norm(r) for r in got]
    w = [norm(r) for r in want]
    assert len(g) == len(w), "accepted-target count differs: got %d, want %d" % (len(g), len(w))
    if not ordered:
        # exact score ties: the reference's std::sort order is unspecified -> compare as sets by pose
        key = lambda r: (round(r[2] / 4), round(r[3] / 4))
        g.sort(key=key)
        w.sort(key=key)
    for i, (a, b) in enumerate(zip(g, w)):
        assert abs(a[0] - b[0]) <= tol_score, "target %d score %r vs %r" % (i, a[0], b[0])
        assert abs(a[1] - b[1]) <= tol_angle, "target %d angle %r vs %r" % (i, a[1], b[1])
        assert abs(a[2] - b[2]) <= tol_pos and abs(a[3] - b[3]) <= tol_pos, "target %d centre %r vs %r" % (i, a[2:4], b[2:4])
        for pa, pb in zip(a[4:], b[4:]):
            assert abs(pa[0] - pb[0]) <= tol_pos and abs(pa[1] - pb[1]) <= tol_pos, "target %d corner %r vs %r" % (i, pa, pb)
