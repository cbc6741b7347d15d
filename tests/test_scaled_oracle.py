"""The CPU oracle of scale-tolerant matching (tests/scaled_oracle.py): [1, 1] is the reference oracle, the scale schedule's
properties, and known answers on seeded scenes with instances pasted at other sizes."""
import math

import numpy as np
import pytest

from oracle import oracle as O
from tests.helpers import configure, get_image
from tests.scaled_oracle import ScaledOracleMatcher, scale_schedule, scale_step, scaled_scene

# 640 x 480 frame, 96 x 72 template: instances at scales 0.8, 1.0 and 1.25 and angles within +-25 degrees
POSES = [(150.0, 130.0, 12.0, 0.8), (440.0, 150.0, -20.0, 1.0), (300.0, 350.0, 7.0, 1.25)]
PARAMS = dict(max_pos=10, score=0.8, tolerance_angle=25, max_overlap=0.2)


@pytest.mark.parametrize("name", ["src8", "test4_src3"])
def test_unit_range_is_the_oracle(golden_cases, name):
    c = golden_cases[name]
    tpl, src = get_image(c["tpl"]), get_image(c["src"])
    a = configure(O.OracleMatcher(), c["params"])
    b = configure(ScaledOracleMatcher(), c["params"])
    assert a.learn_pattern(tpl) and b.learn_pattern(tpl)
    ra, rb = a.match(src), b.match(src)
    assert ra
    assert [(r.ptLT, r.ptRT, r.ptRB, r.ptLB, r.ptCenter, r.angle, r.score) for r in ra] == \
           [(r.ptLT, r.ptRT, r.ptRB, r.ptLB, r.ptCenter, r.angle, r.score) for r in rb]
    assert all(r.scale == 1.0 for r in rb)


@pytest.mark.parametrize("lo,hi,w,h", [(0.8, 1.25, 24, 18), (0.5, 2.0, 14, 14), (0.9, 1.1, 60, 40), (1.0, 1.0001, 30, 30),
                                       (0.7, 0.7, 20, 10)])
def test_schedule_properties(lo, hi, w, h):
    s = scale_schedule(lo, hi, w, h)
    assert s[0] == lo and s[-1] == hi
    if lo == hi:
        assert s == [lo]
        return
    ds = scale_step(w, h)
    assert len(s) >= 2
    for a, b in zip(s, s[1:]):
        assert a < b and b / a <= 1 + ds + 1e-12
    assert len(s) == math.ceil(math.log(hi / lo) / math.log1p(ds)) + 1


def _found(res, pose, tpl, step_l0, ds_l0):
    """pose's angle is OpenCV's sign (paste_scaled); the matcher reports the opposite sign"""
    cx, cy, a, s = pose
    for r in res:
        if math.hypot(r.ptCenter[0] - cx, r.ptCenter[1] - cy) <= 1.0 and abs(r.angle + a) <= step_l0 and \
           abs(r.scale / s - 1) <= ds_l0:
            return True
    return False


@pytest.fixture(scope="module")
def scene():
    return scaled_scene(640, 480, 96, 72, POSES, seed=21)


def test_range_finds_every_scale(scene):
    tpl, src = scene
    m = configure(ScaledOracleMatcher(), PARAMS)
    m.scale_min, m.scale_max = 0.8, 1.25
    assert m.learn_pattern(tpl)
    res = m.match(src)
    step = math.atan(2.0 / 96) * O.R2D
    assert len(res) == 3, [(r.ptCenter, r.angle, r.scale, r.score) for r in res]
    for p in POSES:
        assert _found(res, p, tpl, step, scale_step(96, 72)), (p, [(r.ptCenter, r.angle, r.scale) for r in res])


def test_unscaled_misses_the_other_sizes(scene):
    tpl, src = scene
    m = configure(ScaledOracleMatcher(), PARAMS)
    assert m.learn_pattern(tpl)
    res = m.match(src)
    step = math.atan(2.0 / 96) * O.R2D
    assert len(res) == 1 and _found(res, POSES[1], tpl, step, scale_step(96, 72))


@pytest.mark.parametrize("k", [0, 2])
def test_fixed_scale_finds_its_instance(scene, k):
    tpl, src = scene
    m = configure(ScaledOracleMatcher(), PARAMS)
    m.scale_min = m.scale_max = POSES[k][3]
    assert m.learn_pattern(tpl)
    res = m.match(src)
    step = math.atan(2.0 / 96) * O.R2D
    assert _found(res, POSES[k], tpl, step, 1e-12)
    for r in res:
        assert r.scale == POSES[k][3]
        w = math.hypot(r.ptRT[0] - r.ptLT[0], r.ptRT[1] - r.ptLT[1])
        assert abs(w - 96 * POSES[k][3]) < 1e-3


def test_refusals():
    m = ScaledOracleMatcher()
    m.scale_min, m.scale_max = 1.2, 1.1
    with pytest.raises(ValueError):
        m.match(np.zeros((10, 10), np.uint8))
    m.scale_min, m.scale_max = 0.4, 1.0
    with pytest.raises(ValueError):
        m.match(np.zeros((10, 10), np.uint8))
