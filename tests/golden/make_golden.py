"""Generates tests/golden/* from the reference's Test Images and the CPU oracle.

Run HERE (the build container, where /root/reference is mounted):
    python tests/golden/make_golden.py
Outputs (committed):
    tests/golden/images/*.png   grayscale fixtures, decoded ONCE with cv2 (JPEG decoders differ)
    tests/golden/cases.json     oracle results (count, score, angle, pose) for every fixture case,
                                template statistics, pyramid checksums, top-layer candidate lists
The GPU box has no /root/reference: tests read only these files.
"""
import hashlib
import json
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle.oracle import OracleMatcher  # noqa: E402
import fpm_workloads as synth  # noqa: E402

REF = "/root/reference/Test Images"
FIXTURES = ["Src3.bmp", "Dst3.bmp", "Src4.bmp", "Dst4.bmp", "Src6.jpg", "Dst6.bmp", "Dst7.bmp", "Src8.bmp", "Dst8.bmp",
            "Src9.bmp", "Dst9.bmp", "Dst10.jpg"]

# name -> (src, tpl, params); params follow README.md:63-71 / BASELINE.json configs
CASES = {
    "test4_src3": ("Src3", "Dst3", dict(max_pos=38, score=0.8, tolerance_angle=0, min_reduce_area=256, max_overlap=0.0)),
    "cfg3_src6": ("Src6", "Dst6", dict(max_pos=15, score=0.8, tolerance_angle=180, min_reduce_area=256, max_overlap=0.0)),
    "src8": ("Src8", "Dst8", dict(max_pos=5, score=0.8, tolerance_angle=180, min_reduce_area=256, max_overlap=0.8)),
    "src9": ("Src9", "Dst9", dict(max_pos=5, score=0.8, tolerance_angle=180, min_reduce_area=256, max_overlap=0.0)),
    "src9_subpix": ("Src9", "Dst9", dict(max_pos=5, score=0.8, tolerance_angle=180, min_reduce_area=256, max_overlap=0.0,
                                         sub_pixel=True)),
    "src4": ("Src4", "Dst4", dict(max_pos=70, score=0.7, tolerance_angle=180, min_reduce_area=64, max_overlap=0.0)),
    "cfg1_synth": ("@cfg1", "Dst7", dict(max_pos=3, score=0.8, tolerance_angle=180, min_reduce_area=256, max_overlap=0.0)),
    "cfg2_synth": ("@cfg2", "Dst10", dict(max_pos=200, score=0.7, tolerance_angle=0, min_reduce_area=256, max_overlap=0.0)),
}


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def get_image(name):
    if name == "@cfg1":
        return synth.cfg1_source()
    if name == "@cfg2":
        return synth.cfg2_source()
    return synth.load_fixture(name)


def run_case(src, tpl, params):
    m = OracleMatcher()
    for k, v in params.items():
        setattr(m, k, v)
    m.trace = {}
    assert m.learn_pattern(tpl)
    res = m.match(src)
    td = m.td
    out = dict(
        params=params,
        src_shape=list(src.shape), tpl_shape=list(tpl.shape),
        src_sha=sha(src), tpl_sha=sha(tpl),
        border_color=td.border_color,
        tpl_levels=[dict(w=int(p.shape[1]), h=int(p.shape[0]), sha=sha(p), mean=td.templ_mean[i], norm=td.templ_norm[i],
                         inv_area=td.inv_area[i], equal1=bool(td.result_equal1[i])) for i, p in enumerate(td.pyramid)],
        src_pyr_sha=[sha(p) for p in m.trace["src_pyr"]],
        n_angles=len(m.trace["angles"]),
        n_candidates=len(m.trace["cands"]),
        candidates=[[c[0][0], c[0][1], c[1], c[2]] for c in m.trace["cands"]],
        results=[dict(score=r.score, angle=r.angle, cx=r.ptCenter[0], cy=r.ptCenter[1], lt=list(r.ptLT), rt=list(r.ptRT),
                      rb=list(r.ptRB), lb=list(r.ptLB)) for r in res],
    )
    return out


OCR_PARAMS = dict(max_pos=70, score=0.85, tolerance_angle=0, min_reduce_area=256, max_overlap=0.0)


def ocr_case():
    """36 glyph templates of Test Images/M12 read on M12_D_Test.jpg (MatchToolDlg.cpp:718-770)."""
    from oracle.oracle import OCR_LETTERS, ocr_read
    os.makedirs(os.path.join(HERE, "images", "M12"), exist_ok=True)
    tpls = {}
    for ch in OCR_LETTERS:
        img = cv2.imread(os.path.join(REF, "M12", ch + ".jpg"), cv2.IMREAD_GRAYSCALE)
        assert img is not None, ch
        cv2.imwrite(os.path.join(HERE, "images", "M12", ch + ".png"), img, [cv2.IMWRITE_PNG_COMPRESSION, 9])
        tpls[ch] = img
    src = cv2.imread(os.path.join(REF, "M12", "M12_D_Test.jpg"), cv2.IMREAD_GRAYSCALE)
    cv2.imwrite(os.path.join(HERE, "images", "M12", "M12_D_Test.png"), src, [cv2.IMWRITE_PNG_COMPRESSION, 9])
    text, per = ocr_read(src, tpls, OCR_PARAMS)
    return dict(params=OCR_PARAMS, src="M12/M12_D_Test", src_sha=sha(src), text=text,
                results={ch: [dict(score=r.score, angle=r.angle, cx=r.ptCenter[0], cy=r.ptCenter[1], lt=list(r.ptLT), rt=list(r.ptRT),
                                   rb=list(r.ptRB), lb=list(r.ptLB)) for r in res] for ch, res in per.items()})


def imconv_golden():
    """tests/golden/imconv_ref.json: the values the reference's IM_Conv_SIMD stands for on the pin's seeded inputs -- the
    exact integer dot product of each row pair, and for each cell the float sum of its row dot products in row order
    (src/TemplateMatcher.cpp:505-508: `*r_matResult = *r_matResult + IM_Conv_SIMD(...)`).  Computed here from that
    definition, independently of the oracle; the pin checks the reference's own build (oracle/_ref) against them
    wherever that build is present."""
    from tests.helpers import imconv_pin_digest, imconv_pin_inputs
    rows, cells = imconv_pin_inputs()
    row_dot = [int((k.astype(np.int64) * c).sum()) for k, c in rows]
    cell = []
    for tpl, src in cells:
        acc = np.float32(0)
        for t, s in zip(tpl, src):
            acc = np.float32(acc + np.float32(int((t.astype(np.int64) * s).sum())))
        cell.append(float(acc))
    out = dict(inputs="tests.helpers.imconv_pin_inputs()", inputs_sha256=imconv_pin_digest(rows, cells),
               row_dot=row_dot, cell=cell)
    with open(os.path.join(HERE, "imconv_ref.json"), "w") as f:
        json.dump(out, f, indent=1)


def main():
    os.makedirs(os.path.join(HERE, "images"), exist_ok=True)
    for f in FIXTURES:
        img = cv2.imread(os.path.join(REF, f), cv2.IMREAD_GRAYSCALE)
        assert img is not None, f
        cv2.imwrite(os.path.join(HERE, "images", os.path.splitext(f)[0] + ".png"), img, [cv2.IMWRITE_PNG_COMPRESSION, 9])
        if f.endswith(".jpg"):                             # the JPEG file images themselves: fixtures of the JPEG ingest path
            import shutil
            os.makedirs(os.path.join(HERE, "jpeg"), exist_ok=True)
            shutil.copyfile(os.path.join(REF, f), os.path.join(HERE, "jpeg", f))
    cases = {}
    for name, (s, t, params) in CASES.items():
        src, tpl = get_image(s), get_image(t)
        cases[name] = run_case(src, tpl, params)
        cases[name]["src"] = s
        cases[name]["tpl"] = t
        print(name, "->", len(cases[name]["results"]), "results,", cases[name]["n_candidates"], "candidates")
    cases["ocr_m12"] = ocr_case()
    print("ocr_m12 ->", repr(cases["ocr_m12"]["text"]))
    with open(os.path.join(HERE, "cases.json"), "w") as f:
        json.dump(cases, f, indent=1)
    imconv_golden()


if __name__ == "__main__":
    if sys.argv[1:] == ["imconv"]:
        imconv_golden()
    else:
        main()
