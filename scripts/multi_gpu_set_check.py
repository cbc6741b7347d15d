"""Multi-GPU check of template sets in the angle-sharded latency mode, launched with torchrun (one rank per GPU, NCCL):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29534 scripts/multi_gpu_set_check.py
Every rank must return exactly what one GPU returns for the frame: fpm_match_set_sharded == matchSet and
fpm_match_set_sharded_merged == matchSetMerged, for host and device-resident frames, on two sets: the M12 glyphs (several
groups, one angle) and four 256x256 templates at +-180 degrees on a 4096x4096 frame.  A call adds three collectives with a host
frame (sliced upload + two allgathers) and two with a device frame (none at one rank)."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
from fastest_image_pattern_matching_b200 import TemplateMatcher  # noqa: E402
from fastest_image_pattern_matching_b200 import dist as D  # noqa: E402
import fpm_workloads as synth  # noqa: E402
from oracle import oracle as O  # noqa: E402


def _rows(lst):
    return [(r.dMatchScore, r.dMatchedAngle) + tuple(r.ptCenter) + tuple(r.ptLT) + tuple(r.ptRT) + tuple(r.ptRB) + tuple(r.ptLB)
            for r in lst]


def _workloads():
    glyphs = [synth.load_fixture("M12/" + ch) for ch in O.OCR_LETTERS]
    m12 = (glyphs, synth.load_fixture("M12/M12_D_Test"), dict(max_pos=70, score=0.7, tol=0.0))
    tpls = [synth.synth_template(256, 4 + k) for k in range(4)]
    f = synth.background(4096, 4096, 11, 3.0)
    for t, (cx, cy, a) in zip(tpls, [(1000, 1000, 30.0), (3000, 1000, -100.0), (1000, 3000, 150.0), (3000, 3000, -20.0)]):
        synth.paste_rotated(f, t, float(cx), float(cy), a, fast=True)
    return [("m12", m12), ("rot4", (tpls, f, dict(max_pos=4, score=0.8, tol=180.0)))]


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    for name, (tpls, src, p) in _workloads():
        m = TemplateMatcher(local, result_capacity=512)
        m.setMaxPositions(p["max_pos"]); m.setScore(p["score"]); m.setToleranceAngle(p["tol"]); m.setMinReduceArea(256)
        m.learnPatternSet(tpls)
        want = [_rows(x) for x in m.matchSet(src)]
        want_m = [(t,) + _rows([r])[0] for t, r in m.matchSetMerged(src, 0.3)]
        D.init_sharded(m, dist)
        d = torch.from_numpy(np.ascontiguousarray(src)).to(dev)
        dev_kw = dict(ptr=d.data_ptr(), shape=src.shape, stride=src.shape[1], on_device=True)
        for on_dev in (False, True):
            kw = dev_kw if on_dev else dict(sourceImage=src)
            c0 = m.collectiveCount()
            got = [_rows(x) for x in m.matchSetSharded(**kw)]
            assert got == want, "rank %d %s: fpm_match_set_sharded != matchSet (device frame %s)" % (rank, name, on_dev)
            want_c = 0 if world == 1 else (2 if on_dev else 3)                  # one rank: nothing to exchange
            assert m.collectiveCount() - c0 == want_c, (rank, name, on_dev, m.collectiveCount() - c0)
            got_m = [(t,) + _rows([r])[0] for t, r in m.matchSetShardedMerged(max_overlap=0.3, **kw)]
            assert got_m == want_m, "rank %d %s: fpm_match_set_sharded_merged != matchSetMerged (device frame %s)" % (rank, name, on_dev)
        if rank == 0:
            print("multi_gpu_set_check %s ok: world %d, %d per-template hits, %d merged" % (name, world, sum(map(len, want)), len(want_m)))
        m.commDestroy()
        m.close()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
