"""not-gpu: the native line -> block grouping (`ctd_group_output`, csrc/group.cpp, called through
comic-text-detector_b200/textblock.py) AND the oracle's python restatement (oracle/textblock_ref.py) against what the
unmodified reference `utils.textblock.group_output` returned on identical random inputs (tests/golden/group_output.json
and tests/golden/ref_group_output.json.gz, the latter written by `python tests/test_cpu_textblock.py --regen` through
oracle/ref_shim.py).  Integer fields, structure and order must be identical; float fields are compared to 1e-12
relative for the native code (glibc acos/sin vs numpy's SIMD kernels may differ in the last ulp) and exactly for the
python restatement."""
import functools
import gzip
import json
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ctd_b200 import textblock as tb  # noqa: E402
from oracle import ref_shim, textblock_ref  # noqa: E402

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "group_output.json")
REF = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_group_output.json.gz")


def make_case(seed, im_w=1024, im_h=1024):
    rng = np.random.default_rng(seed)
    nb = int(rng.integers(0, 14))
    boxes, cls = [], []
    for _ in range(nb):
        x0, y0 = int(rng.integers(0, im_w - 80)), int(rng.integers(0, im_h - 80))
        w, h = int(rng.integers(30, 320)), int(rng.integers(30, 320))
        boxes.append([x0, y0, min(im_w - 1, x0 + w), min(im_h - 1, y0 + h)])
        cls.append(int(rng.integers(0, 2)))
    blks = (np.array(boxes, np.int32).reshape(-1, 4), np.array(cls, np.int32), np.round(rng.uniform(0.4, 1, nb), 3))
    lines = []
    for _ in range(int(rng.integers(0, 40))):
        vertical = rng.random() < 0.5
        if nb and rng.random() < 0.75:
            b = boxes[int(rng.integers(0, nb))]
            cx, cy = rng.uniform(b[0], b[2]), rng.uniform(b[1], b[3])
        else:
            cx, cy = rng.uniform(40, im_w - 40), rng.uniform(40, im_h - 40)
        lw, lh = (rng.uniform(10, 40), rng.uniform(40, 260)) if vertical else (rng.uniform(40, 260), rng.uniform(10, 40))
        ang = rng.normal(0, 0.08)
        u = np.array([np.cos(ang), np.sin(ang)]) * lw / 2
        v = np.array([-np.sin(ang), np.cos(ang)]) * lh / 2
        c = np.array([cx, cy])
        q = np.array([c - u - v, c + u - v, c + u + v, c - u + v])
        q[:, 0] = np.clip(q[:, 0], 0, im_w - 1)
        q[:, 1] = np.clip(q[:, 1], 0, im_h - 1)
        lines.append(q.astype(np.int32))
    lines = np.array(lines, np.int32).reshape(-1, 4, 2) if lines else []
    mask = (rng.random((im_h // 8, im_w // 8)) < 0.35).astype(np.uint8) * 255
    mask = np.kron(mask, np.ones((8, 8), np.uint8))
    return blks, lines, im_w, im_h, mask


def blk_summary(b):
    d = dict(xyxy=[int(v) for v in b.xyxy], lines=np.array(b.lines).astype(int).tolist(), language=b.language,
             vertical=bool(b.vertical), font_size=float(b.font_size), angle=int(b.angle),
             distance=None if b.distance is None else [float(x) for x in np.atleast_1d(b.distance)],
             vec=None if b.vec is None else [float(x) for x in b.vec], norm=float(b.norm), merged=bool(b.merged),
             weight=float(b.weight))
    return d


def _run(fn, case):
    blks, lines, w, h, mask = case
    blks = (blks[0].copy(), blks[1].copy(), blks[2].copy())
    lines = lines.copy() if len(lines) else []
    return [blk_summary(b) for b in fn(blks, lines, w, h, mask.copy())]


FLOAT_KEYS = ("font_size", "distance", "vec", "norm", "weight")


def assert_same_blocks(got, ref, rel=1e-12):
    """integer fields / structure exactly, float fields to `rel` (NaN == NaN)."""
    assert len(got) == len(ref), (len(got), len(ref))
    for i, (g, r) in enumerate(zip(got, ref)):
        for k in r:
            if k in FLOAT_KEYS:
                a, b = np.atleast_1d(np.array(g[k], np.float64)), np.atleast_1d(np.array(r[k], np.float64))
                assert a.shape == b.shape, (i, k, a.shape, b.shape)
                assert np.allclose(a, b, rtol=rel, atol=0, equal_nan=True), (i, k, g[k], r[k])
            else:
                assert g[k] == r[k], (i, k, g[k], r[k])


def reference_case(seed):
    return make_case(seed) if seed < 48 else make_case(seed, 1536, 1024)     # landscape pages halve the grid width


@functools.lru_cache(maxsize=None)
def reference_blocks():
    """seed -> blk_summary list of the reference's group_output on reference_case(seed), seeds 0..63"""
    with gzip.open(REF, "rt") as f:
        return json.load(f)


@pytest.mark.parametrize("seed", range(24))
def test_python_restatement_equals_reference(seed):
    assert _run(textblock_ref.group_output, make_case(seed)) == reference_blocks()[str(seed)]


@pytest.mark.parametrize("seed", range(64))
def test_native_group_output_equals_reference(seed):
    assert_same_blocks(_run(tb.group_output, reference_case(seed)), reference_blocks()[str(seed)])


def test_native_group_output_golden():
    gold = json.load(open(GOLD))
    for seed, ref in gold.items():
        assert_same_blocks(_run(tb.group_output, make_case(int(seed))), ref)


@pytest.mark.parametrize("seed", range(100, 140))
def test_native_group_output_equals_python_restatement(seed):
    """runs everywhere (also on the GPU box, where /root/reference is absent)"""
    case = make_case(seed) if seed % 3 else make_case(seed, 1400, 904)
    assert_same_blocks(_run(tb.group_output, case), _run(textblock_ref.group_output, case))


def test_group_output_edge_inputs():
    mask = np.zeros((64, 64), np.uint8)
    none = (np.zeros((0, 4), np.int32), np.zeros((0,), np.int32), np.zeros((0,), np.float32))
    assert tb.group_output(none, [], 64, 64, mask) == []
    # one detector box, no lines, no mask under it -> dropped; with mask -> one synthetic line (xywh2xyxypoly)
    one = (np.array([[8, 8, 40, 24]], np.int32), np.array([0], np.int32), np.array([0.9], np.float32))
    assert tb.group_output(one, [], 64, 64, mask) == []
    mask[:] = 255
    out = tb.group_output(one, [], 64, 64, mask)
    ref = textblock_ref.group_output(one, [], 64, 64, mask)
    assert_same_blocks([blk_summary(b) for b in out], [blk_summary(b) for b in ref])
    assert out[0].lines == [[[6, 8], [42, 8], [42, 24], [6, 24]]] or len(out[0].lines) == 1
    # a box hanging off the page: python slice semantics on the mask (negative indices wrap)
    off = (np.array([[-20, -10, 30, 30]], np.int32), np.array([1], np.int32), np.array([0.9], np.float32))
    a = [blk_summary(b) for b in tb.group_output(off, [], 64, 64, mask)]
    b = [blk_summary(b) for b in textblock_ref.group_output(off, [], 64, 64, mask)]
    assert_same_blocks(a, b)


def test_quads_intersect():
    sq = [(0, 0), (4, 0), (4, 3), (0, 3)]
    assert textblock_ref.quads_intersect(sq, [(4, 3), (6, 3), (6, 5), (4, 5)])
    assert not textblock_ref.quads_intersect(sq, [(5, 0), (6, 0), (6, 1), (5, 1)])
    assert textblock_ref.quads_intersect(sq, [(1, 1), (2, 1), (2, 2), (1, 2)])


if __name__ == "__main__":
    if "--regen" in sys.argv:
        ns = ref_shim.load()
        rec = {str(seed): _run(ns.textblock.group_output, reference_case(seed)) for seed in range(64)}
        with open(REF, "wb") as f:
            f.write(gzip.compress(json.dumps(rec, sort_keys=True).encode(), 9, mtime=0))
        print("wrote", REF)
