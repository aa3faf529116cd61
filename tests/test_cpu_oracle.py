"""not-gpu: pin the oracle against what the UNMODIFIED reference computed on the same inputs: the committed golden
vectors under tests/golden/ (net_*_256.npz and nms_ref.npz from oracle/make_golden.py, ref_*.npz from
`python tests/test_cpu_oracle.py --regen`; both import the reference through oracle/ref_shim.py)."""
import os

import numpy as np
import pytest
import sys
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from oracle import geom_ref, postproc_ref, ref_shim, synth
from oracle.net_ref import RefNet
from util import page_to_net_input, reference_threads

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
REF_NET = os.path.join(GOLD, "ref_net_rough_128x192.npz")
REF_SEG = os.path.join(GOLD, "ref_seg_represent.npz")


def _net_case():
    """rough checkpoint (every tap random) on one 128x192 page"""
    ck = synth.make_checkpoint(0, smooth=False, bn_calibrate=128)
    return ck, page_to_net_input(np.stack([synth.structured_page(3, 128, 192)]))


def test_net_ref_is_bit_identical_to_reference():
    """RefNet == the reference's TextDetBase forward (stored), bit for bit"""
    g = np.load(REF_NET)
    with reference_threads():
        ck, x = _net_case()
        b, m, l = RefNet(ck)(x)
    assert torch.equal(b, torch.from_numpy(g["blks"])) and torch.equal(m, torch.from_numpy(g["mask"])) and \
        torch.equal(l, torch.from_numpy(g["lines"]))


def test_nms_restatement_equals_reference():
    """nms_ref.npz holds the reference's non_max_suppression output for its `pred`"""
    g = np.load(os.path.join(GOLD, "nms_ref.npz"))
    pred = torch.from_numpy(g["pred"])[None]
    got = postproc_ref.non_max_suppression(pred, 0.4, 0.35)[0]
    assert torch.equal(torch.from_numpy(g["det"]), got)


@pytest.mark.parametrize("name", ["net_smooth_256.npz", "net_rough_256.npz"])
def test_oracle_reproduces_reference_goldens(name):
    g = np.load(os.path.join(GOLD, name))
    ck = synth.make_checkpoint(int(g["ckpt_seed"]), smooth=bool(g["smooth"]))
    pages = np.stack([synth.structured_page(1000, 256, 256), synth.noise_page(1001, 256, 256)])
    blks, mask, lines = RefNet(ck)(page_to_net_input(pages))
    # the checkpoint is regenerated here (BN statistics re-estimated on this CPU), so allow fp32 noise
    assert float(np.abs(mask[:, :, ::4, ::4].numpy() - g["mask_sub"]).max()) < 1e-4
    assert float(np.abs(lines[:, :, ::4, ::4].numpy() - g["lines_sub"]).max()) < 1e-4
    gb = g["blks_sub"]
    assert float((np.abs(blks[:, ::17].numpy() - gb) / (np.abs(gb) + 1)).max()) < 1e-4


def test_nms_golden():
    g = np.load(os.path.join(GOLD, "nms_ref.npz"))
    got = postproc_ref.non_max_suppression(torch.from_numpy(g["pred"])[None], 0.4, 0.35)[0].numpy()
    assert np.array_equal(got, g["det"])


def test_clipper_offset_restatement_basic():
    # axis-aligned 10x4 rectangle grown by 1.5: every offset vertex lies within delta (+rounding) of the
    # original outline and the bounding box grows by round(delta) on each side
    pts = geom_ref.clipper_offset_closed_polygon([(0, 0), (10, 0), (10, 4), (0, 4)], 1.5)
    a = np.array(pts)
    assert a[:, 0].min() == -2 and a[:, 0].max() == 12 and a[:, 1].min() == -2 and a[:, 1].max() == 6
    # float input is truncated toward zero like pyclipper's cInt conversion
    assert geom_ref.to_cint_path([(1.9, -1.9)]) == [(1, -1)]
    assert geom_ref.clipper_offset_closed_polygon([(0, 0), (0, 0), (1, 1)], 1.0) == []


def test_geos_restatements():
    sq = [(0, 0), (4, 0), (4, 3), (0, 3)]
    assert geom_ref.geos_ring_area(sq) == 12.0 and geom_ref.geos_ring_length(sq) == 14.0
    assert geom_ref.polygons_intersect(sq, [(4, 3), (6, 3), (6, 5), (4, 5)])       # touching corner counts
    assert not geom_ref.polygons_intersect(sq, [(5, 0), (6, 0), (6, 1), (5, 1)])
    assert geom_ref.polygons_intersect(sq, [(1, 1), (2, 1), (2, 2), (1, 2)])       # containment


def test_seg_represent_restatement_equals_reference_class():
    """oracle/postproc_ref.seg_represent == the reference's SegDetectorRepresenter (stored; pyclipper/shapely were
    shimmed by oracle/geom_ref.py when it ran, hence 'parity unpinned' for those two calls only)."""
    import stress_maps
    g = np.load(REF_SEG)
    assert sorted(g.files) == sorted(k + "_" + name for name in stress_maps.CASES for k in ("boxes", "scores"))
    for name, f in stress_maps.CASES.items():
        ob, os_ = postproc_ref.seg_represent(f(), 0.3)
        assert np.array_equal(g["boxes_" + name], ob) and np.array_equal(g["scores_" + name], os_), name


def regen():
    """Runs the unmodified reference (oracle/ref_shim.py) and writes the ref_*.npz vectors the tests above read."""
    import tempfile
    import stress_maps
    ns = ref_shim.load()
    with reference_threads(), tempfile.TemporaryDirectory() as d:
        ck, x = _net_case()
        f = os.path.join(d, "ck.pt")
        torch.save(ck, f)
        net = ns.basemodel.TextDetBase(f, device="cpu", act="leaky")
        with torch.no_grad():
            rb, rm, rl = net(x)
    np.savez_compressed(REF_NET, blks=rb.numpy(), mask=rm.numpy(), lines=rl.numpy())
    rep = ns.db_utils.SegDetectorRepresenter(thresh=0.3)
    seg = {}
    for name, fn in stress_maps.CASES.items():
        b, s = rep(None, torch.from_numpy(fn())[None, None])
        seg["boxes_" + name], seg["scores_" + name] = np.asarray(b[0]), np.asarray(s[0])
    np.savez_compressed(REF_SEG, **seg)
    print("wrote", REF_NET, REF_SEG)


if __name__ == "__main__":
    if "--regen" in sys.argv:
        regen()
