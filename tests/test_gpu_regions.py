"""-m gpu: OCR line crops on the GPU (`ctd_transform_regions`, csrc/regions.cu) through `TextDetector.get_transformed_regions`
and `TextBlock.get_transformed_region`, against the stored outputs of the unmodified reference
(tests/golden/ref_transformed_regions.npz, see tests/test_cpu_regions.py), against live cv2.findHomography /
cv2.warpPerspective and against the oracle (oracle/regions_ref.py).  Crops must be byte-identical; M within 1e-12
(relative, Frobenius) of cv2's."""
import numpy as np
import pytest

import ctd_b200
from ctd_b200 import binding, inference
from oracle import regions_ref, synth
from test_cpu_regions import case_page, cases, golden, make_page, random_text_quads
from util import get_checkpoint

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def det():
    d = ctd_b200.TextDetector(get_checkpoint(0, True), input_size=512, act="leaky")
    yield d
    d.close()


def _assert_same(got, ref):
    if isinstance(ref, str):
        assert got is None, ref
    else:
        assert got is not None and got.dtype == np.uint8 and got.shape == ref.shape and np.array_equal(got, ref)


def test_golden_cases(det):
    """every stored reference case: the batched call and the per-line method"""
    from ctd_b200.textblock import TextBlock
    for case, ref in zip(cases(), golden()):
        kw, th = case[4], case[5]
        img = case_page(case)
        blk = TextBlock([0, 0, 1, 1], **kw)
        out = det.get_transformed_regions(img, [blk], th)
        assert len(out) == 1 and len(out[0]) == len(ref)
        for i, (g, r) in enumerate(zip(out[0], ref)):
            _assert_same(g, r)
            if isinstance(r, str):
                with pytest.raises(ValueError):
                    blk.get_transformed_region(img, i, th)
            else:
                assert np.array_equal(blk.get_transformed_region(img, i, th), r)


def _random_pages(n_pages, lines_per_page, seed):
    """pages of random size and layout with random text-line quads, flags and textheights"""
    rng = np.random.default_rng(seed)
    quads = random_text_quads(seed, n_pages * lines_per_page)
    for p in range(n_pages):
        ih, iw = int(rng.integers(200, 900)), int(rng.integers(200, 900))
        ch = 1 if p % 2 else 3
        img = make_page(seed * 1000 + p, ih, iw, ch)
        q = np.array([x[3] for x in quads[p * lines_per_page:(p + 1) * lines_per_page]])
        flags = rng.integers(0, 4, len(q)).astype(np.int32)
        font = np.where(rng.random(len(q)) < 0.5, rng.integers(8, 40, len(q)), rng.uniform(8, 40, len(q)))
        th = [24, 32, 48, 64, 40.5][p % 5]
        yield img, q, flags, font, th


def test_live_cv2_random_quads(det):
    """>= 1000 random quads on 1- and 3-channel pages: M against cv2.findHomography, crops against cv2.warpPerspective
    with cv2's own M and against the oracle"""
    import cv2
    n_lines, worst = 0, 0.0
    for img, q, flags, font, th in _random_pages(44, 25, 5):
        ih, iw = img.shape[:2]
        rec, buf = det.net.transform_regions(img, q, flags, font, th)
        for i, r in enumerate(rec):
            vertical = bool(flags[i] & binding.REGION_VERTICAL)
            try:
                src, w, h = regions_ref.line_geometry(q[i], bool(flags[i] & binding.REGION_EXPAND), vertical, font[i],
                                                      iw, ih, th)
                M = cv2.findHomography(src, regions_ref.dst_points(w, h), cv2.RANSAC, 5.0)[0]
            except (OverflowError, ValueError):
                M = None
            if M is None:
                assert r["status"] != 0
                continue
            assert r["status"] == 0 and (int(r["w"]), int(r["h"])) == (w, h)
            worst = max(worst, float(np.linalg.norm(r["M"].reshape(3, 3) - M) / np.linalg.norm(M)))
            want = cv2.warpPerspective(img, M, (w, h))
            if vertical:
                want = cv2.rotate(want, cv2.ROTATE_90_COUNTERCLOCKWISE)
            got = buf[int(r["offset"]):int(r["offset"]) + int(r["bytes"])].reshape(want.shape)
            assert np.array_equal(got, want), (i, int((got != want).sum()))
            oracle = regions_ref.warp_perspective_u8(img, r["M"].reshape(3, 3), (w, h))
            assert np.array_equal(got, np.rot90(oracle) if vertical else oracle)
            n_lines += 1
    assert n_lines >= 1000, n_lines
    assert worst <= 1e-12, worst


@pytest.fixture(scope="module")
def detected(det):
    """two synthetic pages through the detector: one net-sized, one that is letterboxed"""
    out = []
    for seed, (h, w) in ((1000, (512, 512)), (1003, (700, 430))):
        page = synth.structured_page(seed, h, w)
        _m, _r, blks = det(page.copy())
        out.append((page, blks))
    return out


def test_detector_output_equals_oracle(det, detected):
    n = 0
    for page, blks in detected:
        assert sum(len(b.lines) for b in blks) > 3
        got = det.get_transformed_regions(page, blks, 48)
        ref = regions_ref.transformed_regions(page, blks, 48)
        assert [len(x) for x in got] == [len(b.lines) for b in blks]
        for g_blk, r_blk in zip(got, ref):
            for g, r in zip(g_blk, r_blk):
                _assert_same(g, "raised" if r is None else r)
                n += 1
        for blk in blks[:4]:      # the per-line method, on the same engine
            for i in range(len(blk.lines)):
                try:
                    r = regions_ref.get_transformed_region(blk, page, i, 48)
                except Exception:
                    with pytest.raises(ValueError):
                        blk.get_transformed_region(page, i, 48)
                    continue
                assert np.array_equal(blk.get_transformed_region(page, i, 48), r)
    assert n > 10


def test_device_resident_page_and_output(det, detected):
    import torch
    page, blks = detected[0]
    items = [(b, i) for b in blks for i in range(len(b.lines))]
    quads = np.array([np.asarray(b.lines[i], np.float64) for b, i in items])
    flags = np.array([(binding.REGION_EXPAND if regions_ref.expands(b.language, b.vertical) else 0)
                      | (binding.REGION_VERTICAL if b.vertical else 0) for b, _ in items], np.int32)
    font = np.array([b.font_size for b, _ in items], np.float64)
    rec_h, host = det.net.transform_regions(page, quads, flags, font, 48)
    dev_page = torch.from_numpy(page).cuda()
    rec_d, out = det.net.transform_regions(None, quads, flags, font, 48, img_dev=(dev_page.data_ptr(), *page.shape))
    assert np.array_equal(out, host) and np.array_equal(rec_d, rec_h)
    dev_out = torch.zeros(len(host) + 16, dtype=torch.uint8, device="cuda")
    rec_dd, none = det.net.transform_regions(None, quads, flags, font, 48, img_dev=(dev_page.data_ptr(), *page.shape),
                                             out_dev=dev_out.data_ptr(), out_bytes=dev_out.numel())
    assert none is None and np.array_equal(rec_dd, rec_h)
    assert np.array_equal(dev_out[:len(host)].cpu().numpy(), host)


def test_edges(det, detected):
    from ctd_b200.textblock import TextBlock
    page, blks = detected[0]
    assert det.get_transformed_regions(page, [], 48) == []
    empty = TextBlock([0, 0, 10, 10])
    assert det.get_transformed_regions(page, [empty, blks[0], empty], 48)[0] == []
    # vars() of the blocks is unchanged: to_dict and the json writer see the reference's attributes only
    before = [(list(vars(b)), repr(b.to_dict())) for b in blks]
    det.get_transformed_regions(page, blks, 32)
    blks[0].get_transformed_region(page, 0, 32)
    assert [(list(vars(b)), repr(b.to_dict())) for b in blks] == before
    q = np.array([blks[0].lines[0]], np.float64)
    with pytest.raises(binding.CtdError, match="need"):                      # CTD_E_CAPACITY
        det.net.transform_regions(page, q, [0], [12.0], 48, out=np.empty((10,), np.uint8))
    with pytest.raises(binding.CtdError, match="channels"):                  # CTD_E_INVALID
        det.net.transform_regions(np.zeros((64, 64, 2), np.uint8), q, [0], [12.0], 48)
    with pytest.raises(ValueError):
        det.get_transformed_regions(page.astype(np.float32), blks, 48)


def test_no_live_detector_raises(det, detected):
    page, blks = detected[0]
    saved = inference._LIVE_DETECTOR
    try:
        other = ctd_b200.TextDetector(get_checkpoint(0, True), input_size=256, act="leaky")
        assert np.array_equal(blks[0].get_transformed_region(page, 0, 48), det.get_transformed_regions(page, blks[:1], 48)[0][0])
        other.close()
        with pytest.raises(RuntimeError):
            blks[0].get_transformed_region(page, 0, 48)
        del other
        with pytest.raises(RuntimeError):
            blks[0].get_transformed_region(page, 0, 48)
    finally:
        inference._LIVE_DETECTOR = saved
