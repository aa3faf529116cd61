"""not-gpu: the OCR line crop `TextBlock.get_transformed_region(img, idx, textheight)` (reference utils/textblock.py:
162-194).  tests/golden/ref_transformed_regions.npz holds what the UNMODIFIED reference returned (crop bytes) or raised
(exception type) on the seeded cases of `cases()`, written by `python tests/test_cpu_regions.py --regen` through
oracle/ref_shim.py.  Here: the oracle (oracle/regions_ref.py) equals it byte for byte, the native planning call
(`ctd_plan_regions`, host only) gives the same shapes / statuses, and the oracle's numpy restatements of
cv2.findHomography (4 points) and of the fixed-point cv2.warpPerspective are pinned against the installed cv2."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ctd_b200 import binding  # noqa: E402
from ctd_b200.textblock import TextBlock  # noqa: E402
from oracle import ref_shim, regions_ref  # noqa: E402

REF = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_transformed_regions.npz")
LANGS = ["eng", "ja", "unknown"]


def make_page(seed, h, w, channels, gradient=True):
    """gradients + flat rectangles: structure at every scale.  gradient=False (the stored reference cases): a flat
    background with rectangles and thin strokes, whose crops still blend neighbouring values along every edge but
    compress well enough to keep the stored file small"""
    rng = np.random.default_rng(seed)
    img = np.empty((h, w, 3), np.uint8)
    if gradient:
        yy, xx = np.mgrid[0:h, 0:w]
        for c in range(3):
            a, b = rng.uniform(-1, 1, 2)
            img[..., c] = ((xx * a + yy * b) % 256).astype(np.uint8)
    else:
        img[:] = rng.integers(0, 256, 3)
    for _ in range(12):
        x0, y0 = int(rng.integers(0, w)), int(rng.integers(0, h))
        img[y0:y0 + int(rng.integers(4, 60)), x0:x0 + int(rng.integers(4, 90))] = rng.integers(0, 256, 3)
    if not gradient:
        for _ in range(8):
            x0, y0 = int(rng.integers(0, w)), int(rng.integers(0, h))
            if rng.random() < 0.5:
                img[y0:y0 + int(rng.integers(1, 4)), x0:x0 + int(rng.integers(20, 120))] = rng.integers(0, 256, 3)
            else:
                img[y0:y0 + int(rng.integers(20, 120)), x0:x0 + int(rng.integers(1, 4))] = rng.integers(0, 256, 3)
    return img[..., 0].copy() if channels == 1 else img


def case_page(case):
    """the page of a stored reference case"""
    seed, h, w, ch = case[:4]
    return make_page(seed, h, w, ch, gradient=False)


def text_quad(rng, cx, cy, length, thick, vertical, angle, persp, integer):
    lw, lh = (thick, length) if vertical else (length, thick)
    u = np.array([np.cos(angle), np.sin(angle)]) * lw / 2
    v = np.array([-np.sin(angle), np.cos(angle)]) * lh / 2
    c = np.array([cx, cy])
    q = np.array([c - u - v, c + u - v, c + u + v, c - u + v]) + rng.uniform(-persp, persp, (4, 2))
    return np.round(q).astype(int).tolist() if integer else q.tolist()


def cases():
    """-> list of (page seed, h, w, channels, block kwargs, textheight); ~100 cases, deterministic"""
    out = []
    rng = np.random.default_rng(2024)
    ths = [32, 48, 64, 40.5]
    for k in range(84):
        h, w = int(rng.integers(120, 360)), int(rng.integers(120, 480))
        ch = 1 if k % 4 == 3 else 3
        vertical = bool(k % 2)
        lang = LANGS[(k // 2) % 3]
        font = int(rng.integers(8, 40)) if k % 3 else float(rng.uniform(8, 40))
        lines = []
        for _ in range(int(rng.integers(1, 3))):
            if k % 5 == 0:     # touching / crossing a page edge: exercises the clip of expanded quads
                edge = int(rng.integers(0, 4))
                cx = [0, w, rng.uniform(0, w), rng.uniform(0, w)][edge] + rng.uniform(-10, 10)
                cy = [rng.uniform(0, h), rng.uniform(0, h), 0, h][edge] + rng.uniform(-10, 10)
            else:
                cx, cy = rng.uniform(20, w - 20), rng.uniform(20, h - 20)
            length = rng.uniform(20, 160) if k % 7 else rng.uniform(200, 300)   # long lines: crops > 1024 / 16 wide
            thick = rng.uniform(10, 40)
            lines.append(text_quad(rng, cx, cy, length, thick, vertical, rng.normal(0, 0.15), rng.uniform(0, 3),
                                   integer=k % 6 != 5))
        out.append((1000 + k, h, w, ch, dict(lines=lines, language=lang, vertical=vertical, font_size=font),
                    ths[k % 4] if k % 11 else 13))     # textheight 13: crops shorter than 16 rows
    # degenerate lines (the reference raises, or returns a page-sized array for an empty dsize)
    sq = [[40, 30], [140, 30], [140, 60], [40, 60]]
    flat = [[40, 50], [140, 50], [140, 50], [40, 50]]        # no height: ratio 0
    thin = [[80, 20], [80, 20], [80, 120], [80, 120]]        # no width: ratio inf
    dot = [[60, 60]] * 4                                     # ratio nan
    tall = [[50, 10], [51, 10], [51, 90], [50, 90]]          # ratio 80: w = round(32 / 80) = 0 -> page-sized crop
    off = [[300, 300], [340, 300], [340, 320], [300, 320]]   # outside the 96x160 page: clipped onto the corner
    deg = [(sq, "ja", False, 12, 1), (sq, "ja", True, 12, 1),       # h == 1 / w == 1: findHomography -> None
           (sq, "eng", False, 12, 0.5), (sq, "unknown", True, 12, 0.7),   # h == 0 / w == 0: page-sized
           (tall, "ja", False, 12, 32), (tall, "ja", True, 12, 2),
           (flat, "ja", False, 12, 48), (flat, "ja", True, 12, 48), (thin, "ja", False, 12, 48),
           (thin, "ja", True, 12, 48), (dot, "ja", False, 12, 48), (dot, "eng", True, 12, 48),
           (off, "eng", False, 9, 48), (off, "ja", False, 9, 48), (sq, "ja", False, 12, 2), (sq, "ja", True, 12.5, 2)]
    for j, (q, lang, vert, font, th) in enumerate(deg):
        out.append((2000 + j, 96, 160, 3 if j % 2 else 1, dict(lines=[q], language=lang, vertical=vert, font_size=font),
                    th))
    return out


def run_case(fn, case, cls=TextBlock):
    """fn(blk, img, idx, textheight) over every line of the case, blk a `cls` -> crop arrays / exception type names"""
    kw, th = case[4], case[5]
    img = case_page(case)
    res = []
    for i in range(len(kw["lines"])):
        blk = cls([0, 0, 1, 1], **kw)
        try:
            res.append(fn(blk, img, i, th))
        except Exception as e:  # the reference raises OverflowError / ValueError / cv2.error
            res.append(type(e).__name__)
    return res


def _oracle(blk, img, idx, th):
    return regions_ref.get_transformed_region(blk, img, idx, th)


def load_golden():
    """per case, per line: the crop array or the name of the exception the reference raised.  Stored as one packed
    byte array (all crops back to back, which compresses far better than one entry per crop) plus per-line records:
    case, shape (h, w, channels; channels 0 for a 2-D crop) and exception name ('' for a crop)."""
    z = np.load(REF)
    data, case, shape, exc = z["data"], z["case"], z["shape"], z["exc"]
    out, off = [], 0
    for c, (h, w, ch), e in zip(case.tolist(), shape.tolist(), exc.tolist()):
        while len(out) <= c:
            out.append([])
        if e:
            out[c].append(str(e))
            continue
        n = h * w * max(ch, 1)
        crop = data[off:off + n]
        out[c].append(crop.reshape(h, w) if ch == 0 else crop.reshape(h, w, ch))
        off += n
    return out


GOLD = None


def golden():
    global GOLD
    if GOLD is None:
        GOLD = load_golden()
    return GOLD


def test_golden_covers_the_cases():
    g, cs = golden(), cases()
    assert len(g) == len(cs) >= 100
    assert [len(x) for x in g] == [len(c[4]["lines"]) for c in cs]
    flat = [v for x in g for v in x]
    raised = [v for v in flat if isinstance(v, str)]
    assert {"OverflowError", "ValueError", "error"} <= set(raised), set(raised)
    crops = [v for v in flat if not isinstance(v, str)]
    assert any(v.shape[:2] == (96, 160) for v in crops)             # empty dsize: the page's size
    assert any(v.shape[:2] == (160, 96) for v in crops)             # ... rotated for a vertical line
    assert any(v.ndim == 2 for v in crops) and any(v.ndim == 3 for v in crops)
    assert any(v.shape[1] > 64 for v in crops) and any(v.shape[0] < 16 for v in crops)


@pytest.mark.parametrize("k", range(100))
def test_oracle_equals_reference(k):
    cs = cases()
    if k >= len(cs):
        pytest.skip("fewer cases")
    got, ref = run_case(_oracle, cs[k]), golden()[k]
    for g, r in zip(got, ref):
        if isinstance(r, str):
            assert g == r
        else:
            assert not isinstance(g, str), g
            assert g.shape == r.shape and g.dtype == r.dtype and np.array_equal(g, r)


def plan_case(case):
    seed, h, w, ch, kw, th = case
    expand = regions_ref.expands(kw["language"], kw["vertical"])
    flags = [(binding.REGION_EXPAND if expand else 0) | (binding.REGION_VERTICAL if kw["vertical"] else 0)] * len(kw["lines"])
    return binding.plan_regions(np.array(kw["lines"], np.float64), flags, [kw["font_size"]] * len(kw["lines"]), w, h, ch, th)


def test_plan_equals_reference():
    for case, ref in zip(cases(), golden()):
        rec, total = plan_case(case)
        off = 0
        for r, g in zip(rec, ref):
            if isinstance(g, str):
                assert r["status"] != 0 and r["bytes"] == 0, (case[0], g, r)
            else:
                assert r["status"] == 0, (case[0], r)
                assert (int(r["out_h"]), int(r["out_w"])) == g.shape[:2] and int(r["bytes"]) == g.size
            assert int(r["offset"]) == off
            off += int(r["bytes"])
        assert total == off


def test_plan_statuses_name_the_reference_exception():
    for case, ref in zip(cases(), golden()):
        rec, _ = plan_case(case)
        for r, g in zip(rec, ref):
            if isinstance(g, str):
                want = binding.REGION_E_HOMOGRAPHY if g == "error" else binding.REGION_E_RATIO
                assert int(r["status"]) == want, (case[0], g, r)


def test_plan_rejects_bad_arguments():
    lib = binding.load_library()
    total = binding.C.c_size_t()
    q = np.zeros((1, 4, 2))
    f = np.zeros((1,), np.int32)
    fs = np.zeros((1,))
    rec = np.zeros((1,), binding.REGION_DTYPE)
    for ch in (0, 2, 4):
        assert lib.ctd_plan_regions(binding._ptr(q), binding._ptr(f), binding._ptr(fs), 1, 10, 10, ch, 32.0,
                                    binding._ptr(rec), binding.C.byref(total)) == -1
    assert binding.plan_regions(np.zeros((0, 4, 2)), [], [], 10, 10, 3, 32)[1] == 0


def random_text_quads(seed, n):
    """text-line-like quads (rotated rectangles with mild perspective, integer corners as the detector emits them)
    on pages of random size, with random crop sizes"""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        ih, iw = int(rng.integers(64, 400)), int(rng.integers(64, 400))
        vertical = rng.random() < 0.5
        q = text_quad(rng, rng.uniform(-10, iw + 10), rng.uniform(-10, ih + 10), rng.uniform(16, 300),
                      rng.uniform(6, 48), vertical, rng.normal(0, 0.2), rng.uniform(0, 2), integer=rng.random() < 0.8)
        w, h = int(rng.integers(2, 400)), int(rng.integers(2, 70))
        out.append((ih, iw, 1 if rng.random() < 0.3 else 3, np.array(q, np.float64), w, h))
    return out


def test_oracle_warp_equals_cv2():
    """the numpy fixed-point warpPerspective against cv2.warpPerspective on 600 random quads / crop sizes"""
    cv2 = pytest.importorskip("cv2")
    n_px = 0
    for i, (ih, iw, ch, q, w, h) in enumerate(random_text_quads(7, 600)):
        img = make_page(i, ih, iw, ch)
        M, _ = cv2.findHomography(q, regions_ref.dst_points(w, h), cv2.RANSAC, 5.0)
        if M is None:
            continue
        ref = cv2.warpPerspective(img, M, (w, h))
        got = regions_ref.warp_perspective_u8(img, M, (w, h))
        assert got.shape == ref.shape and np.array_equal(got, ref), (i, int((got != ref).sum()))
        n_px += ref.size
    assert n_px > 3_000_000


def test_oracle_homography_equals_cv2():
    """the scalar restatement of findHomography's 4-point kernel against cv2 on 500 random text-line quads: the same
    arithmetic in the same order, so the same bits"""
    cv2 = pytest.importorskip("cv2")
    worst, exact = 0.0, 0
    for ih, iw, ch, q, w, h in random_text_quads(11, 500):
        dst = regions_ref.dst_points(w, h)
        M, _ = cv2.findHomography(q, dst, cv2.RANSAC, 5.0)
        H = regions_ref.homography_4pt(q, dst)
        assert (M is None) == (H is None)
        if M is not None:
            worst = max(worst, float(np.linalg.norm(H - M) / np.linalg.norm(M)))
            exact += int(np.array_equal(H, M))
    assert worst < 1e-12, worst
    assert exact == 500, exact


def test_oracle_homography_degenerate_quads_equal_cv2():
    """three corners on one line (a quad clipped onto a page edge): H[2][2] is ~0 and cv2 returns H unscaled"""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(3)
    n_unscaled = 0
    for _ in range(300):
        q = np.array([[254.7, 0], [409.2, 0], [414.2, 0], [259.7, 27.25]]) + rng.normal(0, 1, (4, 2)) * [1, 0]
        q[2, 1] = 10 ** rng.uniform(-16, 0)
        dst = regions_ref.dst_points(int(rng.integers(3, 900)), int(rng.integers(3, 70)))
        M, _ = cv2.findHomography(q, dst, cv2.RANSAC, 5.0)
        assert np.array_equal(regions_ref.homography_4pt(q, dst), M)
        n_unscaled += abs(M[2, 2] - 1) > 1e-6
    assert 50 < n_unscaled < 250, n_unscaled


if __name__ == "__main__":
    if "--regen" in sys.argv:
        ns = ref_shim.load()

        def _ref(blk, img, idx, th):
            return blk.get_transformed_region(img, idx, th)
        data, case_ids, shapes, excs = [], [], [], []
        for c, case in enumerate(cases()):
            for v in run_case(_ref, case, ns.textblock.TextBlock):
                case_ids.append(c)
                if isinstance(v, str):
                    shapes.append((0, 0, 0))
                    excs.append(v)
                else:
                    assert v.dtype == np.uint8
                    shapes.append((v.shape[0], v.shape[1], v.shape[2] if v.ndim == 3 else 0))
                    excs.append("")
                    data.append(v.reshape(-1))
        np.savez_compressed(REF, data=np.concatenate(data), case=np.array(case_ids, np.int32),
                            shape=np.array(shapes, np.int32), exc=np.array(excs))
        print("wrote", REF, len(case_ids), "lines")
