"""not-gpu: the annotation writer (comic-text-detector_b200/annotations.py, SURVEY 8f row f2) against the files the
UNMODIFIED reference's own writer code path (`model2annotations`' per-page body, inference.py:33-70, run with the
reference's group_output / TextBlock / xyxy2yolo / get_yololabel_strings / NumpyEncoder / imwrite) wrote for the same
pages: every file byte-identical.  What the reference wrote is stored in tests/golden/ref_annotations.json.gz (text
files verbatim, JSON parsed, images as SHA-1 of the bytes), written by `python tests/test_cpu_annotations.py --regen`
through oracle/ref_shim.py; the format itself is also checked stand-alone."""
import gzip
import hashlib
import json
import os
import os.path as osp
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ctd_b200 import annotations as ann  # noqa: E402
from ctd_b200 import textblock as tb  # noqa: E402
from oracle import ref_shim  # noqa: E402
from test_cpu_textblock import make_case  # noqa: E402

REF = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_annotations.json.gz")
SEEDS = [0, 3, 5, 11, 17]


def _page(seed):
    blks, lines, w, h, mask = make_case(seed)
    img = np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)
    return "page %d.jpg" % seed, img, mask, (blks, lines, w, h, mask)


def _group(fn, case):
    blks, lines, w, h, mask = case
    return fn((blks[0].copy(), blks[1].copy(), blks[2].copy()), lines.copy() if len(lines) else [], w, h, mask.copy())


def _file_record(path):
    """what the comparison keeps of a written file: text files verbatim, JSON parsed, images as SHA-1 of the bytes"""
    data = open(path, "rb").read()
    if path.endswith(".json"):
        return json.loads(data)
    if path.endswith(".txt"):
        return data.decode("utf8")
    return hashlib.sha1(data).hexdigest()


def _reference_page_writer(ns, save_dir, imgname, img, mask_refined, blk_list, save_json):
    """inference.py:33-70 with the reference's own helpers (nothing of ours on this path)."""
    from pathlib import Path
    io_utils = sys.modules["utils.io_utils"]
    ip = ns.imgproc_utils
    im_h, im_w = img.shape[:2]
    imname = imgname.replace(Path(imgname).suffix, '')
    polys, blk_xyxy, blk_dict_list = [], [], []
    for blk in blk_list:
        polys += blk.lines
        blk_xyxy.append(blk.xyxy)
        blk_dict_list.append(blk.to_dict())
    blk_xyxy = ip.xyxy2yolo(blk_xyxy, im_w, im_h)
    yolo_label = ip.get_yololabel_strings([1] * len(blk_xyxy), blk_xyxy) if blk_xyxy is not None else ''
    with open(osp.join(save_dir, imname + '.txt'), 'w', encoding='utf8') as f:
        f.write(yolo_label)
    if len(polys) != 0:
        np.savetxt(osp.join(save_dir, 'line-' + imname + '.txt'), np.array(polys).reshape(-1, 8), fmt='%d')
    if save_json:
        with open(osp.join(save_dir, imname + '.json'), 'w', encoding='utf8') as f:
            f.write(json.dumps(blk_dict_list, ensure_ascii=False, cls=io_utils.NumpyEncoder))
    io_utils.imwrite(osp.join(save_dir, imgname), img)
    io_utils.imwrite(osp.join(save_dir, 'mask-' + imname + '.png'), mask_refined)


@pytest.mark.parametrize("seed", SEEDS)
def test_files_equal_reference_writer(tmp_path, seed):
    with gzip.open(REF, "rt") as f:
        ref = json.load(f)[str(seed)]
    name, img, mask, case = _page(seed)
    ann.write_annotations(str(tmp_path), name, img, mask, _group(tb.group_output, case), save_json=True)
    fa = sorted(os.listdir(tmp_path))
    assert fa == sorted(ref) and len(fa) >= 4
    for f in fa:
        ja, jb = _file_record(str(tmp_path / f)), ref[f]
        if f.endswith(".json"):
            # same blocks, same keys, same values (key ORDER follows each class's attribute order)
            assert len(ja) == len(jb)
            for x, y in zip(ja, jb):
                for k in y:
                    assert k in x, (f, k)
                    if k in ("distance", "vec", "norm", "weight", "font_size"):
                        # float fields of the native group_output: glibc acos/sin vs numpy's SIMD kernels may differ in
                        # the last ulp; the TYPE written (int vs float) must still agree
                        assert type(x[k]) is type(y[k]), (f, k, x[k], y[k])
                        assert np.allclose(np.array(x[k], np.float64), np.array(y[k], np.float64), rtol=1e-12, atol=0,
                                           equal_nan=True), (f, k)
                    else:
                        assert x[k] == y[k], (f, k)
        else:
            assert ja == jb, f


def test_label_and_line_formats(tmp_path):
    blk = tb.TextBlock([10, 20, 110, 220], lines=[[[10, 20], [110, 20], [110, 60], [10, 60]]])
    img = np.zeros((400, 200, 3), np.uint8)
    ann.write_annotations(str(tmp_path), "p.png", img, np.zeros((400, 200), np.uint8), [blk], save_json=True)
    assert (tmp_path / "p.txt").read_text() == "1 0.3 0.3 0.5 0.5"
    assert (tmp_path / "line-p.txt").read_text() == "10 20 110 20 110 60 10 60\n"
    assert json.loads((tmp_path / "p.json").read_text())[0]["xyxy"] == [10, 20, 110, 220]
    assert (tmp_path / "p.png").exists() and (tmp_path / "mask-p.png").exists()
    ann.write_annotations(str(tmp_path), "q.jpg", img, np.zeros((400, 200), np.uint8), [], save_json=False)
    assert (tmp_path / "q.txt").read_text() == "" and not (tmp_path / "line-q.txt").exists()
    assert ann.find_all_imgs(str(tmp_path)) and all(f.endswith(".png") for f in ann.find_all_imgs(str(tmp_path)))


if __name__ == "__main__":
    if "--regen" in sys.argv:
        import tempfile
        ns = ref_shim.load()
        rec = {}
        for seed in SEEDS:
            name, img, mask, case = _page(seed)
            with tempfile.TemporaryDirectory() as d:
                _reference_page_writer(ns, d, name, img, mask, _group(ns.textblock.group_output, case), True)
                rec[str(seed)] = {f: _file_record(os.path.join(d, f)) for f in sorted(os.listdir(d))}
        with open(REF, "wb") as f:
            f.write(gzip.compress(json.dumps(rec, sort_keys=True).encode(), 9, mtime=0))
        print("wrote", REF)
