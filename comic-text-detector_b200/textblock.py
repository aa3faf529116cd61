"""`TextBlock` records and the line -> block grouping of the drop-in detector.

The grouping itself (`group_output`, reference utils/textblock.py:421-508 and its callees) is native code:
`ctd_group_output` in libctd_b200.so (csrc/group.cpp, declared in include/ctd_b200.h).  This module only converts
between the reference's python types -- the `(boxes, cls, conf)` tuple of `postprocess_yolo`, the int32 line quads,
the `TextBlock` objects callers of `TextDetector.__call__` receive (field names of utils/textblock.py:12-85) -- and the
flat C arrays of that call.
"""
import copy
import ctypes as C

import numpy as np

from . import binding

LANG_LIST = ["eng", "ja", "unknown"]
LANGCLS2IDX = {"eng": 0, "ja": 1, "unknown": 2}


class TextBlock(object):
    """Result record with the reference's field names (textblock.py:12-85).  `get_transformed_region` (the OCR crop
    of one line, textblock.py:162-194) runs on the GPU through the most recently created live `TextDetector`; the
    other UI helpers of the reference class (min_rect, colours ...) are not part of the detection path.  Instances
    carry only the reference's attributes: `vars(blk)` feeds to_dict and the annotation writer."""

    def __init__(self, xyxy, lines=None, language="unknown", vertical=False, font_size=-1, distance=None, angle=0,
                 vec=None, norm=-1, merged=False, weight=-1, text=None, translation="", fg_r=0, fg_g=0, fg_b=0,
                 bg_r=0, bg_g=0, bg_b=0, line_spacing=1., font_family="", bold=False, underline=False, italic=False,
                 alignment=-1, alpha=255, rich_text="", _bounding_rect=None, accumulate_color=True,
                 default_stroke_width=0.2, target_lang="", **kwargs):
        self.xyxy = [int(v) for v in xyxy]
        self.lines = [] if lines is None else lines
        self.vertical = vertical
        self.language = language
        self.font_size = font_size
        self.distance = None if distance is None else np.array(distance, np.float64)
        self.angle = angle
        self.vec = None if vec is None else np.array(vec, np.float64)
        self.norm = norm
        self.merged = merged
        self.weight = weight
        self.text = text if text is not None else []
        self.prob = 1
        self.translation = translation
        self.fg_r, self.fg_g, self.fg_b = fg_r, fg_g, fg_b
        self.bg_r, self.bg_g, self.bg_b = bg_r, bg_g, bg_b
        self.font_family = font_family
        self.bold, self.underline, self.italic = bold, underline, italic
        self.alpha = alpha
        self.rich_text = rich_text
        self.line_spacing = line_spacing
        self._alignment = alignment
        self._target_lang = target_lang
        self._bounding_rect = _bounding_rect
        self.default_stroke_width = default_stroke_width
        self.accumulate_color = accumulate_color

    def lines_array(self, dtype=np.float64):
        return np.array(self.lines, dtype=dtype)

    def __len__(self):
        return len(self.lines)

    def __getitem__(self, idx):
        return self.lines[idx]

    def to_dict(self):
        return copy.deepcopy(vars(self))

    def get_transformed_region(self, img, idx, textheight):
        """reference textblock.py:162-194: line `idx` cropped from the page and straightened to `textheight` pixels
        (rotated 90 degrees counter-clockwise for vertical blocks), bit-exact with the reference's cv2 calls.  Runs on the
        GPU of the most recently created live TextDetector (RuntimeError when there is none; there is no CPU path);
        raises ValueError where the reference raises (OverflowError / ValueError / cv2.error)."""
        from .inference import live_detector, _REGION_ERRORS
        det = live_detector()
        if det is None:
            raise RuntimeError("TextBlock.get_transformed_region runs on a TextDetector's GPU engine; create one first")
        self.lines[idx]   # IndexError like the reference
        crops, status = det._crop_lines(img, [(self, idx)], textheight)
        if crops[0] is None:
            raise ValueError("line %d cannot be cropped: %s" % (idx, _REGION_ERRORS.get(status[0], status[0])))
        return crops[0]


def blocks_from_records(blocks, lines, dist):
    """ctd_block records (+ the flat line / distance arrays they index) -> list of TextBlock.  The record fields are
    converted column-wise (one numpy call per field): indexing a structured array row by row costs ~1 us per field and
    was a third of the single-page latency of `TextDetector.__call__` at 256 blocks."""
    n = len(blocks)
    if n == 0:
        return []
    lo, nl = blocks["line_off"].tolist(), blocks["n_lines"].tolist()
    d0, nd = blocks["dist_off"].tolist(), blocks["n_dist"].tolist()
    fs, fif = blocks["font_size"].tolist(), blocks["font_is_float"].tolist()
    xy, lang = blocks["xyxy"].tolist(), blocks["language"].tolist()
    vert, ang, mrg = blocks["vertical"].tolist(), blocks["angle"].tolist(), blocks["merged"].tolist()
    vec = np.ascontiguousarray(blocks["vec"], np.float64)
    norm = np.ascontiguousarray(blocks["norm"], np.float64)
    weight = np.ascontiguousarray(blocks["weight"], np.float64)
    ll = np.asarray(lines).reshape(-1, 4, 2).tolist()     # every line quad as python ints, once
    dist = np.asarray(dist, np.float64)
    tpl = _template()
    out = []
    for i in range(n):
        # same attributes, in the same order, as TextBlock.__init__ would set (to_dict / the json writer depend on it)
        d = tpl.copy()
        d["xyxy"] = xy[i]
        d["lines"] = ll[lo[i]:lo[i] + nl[i]]
        d["vertical"] = bool(vert[i])
        d["language"] = LANG_LIST[lang[i]]
        d["font_size"] = float(fs[i]) if fif[i] else int(fs[i])
        d["distance"] = dist[d0[i]:d0[i] + nd[i]].copy()
        d["angle"] = int(ang[i])
        d["vec"] = vec[i].copy()
        d["norm"] = norm[i]
        d["merged"] = bool(mrg[i])
        d["weight"] = weight[i]
        d["text"] = []
        blk = TextBlock.__new__(TextBlock)
        blk.__dict__ = d
        out.append(blk)
    return out


_TEMPLATE = None


def _template():
    """attribute dict of a default TextBlock (insertion order = the order __init__ assigns them)"""
    global _TEMPLATE
    if _TEMPLATE is None:
        _TEMPLATE = dict(vars(TextBlock([0, 0, 0, 0], distance=[0.0], vec=[0.0, 0.0])))
    return _TEMPLATE


def group_output(blks, lines, im_w, im_h, mask=None, sort_blklist=True):
    """`group_output` (textblock.py:421-508) through the native library.  blks = (boxes int32 [n,4], cls int32 [n],
    conf f32 [n]); lines = int32 [m,4,2] (or []); mask = u8 page mask [im_h, im_w] or None."""
    lib = binding.load_library()
    boxes = np.ascontiguousarray(np.asarray(blks[0], np.int32).reshape(-1, 4))
    cls = np.ascontiguousarray(np.asarray(blks[1], np.int32).reshape(-1))
    ln = np.ascontiguousarray(np.asarray(lines, np.int32).reshape(-1, 4, 2))
    nb, nl = len(boxes), len(ln)
    if mask is not None:
        mask = np.ascontiguousarray(mask, np.uint8)
        assert mask.shape == (im_h, im_w), (mask.shape, im_h, im_w)
    cap_b, cap_l = nb + nl + 1, nb + nl + 1
    cap_d = cap_l * max(nl, 1) + 1
    rec = np.zeros((cap_b,), binding.BLOCK_DTYPE)
    lout = np.zeros((cap_l, 8), np.int32)
    dout = np.zeros((cap_d,), np.float64)
    n = C.c_int32()
    rc = lib.ctd_group_output(binding._ptr(boxes), binding._ptr(cls), nb, binding._ptr(ln), nl, int(im_w), int(im_h),
                              binding._ptr(mask), int(bool(sort_blklist)), binding._ptr(rec), cap_b, binding._ptr(lout),
                              cap_l, binding._ptr(dout), cap_d, C.byref(n))
    if rc != 0:
        raise binding.CtdError("ctd_group_output failed (%d)" % rc)
    return blocks_from_records(rec[:n.value], lout, dout)


def overlap_area(a, b):
    """`union_area` of the reference (imgproc_utils.py:13-20): the INTERSECTION area, -1 when disjoint."""
    x1, y1 = max(a[0], b[0]), max(a[1], b[1])
    x2, y2 = min(a[2], b[2]), min(a[3], b[3])
    if y2 < y1 or x2 < x1:
        return -1
    return (y2 - y1) * (x2 - x1)
