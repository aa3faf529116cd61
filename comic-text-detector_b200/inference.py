"""Drop-in `TextDetector` over the B200 engine.

Same constructor and call signature as the reference's `inference.TextDetector`
(inference.py:116-178): `TextDetector(model_path, input_size=1024, device=..., half=False, nms_thresh=0.35,
conf_thresh=0.4, mask_thresh=0.3, act='leaky')` and
`detector(img, refine_mode=REFINEMASK_INPAINT, keep_undetected_mask=False) -> (mask, mask_refined, blk_list)`.

Everything runs in libctd_b200.so: network, NMS, mask u8, DB binarize, connected components, contour boxes + scores,
refine_mask on the GPU; ratio scaling, `group_output` and the window expansion in host C++ (csrc/group.cpp,
csrc/pipeline.cu).  This module is the reference-shaped Python surface over `ctd_detect_page`.
"""
import weakref
from pathlib import Path
from typing import List

import numpy as np

from . import compiler
from .binding import Engine, PREC_FP16_TC, PREC_FP32_SIMT, REGION_EXPAND, REGION_OK, REGION_VERTICAL
from .textblock import TextBlock, blocks_from_records, group_output, overlap_area  # noqa: F401

REFINEMASK_INPAINT = 0
REFINEMASK_ANNOTATION = 1


_LIVE_DETECTOR = None   # weak reference to the most recently created TextDetector (TextBlock.get_transformed_region)


def live_detector():
    """the most recently created TextDetector if it is still alive and open, else None"""
    det = _LIVE_DETECTOR() if _LIVE_DETECTOR is not None else None
    return det if det is not None and det.net.h else None


# what the reference raises for a line it cannot crop, by ctd_region status (textblock.py:175-191)
_REGION_ERRORS = {1: "the line's aspect ratio is 0, inf or nan (round() raises OverflowError / ValueError)",
                  2: "cv2.findHomography returns None for this line (w or h is 1, or the quad has no extent along an "
                     "axis), so cv2.warpPerspective raises cv2.error",
                  3: "the crop would exceed 2 GiB"}


def letterbox_geometry(shape_hw, new_shape=(1024, 1024)):
    """The size arithmetic of `letterbox(im, new_shape, auto=False)` (utils/imgproc_utils.py:86-117): aspect-preserving
    scale r, resized size (w, h) = round(size * r) (Python's round), bottom/right padding (dw, dh)."""
    r = min(new_shape[0] / shape_hw[0], new_shape[1] / shape_hw[1])
    new_unpad = int(round(shape_hw[1] * r)), int(round(shape_hw[0] * r))
    dw, dh = new_shape[1] - new_unpad[0], new_shape[0] - new_unpad[1]
    return r, new_unpad, int(dw), int(dh)


def letterbox(im, new_shape=(1024, 1024)):
    """Host restatement of the reference's `letterbox` (kept for tests / tools; the detector itself resizes on the
    GPU through `Engine.forward_resized`, bit-exact with cv2.INTER_LINEAR)."""
    r, new_unpad, dw, dh = letterbox_geometry(im.shape[:2], new_shape)
    if im.shape[:2][::-1] != new_unpad:
        import cv2
        im = cv2.resize(im, new_unpad, interpolation=cv2.INTER_LINEAR)
    if dw or dh:
        padded = np.zeros((new_shape[0], new_shape[1], 3), np.uint8)
        padded[:im.shape[0], :im.shape[1]] = im
        im = padded
    return im, (r, r), (dw, dh)


def expand_textwindow(img_size, xyxy, expand_r=8):
    """utils/imgproc_utils.py:151-161"""
    im_h, im_w = img_size[:2]
    x1, y1, x2, y2 = xyxy
    w, h = x2 - x1, y2 - y1
    pad = int(round((max(h, w) * 0.25 + min(h, w) * 0.75) / expand_r))
    return [max(0, x1 - pad), max(0, y1 - pad), min(im_w - 1, x2 + pad), min(im_h - 1, y2 + pad)]


class TextDetector:
    lang_list = ['eng', 'ja', 'unknown']
    langcls2idx = {'eng': 0, 'ja': 1, 'unknown': 2}

    def __init__(self, model_path, input_size=1024, device='cuda', half=False, nms_thresh=0.35, conf_thresh=0.4,
                 mask_thresh=0.3, act='leaky', precision=None, device_index=0):
        if isinstance(model_path, (str, Path)):
            import torch
            ckpt = torch.load(str(model_path), map_location='cpu')  # reference basemodel.py:212
        else:
            ckpt = model_path  # already a checkpoint dict
        if isinstance(input_size, int):
            input_size = (input_size, input_size)
        self.input_size = input_size
        self.device = device
        self.half = half
        self.conf_thresh = conf_thresh
        self.nms_thresh = nms_thresh
        self.backend = 'b200'
        if precision is None:
            precision = PREC_FP16_TC
        # fused Bottleneck ops exist on the fp16 tensor-core engine only (bit-identical to the two-op form)
        self.program = compiler.compile_checkpoint(ckpt, head_act=act, fuse=compiler.fuse_default(precision == PREC_FP16_TC))
        # DB threshold is hard-coded 0.3 in the reference (inference.py:139 ignores mask_thresh)
        self.net = Engine(self.program, device=device_index, precision=precision, max_batch=1, max_h=input_size[0],
                          max_w=input_size[1], conf_thresh=conf_thresh, nms_thresh=nms_thresh, db_thresh=0.3)
        global _LIVE_DETECTOR
        _LIVE_DETECTOR = weakref.ref(self)

    def close(self):
        self.net.close()

    def __call__(self, img, refine_mode=REFINEMASK_INPAINT, keep_undetected_mask=False):
        """reference inference.py:141-178.  One native call (`ctd_detect_page`): letterbox (cv2-exact INTER_LINEAR) +
        network + NMS + mask u8 + DB boxes on the GPU, postprocess_yolo casts / box_thresh / group_output on the host
        in C++, refine_mask (and refine_undetected_mask) on the GPU with the page and its mask resident in HBM; this
        method only turns the block records into `TextBlock` objects."""
        img = np.ascontiguousarray(img)
        mask, mask_refined, rec, lines, dist = self.net.detect_page(img, self.input_size[0], self.input_size[1], refine_mode,
                                                                    keep_undetected_mask)
        return mask, mask_refined, blocks_from_records(rec, lines, dist)

    def get_transformed_regions(self, img, blk_list, textheight):
        """`TextBlock.get_transformed_region(img, idx, textheight)` (reference utils/textblock.py:162-194) for every line
        of every block, in one native call (ctd_transform_regions: homographies and warps on the GPU, bit-exact with
        cv2.findHomography + cv2.warpPerspective).  Returns one list per block with one uint8 crop per line in the
        reference's shape (h x w, or w x h rotated for vertical lines; 2-D for a 2-D or single-channel page), and None
        for a line on which the reference raises.  The crops are views of one packed buffer."""
        items = [(blk, i) for blk in blk_list for i in range(len(blk.lines))]
        crops, _status = self._crop_lines(img, items, textheight)
        out, k = [], 0
        for blk in blk_list:
            out.append(crops[k:k + len(blk.lines)])
            k += len(blk.lines)
        return out

    def _crop_lines(self, img, items, textheight):
        """(blk, line index) pairs -> (list of crops or None, ctd_region statuses)"""
        img = np.ascontiguousarray(img)
        if img.dtype != np.uint8 or img.ndim not in (2, 3):
            raise ValueError("expected a uint8 HxW or HxWxC page, got %s %s" % (img.dtype, img.shape))
        ch = 1 if img.ndim == 2 else img.shape[2]
        if not items:
            return [], []
        quads = np.array([np.asarray(blk.lines[i], np.float64).reshape(4, 2) for blk, i in items])
        flags = np.array([(REGION_EXPAND if blk.language == "eng" or (blk.language == "unknown" and not blk.vertical)
                           else 0) | (REGION_VERTICAL if blk.vertical else 0) for blk, _i in items], np.int32)
        font = np.array([blk.font_size for blk, _i in items], np.float64)
        rec, buf = self.net.transform_regions(img, quads, flags, font, float(textheight))
        crops = []
        for r in rec.tolist():
            status, out_h, out_w, off, nbytes = r[0], r[1], r[2], r[6], r[7]
            if status != REGION_OK:
                crops.append(None)
                continue
            crop = buf[off:off + nbytes]
            crops.append(crop.reshape(out_h, out_w) if ch == 1 else crop.reshape(out_h, out_w, ch))
        return crops, rec["status"].tolist()
