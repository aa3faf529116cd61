"""Shared helpers for the parity tests."""
import contextlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import ctd_b200  # noqa: E402
from ctd_b200 import compiler as cc  # noqa: E402
from ctd_b200.binding import PREC_FP16_TC, PREC_FP32_SIMT, PREC_FP16_SIMT, PREC_SPLIT_TC  # noqa: E402

_CKPT_CACHE = {}

REFERENCE_THREADS = 8   # torch CPU threads the stored reference outputs (tests/golden/ref_*) were computed with


@contextlib.contextmanager
def reference_threads():
    """torch's CPU kernels split their sums by thread count and each split rounds differently, so a float result (the
    BN statistics of a synthetic checkpoint, a network map) is reproduced bit for bit only with the same count."""
    old = torch.get_num_threads()
    torch.set_num_threads(REFERENCE_THREADS)
    try:
        yield
    finally:
        torch.set_num_threads(old)


def get_checkpoint(seed=0, smooth=True):
    from oracle import synth
    key = (seed, smooth)
    if key not in _CKPT_CACHE:
        _CKPT_CACHE[key] = synth.make_checkpoint(seed, smooth=smooth)
    return _CKPT_CACHE[key]


def h16(a):
    """round to fp16 and back (what the fp16 engine stores)."""
    return np.asarray(a, np.float32).astype(np.float16).astype(np.float32)


def page_to_net_input(pages):
    """u8 [n][h][w][3] BGR -> f32 (n,3,h,w) BGR /255: what preprocess_img feeds the torch backend
    for net-sized pages (inference.py:72-83)."""
    return torch.from_numpy(np.ascontiguousarray(pages.transpose(0, 3, 1, 2)).astype(np.float32) / 255)


class SingleOp:
    """Builds a one-op program around Program.conv/deconv4 with writable source buffers."""

    def __init__(self, src_channels, down=1, extra_channels=0):
        self.P = cc.Program()
        self.P.nc = 2
        self.srcs = []
        for c in src_channels:
            # source tensors sit at a channel offset inside wider buffers to exercise slicing
            b = self.P.newbuf(c + extra_channels, down)
            self.srcs.append(self.P.tensor(b, extra_channels, c))

    def run(self, out_tensor, inputs, n, h, w, precision, dst_init=None):
        eng = ctd_b200.Engine(self.P, precision=precision, max_batch=n, max_h=h, max_w=w, skip_postproc=True)
        try:
            for t, arr in zip(self.srcs, inputs):
                ch = self.P.bufs[t["buf"]][0]
                full = np.zeros(arr.shape[:3] + (ch,), np.float32)
                full[..., t["coff"]:t["coff"] + t["c"]] = arr
                eng.debug_write(t, full, n, h, w)
            if dst_init is not None:
                eng.debug_write(out_tensor, dst_init, n, h, w)
            eng.forward(np.zeros((n, h, w, 3), np.uint8))
            return eng.debug_read(out_tensor)
        finally:
            eng.close()
