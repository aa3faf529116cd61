"""ctypes binding of libctd_b200.so (include/ctd_b200.h).  Thin: numpy arrays in/out, every
non-zero return code becomes a Python exception carrying ctd_last_error().  There is no CPU
fallback: if the library is missing or no sm_100 GPU is visible, construction raises."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libctd_b200.so")
MAX_SRC = 3
ABI_VERSION = 2
PREC_FP16_TC, PREC_FP32_SIMT, PREC_FP16_SIMT, PREC_SPLIT_TC = 0, 1, 2, 3


class CtdOp(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_src", C.c_int32), ("src_buf", C.c_int32 * MAX_SRC),
                ("src_coff", C.c_int32 * MAX_SRC), ("src_c", C.c_int32 * MAX_SRC), ("dst_buf", C.c_int32),
                ("dst_coff", C.c_int32), ("cout", C.c_int32), ("cout_pad", C.c_int32), ("ksize", C.c_int32),
                ("stride", C.c_int32), ("act", C.c_int32), ("residual", C.c_int32), ("aux", C.c_int32),
                ("w16_off", C.c_int64), ("w32_off", C.c_int64), ("b_off", C.c_int64), ("p_off", C.c_int64)]


class CtdBufDesc(C.Structure):
    _fields_ = [("channels", C.c_int32), ("down", C.c_int32)]


class CtdConfig(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("device", C.c_int32), ("precision", C.c_int32), ("max_batch", C.c_int32),
                ("max_h", C.c_int32), ("max_w", C.c_int32), ("nc", C.c_int32), ("use_graph", C.c_int32),
                ("conf_thresh", C.c_float), ("nms_thresh", C.c_float), ("db_thresh", C.c_float),
                ("debug_skip_postproc", C.c_int32)]


class CtdDeviceOutputs(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("stream", "mask_u8", "det", "det_count", "bitmap", "labels", "n_labels",
                                          "line_boxes", "line_scores", "line_count", "results_base")] + \
               [("results_bytes", C.c_size_t)]


# numpy mirror of `ctd_block` (include/ctd_b200.h)
BLOCK_DTYPE = np.dtype([("xyxy", np.int32, (4,)), ("language", np.int32), ("vertical", np.int32), ("angle", np.int32),
                        ("merged", np.int32), ("n_lines", np.int32), ("line_off", np.int32), ("n_dist", np.int32),
                        ("dist_off", np.int32), ("font_is_float", np.int32), ("reserved", np.int32),
                        ("font_size", np.float64), ("vec", np.float64, (2,)), ("norm", np.float64),
                        ("weight", np.float64)], align=True)

class CtdResultsLayout(C.Structure):
    _fields_ = [("max_batch", C.c_int32), ("max_h", C.c_int32), ("max_w", C.c_int32), ("reserved", C.c_int32)] + \
               [(k, C.c_size_t) for k in ("total_bytes", "phase_a_bytes", "mask_u8", "det", "det_count", "n_labels",
                                          "line_boxes", "line_scores", "line_count", "mask_refined", "blocks",
                                          "blocks_stride", "blk_records_off", "blk_lines_off", "blk_dist_off")]


MAX_BLOCKS, MAX_BLOCK_DIST = 1300, 8192   # CTD_MAX_BLOCKS / CTD_MAX_BLOCK_DIST

# numpy mirror of `ctd_region` (include/ctd_b200.h) and its flag / status values
REGION_DTYPE = np.dtype([("status", np.int32), ("out_h", np.int32), ("out_w", np.int32), ("w", np.int32),
                         ("h", np.int32), ("reserved", np.int32), ("offset", np.uint64), ("bytes", np.uint64),
                         ("M", np.float64, (9,))], align=True)
REGION_EXPAND, REGION_VERTICAL = 1, 2
REGION_OK, REGION_E_RATIO, REGION_E_HOMOGRAPHY, REGION_E_SIZE = 0, 1, 2, 3

EXPORTS = ["ctd_create", "ctd_destroy", "ctd_last_error", "ctd_forward", "ctd_get_net_outputs", "ctd_get_mask_u8",
           "ctd_get_detections", "ctd_get_db_components", "ctd_last_forward_ms", "ctd_last_launch_count",
           "ctd_debug_read_buffer", "ctd_debug_write_buffer", "ctd_connected_components", "ctd_nms",
           "ctd_timer_start", "ctd_timer_stop", "ctd_profile_forward", "ctd_get_device_outputs",
           "ctd_get_text_lines", "ctd_seg_represent", "ctd_refine_mask", "ctd_submit", "ctd_collect",
           "ctd_results_bytes", "ctd_join", "ctd_forward_resized", "ctd_get_mask_u8_resized",
           "ctd_resize_linear_u8", "ctd_debug_run_ops", "ctd_get_nms_status", "ctd_group_output",
           "ctd_expand_textwindow", "ctd_detect_page", "ctd_results_layout", "ctd_submit_full", "ctd_device_arena",
           "ctd_plan_regions", "ctd_transform_regions"]

_lib = None


class CtdError(RuntimeError):
    pass


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise CtdError("libctd_b200.so is not built (%s); run `python -c 'import __graft_entry__ as g; g.build()'` "
                       "-- there is no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, i32 = C.c_void_p, C.c_int32
    lib.ctd_create.argtypes = [C.POINTER(vp), C.POINTER(CtdConfig), C.POINTER(CtdOp), i32, C.POINTER(CtdBufDesc), i32,
                               vp, C.c_size_t]
    lib.ctd_create.restype = C.c_int
    lib.ctd_destroy.argtypes = [vp]
    lib.ctd_destroy.restype = None
    lib.ctd_last_error.argtypes = [vp]
    lib.ctd_last_error.restype = C.c_char_p
    lib.ctd_forward.argtypes = [vp, vp, i32, i32, i32, i32]
    lib.ctd_get_net_outputs.argtypes = [vp, vp, vp, vp]
    lib.ctd_get_mask_u8.argtypes = [vp, vp]
    lib.ctd_get_detections.argtypes = [vp, vp, vp]
    lib.ctd_get_db_components.argtypes = [vp, vp, vp, vp]
    lib.ctd_last_forward_ms.argtypes = [vp, C.POINTER(C.c_float)]
    lib.ctd_last_launch_count.argtypes = [vp, C.POINTER(i32)]
    lib.ctd_debug_read_buffer.argtypes = [vp, i32, vp, C.c_size_t]
    lib.ctd_debug_write_buffer.argtypes = [vp, i32, vp, i32, i32, i32]
    lib.ctd_connected_components.argtypes = [vp, vp, i32, i32, vp, vp, i32, vp]
    lib.ctd_nms.argtypes = [vp, vp, i32, C.c_float, C.c_float, vp, vp]
    lib.ctd_get_text_lines.argtypes = [vp, vp, vp, vp]
    lib.ctd_seg_represent.argtypes = [vp, vp, i32, i32, C.c_float, vp, vp, vp]
    lib.ctd_refine_mask.argtypes = [vp, vp, vp, i32, i32, vp, i32, i32, vp]
    lib.ctd_timer_start.argtypes = [vp]
    lib.ctd_timer_stop.argtypes = [vp, C.POINTER(C.c_float)]
    lib.ctd_profile_forward.argtypes = [vp, vp, i32, i32, i32, i32, vp, i32]
    lib.ctd_get_device_outputs.argtypes = [vp, C.POINTER(CtdDeviceOutputs)]
    lib.ctd_submit.argtypes = [vp, i32, vp, i32, i32, i32, vp]
    lib.ctd_collect.argtypes = [vp, i32]
    lib.ctd_results_bytes.argtypes = [vp, C.POINTER(C.c_size_t)]
    lib.ctd_join.argtypes = [vp, vp]
    lib.ctd_forward_resized.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32]
    lib.ctd_get_mask_u8_resized.argtypes = [vp, i32, i32, i32, i32, vp]
    lib.ctd_resize_linear_u8.argtypes = [vp, vp, i32, i32, i32, vp, i32, i32]
    lib.ctd_debug_run_ops.argtypes = [vp, vp, i32, i32, i32, i32, i32]
    lib.ctd_get_nms_status.argtypes = [vp, vp, C.POINTER(i32)]
    lib.ctd_group_output.argtypes = [vp, vp, i32, vp, i32, i32, i32, vp, i32, vp, i32, vp, i32, vp, i32, C.POINTER(i32)]
    lib.ctd_expand_textwindow.argtypes = [i32, i32, vp, i32, vp]
    lib.ctd_detect_page.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, vp, i32, vp, i32, vp, i32, C.POINTER(i32)]
    lib.ctd_results_layout.argtypes = [vp, C.POINTER(CtdResultsLayout)]
    lib.ctd_submit_full.argtypes = [vp, i32, vp, i32, i32, i32, i32, i32, vp]
    lib.ctd_device_arena.argtypes = [vp, i32, C.POINTER(vp), C.POINTER(vp)]
    lib.ctd_plan_regions.argtypes = [vp, vp, vp, i32, i32, i32, i32, C.c_double, vp, C.POINTER(C.c_size_t)]
    lib.ctd_transform_regions.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp, vp, i32, C.c_double, vp, vp, i32,
                                          C.c_size_t]
    for name in EXPORTS[3:]:
        getattr(lib, name).restype = C.c_int
    lib.ctd_expand_textwindow.restype = None
    _lib = lib
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _region_args(quads, flags, font_size):
    quads = np.ascontiguousarray(np.asarray(quads, np.float64).reshape(-1, 4, 2))
    flags = np.ascontiguousarray(np.asarray(flags, np.int32).reshape(-1))
    font_size = np.ascontiguousarray(np.asarray(font_size, np.float64).reshape(-1))
    assert len(flags) == len(quads) and len(font_size) == len(quads), (quads.shape, flags.shape, font_size.shape)
    return quads, flags, font_size


def plan_regions(quads, flags, font_size, im_w, im_h, channels, textheight):
    """ctd_plan_regions (host only, no handle): per-line status / crop shape / packed offset of
    `TextBlock.get_transformed_region` -> (REGION_DTYPE records, total bytes)."""
    lib = load_library()
    quads, flags, font_size = _region_args(quads, flags, font_size)
    rec = np.zeros((len(quads),), REGION_DTYPE)
    total = C.c_size_t()
    rc = lib.ctd_plan_regions(_ptr(quads), _ptr(flags), _ptr(font_size), len(quads), int(im_w), int(im_h), int(channels),
                              float(textheight), _ptr(rec), C.byref(total))
    if rc != 0:
        raise CtdError("ctd_plan_regions failed (%d)" % rc)
    return rec, int(total.value)


class Engine:
    """One engine handle = one GPU + one stream + one compiled program."""

    def __init__(self, program, device=0, precision=PREC_FP16_TC, max_batch=1, max_h=1024, max_w=1024, use_graph=False,
                 conf_thresh=0.4, nms_thresh=0.35, db_thresh=0.3, skip_postproc=False):
        self.lib = load_library()
        self.h = C.c_void_p()
        self.program = program
        self.nc = int(getattr(program, "nc", 2))
        ops = (CtdOp * len(program.ops))()
        for o, d in zip(ops, program.ops):
            for k, v in d.items():
                if k in ("src_buf", "src_coff", "src_c"):
                    for i in range(MAX_SRC):
                        getattr(o, k)[i] = int(v[i])
                else:
                    setattr(o, k, int(v))
        bufs = (CtdBufDesc * len(program.bufs))(*[CtdBufDesc(c, d) for c, d in program.bufs])
        cfg = CtdConfig(ABI_VERSION, device, precision, max_batch, max_h, max_w, self.nc, int(use_graph), conf_thresh,
                        nms_thresh, db_thresh, int(skip_postproc))
        blob = (C.c_char * len(program.blob)).from_buffer(program.blob)
        rc = self.lib.ctd_create(C.byref(self.h), C.byref(cfg), ops, len(program.ops), bufs, len(program.bufs),
                                 C.cast(blob, C.c_void_p), len(program.blob))
        if rc != 0:
            raise CtdError("ctd_create failed (%d): %s" % (rc, self.lib.ctd_last_error(None).decode()))
        self.shape = None

    def _ck(self, rc):
        if rc != 0:
            raise CtdError("ctd error %d: %s" % (rc, self.lib.ctd_last_error(self.h).decode()))

    def close(self):
        if getattr(self, "h", None):
            self.lib.ctd_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- forward ------------------------------------------------------------------------
    def forward(self, pages):
        """pages: uint8 [n][h][w][3] BGR (host numpy) -> runs the whole device pipeline."""
        pages = np.ascontiguousarray(pages, dtype=np.uint8)
        if pages.ndim == 3:
            pages = pages[None]
        n, h, w, c = pages.shape
        assert c == 3
        self._ck(self.lib.ctd_forward(self.h, _ptr(pages), n, h, w, 0))
        self.shape = (n, h, w)

    def forward_resized(self, page, unpad_h, unpad_w, net_h, net_w):
        """letterbox on the GPU: page u8 [ih][iw][3] of any size -> cv2-exact INTER_LINEAR resize to
        unpad_h x unpad_w, zero padding to net_h x net_w, forward (n = 1)."""
        page = np.ascontiguousarray(page, dtype=np.uint8)
        ih, iw, c = page.shape
        assert c == 3
        self._ck(self.lib.ctd_forward_resized(self.h, _ptr(page), ih, iw, unpad_h, unpad_w, net_h, net_w))
        self.shape = (1, net_h, net_w)

    def mask_u8_resized(self, crop_h, crop_w, out_h, out_w):
        """`cv2.resize(mask[:crop_h, :crop_w], (out_w, out_h), INTER_LINEAR)` of page 0 (inference.py:164-168)."""
        out = np.empty((out_h, out_w), np.uint8)
        self._ck(self.lib.ctd_get_mask_u8_resized(self.h, crop_h, crop_w, out_h, out_w, _ptr(out)))
        return out

    def resize_linear_u8(self, src, dsize_wh):
        """`cv2.resize(src, dsize_wh, interpolation=cv2.INTER_LINEAR)` for uint8 [H,W] / [H,W,3] (bit-exact)."""
        src = np.ascontiguousarray(src, dtype=np.uint8)
        ch = 1 if src.ndim == 2 else src.shape[2]
        dw, dh = int(dsize_wh[0]), int(dsize_wh[1])
        out = np.empty((dh, dw) if src.ndim == 2 else (dh, dw, ch), np.uint8)
        self._ck(self.lib.ctd_resize_linear_u8(self.h, _ptr(src), src.shape[0], src.shape[1], ch, _ptr(out), dh, dw))
        return out

    def forward_device(self, dev_ptr, n, h, w):
        """pages already resident in HBM (device pointer as int)."""
        self._ck(self.lib.ctd_forward(self.h, C.c_void_p(dev_ptr), n, h, w, 1))
        self.shape = (n, h, w)

    def rows_per_image(self):
        n, h, w = self.shape
        return 3 * ((h // 8) * (w // 8) + (h // 16) * (w // 16) + (h // 32) * (w // 32))

    def net_outputs(self, want_blks=True, want_mask=True, want_lines=True):
        n, h, w = self.shape
        blks = np.empty((n, self.rows_per_image(), 5 + self.nc), np.float32) if want_blks else None
        mask = np.empty((n, 1, h, w), np.float32) if want_mask else None
        lines = np.empty((n, 2, h, w), np.float32) if want_lines else None
        self._ck(self.lib.ctd_get_net_outputs(self.h, _ptr(blks), _ptr(mask), _ptr(lines)))
        return blks, mask, lines

    def mask_u8(self):
        n, h, w = self.shape
        m = np.empty((n, h, w), np.uint8)
        self._ck(self.lib.ctd_get_mask_u8(self.h, _ptr(m)))
        return m

    def detections(self):
        n = self.shape[0]
        det = np.empty((n, 300, 6), np.float32)
        cnt = np.empty((n,), np.int32)
        self._ck(self.lib.ctd_get_detections(self.h, _ptr(det), _ptr(cnt)))
        return [det[i, :cnt[i]].copy() for i in range(n)]

    def nms_status(self, n=1):
        """(candidates per page before the capacity cut, capacity): see ctd_get_nms_status."""
        tot = np.zeros((n,), np.int32)
        cap = C.c_int32()
        self._ck(self.lib.ctd_get_nms_status(self.h, _ptr(tot), C.byref(cap)))
        return tot, cap.value

    def db_components(self, want_bitmap=True, want_labels=True):
        n, h, w = self.shape
        bm = np.empty((n, h, w), np.uint8) if want_bitmap else None
        lab = np.empty((n, h, w), np.int32) if want_labels else None
        nl = np.empty((n,), np.int32)
        self._ck(self.lib.ctd_get_db_components(self.h, _ptr(bm), _ptr(lab), _ptr(nl)))
        return bm, lab, nl

    def text_lines(self):
        """per page (boxes int16 [k,4,2], scores f32 [k]) exactly as SegDetectorRepresenter returns them."""
        n = self.shape[0]
        boxes = np.empty((n, 1000, 4, 2), np.int16)
        scores = np.empty((n, 1000), np.float32)
        cnt = np.empty((n,), np.int32)
        self._ck(self.lib.ctd_get_text_lines(self.h, _ptr(boxes), _ptr(scores), _ptr(cnt)))
        return [boxes[i, :cnt[i]].copy() for i in range(n)], [scores[i, :cnt[i]].copy() for i in range(n)]

    def seg_represent(self, pred, thresh=0.3):
        pred = np.ascontiguousarray(pred, np.float32)
        h, w = pred.shape
        boxes = np.empty((1000, 4, 2), np.int16)
        scores = np.empty((1000,), np.float32)
        cnt = np.zeros((1,), np.int32)
        self._ck(self.lib.ctd_seg_represent(self.h, _ptr(pred), h, w, thresh, _ptr(boxes), _ptr(scores), _ptr(cnt)))
        k = int(cnt[0])
        return boxes[:k].copy(), scores[:k].copy()

    def refine_mask(self, img, mask, windows, refine_mode=0):
        """windows: int32 [k,4] already-expanded xyxy windows (expand_textwindow of every block)."""
        img = np.ascontiguousarray(img, np.uint8)
        mask = np.ascontiguousarray(mask, np.uint8)
        win = np.ascontiguousarray(np.asarray(windows, np.int32).reshape(-1, 4))
        out = np.empty(mask.shape, np.uint8)
        self._ck(self.lib.ctd_refine_mask(self.h, _ptr(img), _ptr(mask), mask.shape[0], mask.shape[1], _ptr(win), len(win),
                                          int(refine_mode), _ptr(out)))
        return out

    def last_forward_ms(self):
        ms = C.c_float()
        self._ck(self.lib.ctd_last_forward_ms(self.h, C.byref(ms)))
        return ms.value

    def last_launch_count(self):
        v = C.c_int32()
        self._ck(self.lib.ctd_last_launch_count(self.h, C.byref(v)))
        return v.value

    def debug_read(self, tensor):
        """tensor: dict(buf, coff, c, down) from the compiler -> float32 [n][h/down][w/down][c]."""
        n, h, w = self.shape
        ch = self.program.bufs[tensor["buf"]][0]
        d = tensor["down"]
        out = np.empty((n, h // d, w // d, ch), np.float32)
        self._ck(self.lib.ctd_debug_read_buffer(self.h, tensor["buf"], _ptr(out), out.size))
        return out[..., tensor["coff"]:tensor["coff"] + tensor["c"]]

    def timer_start(self):
        self._ck(self.lib.ctd_timer_start(self.h))

    def timer_stop(self):
        ms = C.c_float()
        self._ck(self.lib.ctd_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def profile_forward(self, pages=None, dev_ptr=None, shape=None):
        """per-op device milliseconds of one un-graphed forward: (op_ms[n_ops], nms_ms, ccl_ms)."""
        nops = len(self.program.ops)
        out = np.zeros((nops + 2,), np.float32)
        if pages is not None:
            pages = np.ascontiguousarray(pages, dtype=np.uint8)
            n, h, w, _ = pages.shape
            self._ck(self.lib.ctd_profile_forward(self.h, _ptr(pages), n, h, w, 0, _ptr(out), out.size))
        else:
            n, h, w = shape
            self._ck(self.lib.ctd_profile_forward(self.h, C.c_void_p(dev_ptr), n, h, w, 1, _ptr(out), out.size))
        self.shape = (n, h, w)
        return out[:nops], float(out[nops]), float(out[nops + 1])

    # ---- pipelined host path: two batches in flight, copies under compute -----------------------
    def results_bytes(self):
        n = C.c_size_t()
        self._ck(self.lib.ctd_results_bytes(self.h, C.byref(n)))
        return int(n.value)

    def submit(self, slot, pages_ptr, n, h, w, results_ptr):
        """asynchronous forward of HOST pages (raw pointers, ideally pinned) into HOST `results`
        (results_bytes() bytes; unpack with multigpu.unpack_arena)."""
        self._ck(self.lib.ctd_submit(self.h, slot, C.c_void_p(pages_ptr), n, h, w, C.c_void_p(results_ptr)))
        self.shape = (n, h, w)

    def results_layout(self):
        """byte offsets of the result arena (ctd_results_layout): dict of ints."""
        lay = CtdResultsLayout()
        self._ck(self.lib.ctd_results_layout(self.h, C.byref(lay)))
        return {k: int(getattr(lay, k)) for k, _t in CtdResultsLayout._fields_}

    def submit_full(self, slot, pages_ptr, n, h, w, results_ptr, refine_mode=0, pages_on_device=False):
        """asynchronous full pipeline (network + post-processing + group_output + refine_mask) of a batch of
        net-sized pages into HOST `results` (results_layout()['total_bytes'] bytes, pinned): see ctd_submit_full."""
        self._ck(self.lib.ctd_submit_full(self.h, slot, C.c_void_p(pages_ptr), n, h, w, int(bool(pages_on_device)),
                                          int(refine_mode), C.c_void_p(results_ptr)))
        self.shape = (n, h, w)

    def device_arena(self, slot):
        """(device pointer of slot's complete result arena copy, cudaStream_t its last writes were enqueued on)."""
        base, st = C.c_void_p(), C.c_void_p()
        self._ck(self.lib.ctd_device_arena(self.h, slot, C.byref(base), C.byref(st)))
        return base.value, st.value

    def detect_page(self, page, net_h, net_w, refine_mode=0, keep_undetected=False):
        """the whole of TextDetector.__call__ for one page of any size (ctd_detect_page): returns
        (mask u8 [ih,iw], mask_refined u8 [ih,iw], block records, lines i32 [.,8], distances f64)."""
        page = np.ascontiguousarray(page, dtype=np.uint8)
        ih, iw, c = page.shape
        assert c == 3
        mask = np.empty((ih, iw), np.uint8)
        refined = np.empty((ih, iw), np.uint8)
        rec = np.zeros((MAX_BLOCKS,), BLOCK_DTYPE)
        lines = np.zeros((MAX_BLOCKS, 8), np.int32)
        dist = np.zeros((MAX_BLOCK_DIST,), np.float64)
        nb = C.c_int32()
        self._ck(self.lib.ctd_detect_page(self.h, _ptr(page), ih, iw, net_h, net_w, int(refine_mode), int(bool(keep_undetected)),
                                          _ptr(mask), _ptr(refined), _ptr(rec), MAX_BLOCKS, _ptr(lines), MAX_BLOCKS, _ptr(dist),
                                          MAX_BLOCK_DIST, C.byref(nb)))
        self.shape = (1, net_h, net_w)
        return mask, refined, rec[:nb.value], lines, dist

    def transform_regions(self, img, quads, flags, font_size, textheight, out=None, img_dev=None, out_dev=None,
                          out_bytes=None):
        """every line crop of one page in one call (ctd_transform_regions) -> (REGION_DTYPE records, packed u8 output).
        img: u8 [H,W] or [H,W,C] host array, or with img_dev = (device pointer, H, W, C) a page already in HBM.
        out: host u8 array to fill (allocated from the plan when None); with out_dev = device pointer the crops stay on
        the device (out_bytes = its capacity) and the second result is None."""
        quads, flags, font_size = _region_args(quads, flags, font_size)
        if img_dev is None:
            img = np.ascontiguousarray(img, np.uint8)
            ih, iw = img.shape[:2]
            ch = 1 if img.ndim == 2 else img.shape[2]
            src, on_dev = _ptr(img), 0
        else:
            ptr, ih, iw, ch = img_dev
            src, on_dev = C.c_void_p(ptr), 1
        rec = np.zeros((len(quads),), REGION_DTYPE)
        if out_dev is not None:
            dst, cap = C.c_void_p(out_dev), int(out_bytes)
        else:
            if out is None:   # other channel counts are rejected by the call itself (CTD_E_INVALID)
                total = plan_regions(quads, flags, font_size, iw, ih, ch, textheight)[1] if ch in (1, 3) else 0
                out = np.empty((total,), np.uint8)
            dst, cap = _ptr(out), out.nbytes if out_bytes is None else int(out_bytes)
        self._ck(self.lib.ctd_transform_regions(self.h, src, ih, iw, ch, on_dev, _ptr(quads), _ptr(flags), _ptr(font_size),
                                                len(quads), float(textheight), _ptr(rec), dst, int(out_dev is not None),
                                                cap))
        return rec, (None if out_dev is not None else out)

    def collect(self, slot):
        self._ck(self.lib.ctd_collect(self.h, slot))

    def join(self, other):
        """everything enqueued so far on `other`'s stream becomes a dependency of this engine's stream."""
        self._ck(self.lib.ctd_join(self.h, other.h))

    def device_outputs(self):
        o = CtdDeviceOutputs()
        self._ck(self.lib.ctd_get_device_outputs(self.h, C.byref(o)))
        return o

    def debug_write(self, tensor, arr, n, h, w):
        """fill a whole buffer (all its channels) from float32 [n][h/down][w/down][channels]."""
        arr = np.ascontiguousarray(arr, np.float32)
        ch = self.program.bufs[tensor["buf"]][0]
        assert arr.shape == (n, h // tensor["down"], w // tensor["down"], ch), arr.shape
        self._ck(self.lib.ctd_debug_write_buffer(self.h, tensor["buf"], _ptr(arr), n, h, w))

    def debug_run_ops(self, first, last, n, h, w, pages=None):
        """run ops [first, last] only, on the current buffer contents (see ctd_debug_run_ops)."""
        if pages is not None:
            pages = np.ascontiguousarray(pages, dtype=np.uint8)
        self._ck(self.lib.ctd_debug_run_ops(self.h, _ptr(pages), n, h, w, first, last))
        self.shape = (n, h, w)

    # ---- stand-alone array kernels --------------------------------------------------------
    def connected_components(self, img, stats_cap=0):
        img = np.ascontiguousarray(img, np.uint8)
        h, w = img.shape
        labels = np.empty((h, w), np.int32)
        nl = np.zeros((1,), np.int32)
        stats = np.empty((stats_cap, 5), np.int32) if stats_cap else None
        self._ck(self.lib.ctd_connected_components(self.h, _ptr(img), h, w, _ptr(labels), _ptr(stats), stats_cap, _ptr(nl)))
        n = int(nl[0])
        return n, labels, (stats[:n] if stats is not None else None)

    def nms(self, pred, conf_thresh=0.4, iou_thresh=0.35):
        pred = np.ascontiguousarray(pred, np.float32)
        det = np.empty((300, 6), np.float32)
        cnt = np.zeros((1,), np.int32)
        self._ck(self.lib.ctd_nms(self.h, _ptr(pred), pred.shape[0], conf_thresh, iou_thresh, _ptr(det), _ptr(cnt)))
        return det[:int(cnt[0])].copy()
