/*
 * ctd_b200.h -- C ABI of libctd_b200.so, the B200 (sm_100a) engine behind the reference's
 * inference path  page -> (block boxes, text-line map, segmentation mask).
 *
 * The reference is pure Python and has no FFI; the seam this library replaces is the
 * backend object built in `inference.TextDetector.__init__` (reference inference.py:124-130:
 * `self.net = TextDetBase(...)` / `TextDetBaseDNN(...)`, a callable
 * `net(img_in) -> (blks, mask, lines_map)`, basemodel.py:240-244) plus the array-level
 * post-processing calls made from `TextDetector.__call__` (inference.py:141-178).
 * Each entry point cites the reference interface it stands in for.  Plain C types only:
 * no torch, no C++ types, nothing thrown across the boundary.  Every function returns 0 on
 * success or a negative CTD_E_* code; `ctd_last_error()` gives the message.
 *
 * Threading: a handle is bound to one CUDA device and one internal stream and is NOT
 * thread-safe; independent handles (one per GPU / per process) are independent.
 */
#ifndef CTD_B200_H_
#define CTD_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CTD_ABI_VERSION 2
#if defined(__GNUC__)
#define CTD_API __attribute__((visibility("default")))
#else
#define CTD_API
#endif

/* ---- error codes ---------------------------------------------------------------------- */
#define CTD_OK 0
#define CTD_E_INVALID (-1)   /* bad argument / malformed program                            */
#define CTD_E_CUDA (-2)      /* CUDA runtime/driver error (message has the CUDA string)     */
#define CTD_E_NO_DEVICE (-3) /* no sm_100 GPU visible: the engine has NO CPU fallback       */
#define CTD_E_SHAPE (-4)     /* page size not a multiple of 64 (basemodel.py:62-78 stride)  */
#define CTD_E_CAPACITY (-5)  /* batch larger than the reserved workspace                    */

/* ---- network program ------------------------------------------------------------------
 * The Python host (comic-text-detector_b200/compiler.py) plays the role of the reference's
 * `parse_model` + `load_state_dict` + `fuse` (models/yolov5/yolo.py:208-259,285-311;
 * utils/yolov5_utils.py:23-43; basemodel.py:211-220): it walks the checkpoint's cfg, folds
 * every BatchNorm and emits a flat list of ops over numbered NHWC activation buffers plus one
 * weight blob.  The engine owns no architecture knowledge beyond these op kinds.           */

enum ctd_op_kind {
  CTD_OP_STEM = 0,      /* 6x6 s2 p2 conv on the u8 BGR page (/255 fused), common.py:30-49 cfg L0 */
  CTD_OP_CONV = 1,      /* k in {1,3}, stride in {1,2}, pad k/2; K-concatenated sources     */
  CTD_OP_DECONV4 = 2,   /* ConvTranspose2d 4x4 s2 p1 (basemodel.py:26) as 4 sub-pixel phases */
  CTD_OP_AVGPOOL2 = 3,  /* AvgPool2d(2,2)                (basemodel.py:38)                  */
  CTD_OP_SPPF_POOL = 4, /* 3 chained MaxPool2d(5,1,2)    (common.py:188-196)                */
  CTD_OP_UPSAMPLE2 = 5, /* nn.Upsample(x2, nearest)      (cfg layers 11,15)                 */
  CTD_OP_DETECT = 6,    /* Detect 1x1 conv + sigmoid + box decode (yolo.py:23-44)           */
  CTD_OP_SEG_TAIL = 7,  /* ConvT4x4s2 64->1 + sigmoid    (basemodel.py:57-60)               */
  CTD_OP_DB_TAIL = 8,   /* ConvT2x2s2+BN+ReLU -> ConvT2x2s2 -> sigmoid, both branches
                           (basemodel.py:99-103,138-142)                                    */
  CTD_OP_S2D = 9,       /* u8 BGR page -> /255 -> 2x2 space-to-depth, 12(+4 zero) channels at 1/2 resolution:
                           turns the 6x6 s2 p2 stem conv into a 3x3 s1 p1 conv for the tensor cores       */
  CTD_OP_BNECK = 10     /* fused Bottleneck (common.py:94-104): dst = [src +] act(conv3x3(act(conv1x1(src)))), c -> c -> c
                           channels (c = cout in {32, 64}), src and dst in DIFFERENT buffers; w16_off / w32_off: W1 [c][c]
                           followed by W2 [c][9c] (K = (ky, kx, ci)); b_off: bias1[c] | bias2[c]; residual = the `+ src`.
                           CTD_PREC_FP16_TC only (the compiler emits it on request, compiler.py fuse=True)              */
};

enum ctd_act { CTD_ACT_NONE = 0, CTD_ACT_SILU = 1, CTD_ACT_LEAKY = 2, CTD_ACT_RELU = 3, CTD_ACT_SIGMOID = 4 };

#define CTD_MAX_SRC 3

typedef struct ctd_op {
  int32_t kind;                  /* enum ctd_op_kind                                        */
  int32_t n_src;                 /* 1..CTD_MAX_SRC K-concatenated inputs (torch.cat on dim 1) */
  int32_t src_buf[CTD_MAX_SRC];  /* activation buffer ids                                   */
  int32_t src_coff[CTD_MAX_SRC]; /* first channel read in that buffer                       */
  int32_t src_c[CTD_MAX_SRC];    /* channels read                                           */
  int32_t dst_buf;               /* activation buffer id (-1 for ops writing engine outputs) */
  int32_t dst_coff;              /* first channel written                                   */
  int32_t cout;                  /* true output channels                                    */
  int32_t cout_pad;              /* rows in the packed weight matrix (multiple of 16)       */
  int32_t ksize;                 /* 1, 3 (conv), 4 (deconv), 6 (stem)                       */
  int32_t stride;                /* 1 or 2                                                  */
  int32_t act;                   /* enum ctd_act                                            */
  int32_t residual;              /* 1: dst = act(conv)+dst in place (Bottleneck.add, common.py:104) */
  int32_t aux;                   /* DETECT: pyramid level (0,1,2)                           */
  int64_t w16_off;               /* blob offset: fp16 weights [phase][cout_pad][taps*Cin] K-major */
  int64_t w32_off;               /* blob offset: fp32 weights, same layout                  */
  int64_t b_off;                 /* blob offset: fp32 bias[cout_pad] (BN folded)            */
  int64_t p_off;                 /* blob offset: extra fp32 params (DETECT anchors, tails)  */
} ctd_op;

typedef struct ctd_bufdesc {
  int32_t channels; /* total channels of the NHWC buffer                                   */
  int32_t down;     /* spatial size = page size / down                                     */
} ctd_bufdesc;

enum ctd_precision {
  CTD_PREC_FP16_TC = 0,   /* fp16 storage, tcgen05 implicit GEMM, fp32 accumulate (default) */
  CTD_PREC_FP32_SIMT = 1, /* fp32 storage + CUDA-core fp32 kernels ("vs reference fp32" config) */
  CTD_PREC_FP16_SIMT = 2, /* fp16 storage + CUDA-core kernels (bisecting aid)               */
  CTD_PREC_SPLIT_TC = 3   /* fp32 storage; tcgen05 with every operand split into fp16 hi + lo planes
                             (hi*hi + lo*hi + hi*lo, fp32 accumulate: ~22 significant bits) -- the
                             tensor-core path that meets the 1e-3 "vs reference fp32" tolerance  */
};

typedef struct ctd_config {
  int32_t abi_version; /* CTD_ABI_VERSION                                                  */
  int32_t device;      /* CUDA device ordinal                                              */
  int32_t precision;   /* enum ctd_precision                                               */
  int32_t max_batch;   /* pages per ctd_infer call the workspace is sized for              */
  int32_t max_h, max_w; /* largest page (multiples of 64)                                  */
  int32_t nc;          /* classes of the Detect head (reference: 2, inference.py:117-118)  */
  int32_t use_graph;   /* 1: capture the op list into a CUDA graph per (n,h,w)             */
  float conf_thresh;   /* 0.4  (inference.py:120)                                          */
  float nms_thresh;    /* 0.35 (inference.py:120)                                          */
  float db_thresh;     /* 0.3  (inference.py:139 -> db_utils.py:71-72)                     */
  int32_t debug_skip_postproc; /* 1: ctd_forward stops after the op list (kernel unit tests)  */
} ctd_config;

typedef struct ctd_handle ctd_handle;

/* Replaces TextDetBase.__init__ / get_base_det_models (basemodel.py:211-227).
 * `blob` is copied to the device; the arrays may be freed after the call.                 */
CTD_API int ctd_create(ctd_handle** out, const ctd_config* cfg, const ctd_op* ops, int32_t n_ops,
               const ctd_bufdesc* bufs, int32_t n_bufs, const void* blob, size_t blob_bytes);
CTD_API void ctd_destroy(ctd_handle* h);
CTD_API const char* ctd_last_error(const ctd_handle* h); /* h may be NULL: last create() error     */

/* ---- the forward pass --------------------------------------------------------------------
 * Replaces `TextDetBase.forward` (basemodel.py:240-244) fed by `preprocess_img` for
 * net-sized pages (inference.py:72-83: BGR u8 HWC -> BGR f32 NCHW /255; the /255 and the
 * layout change are fused into the stem kernel).
 *
 * pages : n*h*w*3 bytes, BGR, HWC, u8.  `pages_on_device` != 0 means a device pointer.
 * The result stays on the device inside the handle; fetch what you need with ctd_get_*.   */
CTD_API int ctd_forward(ctd_handle* h, const uint8_t* pages, int32_t n, int32_t ph, int32_t pw, int32_t pages_on_device);

/* Net-level outputs (the tuple TextDetBase.forward returns), copied to HOST memory.
 * blks  : f32 [n][A][5+nc], A = 3*(h/8*w/8 + h/16*w/16 + h/32*w/32)     (yolo.py:44)
 * mask  : f32 [n][h][w] in (0,1)                                        (basemodel.py:57-60)
 * lines : f32 [n][2][h][w] = (shrink, threshold)                        (basemodel.py:125)
 * Any pointer may be NULL to skip it.                                                      */
CTD_API int ctd_get_net_outputs(ctd_handle* h, float* blks, float* mask, float* lines);

/* `postprocess_mask` (inference.py:85-99): (mask*255) truncated to u8, [n][h][w], HOST.   */
CTD_API int ctd_get_mask_u8(ctd_handle* h, uint8_t* mask_u8);

/* `postprocess_yolo` up to the numpy conversion (inference.py:101-105) =
 * `non_max_suppression(det, conf, iou)[i]` (utils/yolov5_utils.py:124-218): rows
 * [x1,y1,x2,y2,conf,cls] f32, score-descending, at most 300 per page.
 * det: HOST f32 [n][300][6]; det_count: HOST i32 [n].                                      */
CTD_API int ctd_get_detections(ctd_handle* h, float* det, int32_t* det_count);
/* Candidate capacity of the NMS stage.  The reference keeps up to max_nms = 30000 candidates per page
 * (yolov5_utils.py:143,191-194); this engine holds *cap = 4096.  A page with more rows above conf_thresh keeps
 * exactly the 4096 best by (score descending, row ascending) -- deterministic, and identical to the reference
 * whenever the reference's own 300-detection cut (max_det) is reached inside those rows.  cand_total: HOST i32 [n],
 * the number of candidates each page of the last forward (or the last ctd_nms call, n = 1) really had, so a caller
 * can detect cand_total[i] > *cap.  Either pointer may be NULL.                                */
CTD_API int ctd_get_nms_status(ctd_handle* h, int32_t* cand_total, int32_t* cap);

/* `SegDetectorRepresenter.binarize` + connected components of the shrink map
 * (db_utils.py:71-72 and the labelling findContours/connectedComponents imply):
 * bitmap u8 [n][h][w] (0/1), labels i32 [n][h][w] numbered like
 * cv2.connectedComponents(connectivity=8) (0 = background), n_labels i32 [n] (incl. bg).
 * Any pointer may be NULL.                                                                 */
CTD_API int ctd_get_db_components(ctd_handle* h, uint8_t* bitmap, int32_t* labels, int32_t* n_labels);

/* `SegDetectorRepresenter.__call__` -> `boxes_from_bitmap` (db_utils.py:40-69,123-166) on the shrink map of
 * the last forward: per page the contours in OpenCV's findContours(RETR_LIST) order, capped at 1000
 * (max_candidates); rows of skipped contours (short side < 2) are zero with score 0 exactly like the
 * reference.  boxes: HOST i16 [n][1000][4][2] (x,y; order TL,TR,BR,BL), scores: HOST f32 [n][1000],
 * counts: HOST i32 [n] = min(#contours, 1000).  The box_thresh (0.6) filter of inference.py:159-161 is
 * left to the caller, as in the reference.                                                        */
CTD_API int ctd_get_text_lines(ctd_handle* h, int16_t* boxes, float* scores, int32_t* counts);

/* ---- pages that are not net-sized (SURVEY 8f row f1) -----------------------------------------
 * `letterbox(im, new_shape, auto=False)` + `preprocess_img` (imgproc_utils.py:86-117, inference.py:72-83) on the
 * GPU: the HOST page (u8 BGR HWC, any size ih x iw) is resized with OpenCV-exact INTER_LINEAR to
 * unpad_h x unpad_w (the caller computes these with the reference's formula: r = min(net_h/ih, net_w/iw),
 * unpad = round(size * r)), zero-padded bottom/right to net_h x net_w (multiples of 64) and forwarded (n = 1).   */
CTD_API int ctd_forward_resized(ctd_handle* h, const uint8_t* page, int32_t ih, int32_t iw, int32_t unpad_h, int32_t unpad_w,
                                int32_t net_h, int32_t net_w);
/* Mask back-projection (inference.py:164-168): `mask[:crop_h, :crop_w]` of page 0 of the last forward,
 * `cv2.resize(.., (out_w, out_h), INTER_LINEAR)` -> HOST u8 [out_h][out_w].                                      */
CTD_API int ctd_get_mask_u8_resized(ctd_handle* h, int32_t crop_h, int32_t crop_w, int32_t out_h, int32_t out_w,
                                    uint8_t* mask_out);
/* Stand-alone `cv2.resize(src, (dw, dh), interpolation=cv2.INTER_LINEAR)` for u8 images with 1 or 3 channels
 * (HOST in, HOST out); bit-exact with OpenCV 4.x, see csrc/resize.cu.                                            */
CTD_API int ctd_resize_linear_u8(ctd_handle* h, const uint8_t* src, int32_t sh, int32_t sw, int32_t channels, uint8_t* dst,
                                 int32_t dh, int32_t dw);

/* ---- pipelined host-buffer path (throughput mode of ctd_forward + ctd_get_*) -----------------
 * The reference serves pages one call at a time (inference.py:141-178: H2D, net, D2H, numpy post-
 * processing, all serial).  A caller that streams batches keeps two in flight instead:
 *   ctd_submit(h, slot, pages, n, ph, pw, results)   asynchronous: H2D of the HOST pages on a copy
 *       stream, the whole forward + post-processing on the engine stream, D2H of the result arena
 *       (mask_u8 | det | det_count | n_labels | line_boxes | line_scores | line_count, layout of
 *       ctd_device_outputs / ctd_results_bytes) into HOST `results` on a second copy stream;
 *   ctd_collect(h, slot)                              blocks until that slot's `results` are complete.
 * slot is 0 or 1; a slot must be collected before it is submitted again.  `pages` and `results`
 * should be pinned (cudaHostAlloc / torch pin_memory) or the copies serialise.  Submissions execute
 * in order; ctd_get_* after a submit refer to the most recently submitted batch.               */
CTD_API int ctd_submit(ctd_handle* h, int32_t slot, const uint8_t* pages_host, int32_t n, int32_t ph, int32_t pw,
                       void* results_host);
CTD_API int ctd_collect(ctd_handle* h, int32_t slot);
CTD_API int ctd_results_bytes(ctd_handle* h, size_t* bytes);

/* Several handles on ONE GPU (one workspace each) let independent batches overlap: the kernels of batch i+1 fill the
 * tails and dependency gaps of batch i (+8 % pages/s with two handles, bench.py).  ctd_join makes everything
 * enqueued so far on `other`'s stream a dependency of `h`'s stream (device-side, no host wait) -- used to close a
 * timed region or to hand results over.                                                         */
CTD_API int ctd_join(ctd_handle* h, ctd_handle* other);

/* Device-side timing of the last ctd_forward (CUDA events on the engine stream), ms.       */
CTD_API int ctd_last_forward_ms(ctd_handle* h, float* ms);
/* Number of kernels the last ctd_forward launched (graph nodes when captured).             */
CTD_API int ctd_last_launch_count(ctd_handle* h, int32_t* launches);
/* Debug/bisect: copy activation buffer `buf` of the last forward to HOST as f32 NHWC.      */
CTD_API int ctd_debug_read_buffer(ctd_handle* h, int32_t buf, float* out, size_t out_elems);
/* Debug/unit tests: fill activation buffer `buf` (f32 NHWC on the host, converted to the engine's
 * storage type) for a forward of shape (n, ph, pw); used with programs that have no STEM op.  */
CTD_API int ctd_debug_write_buffer(ctd_handle* h, int32_t buf, const float* in, int32_t n, int32_t ph, int32_t pw);

/* Debug/unit tests: run only ops [first_op, last_op] of the program on the CURRENT buffer contents (fill sources
 * with ctd_debug_write_buffer, read the result with ctd_debug_read_buffer): one launch plan of the real network at
 * the real shape, checked in isolation.  `pages` (HOST u8 [n][ph][pw][3]) may be NULL unless the range contains
 * the STEM op.  Synchronous, never graph-captured, no post-processing.                              */
CTD_API int ctd_debug_run_ops(ctd_handle* h, const uint8_t* pages, int32_t n, int32_t ph, int32_t pw, int32_t first_op,
                              int32_t last_op);

/* ---- measurement / interop ------------------------------------------------------------------
 * CUDA-event timer on the ENGINE stream (bench.py times K forwards between start and stop).    */
CTD_API int ctd_timer_start(ctd_handle* h);
CTD_API int ctd_timer_stop(ctd_handle* h, float* ms); /* synchronises the engine stream          */
/* One un-graphed forward with an event after every op: op_ms[i] = device ms of op i; the two
 * entries after the last op are the NMS and the CCL stage.  cap >= n_ops + 2.                   */
CTD_API int ctd_profile_forward(ctd_handle* h, const uint8_t* pages, int32_t n, int32_t ph, int32_t pw,
                                int32_t pages_on_device, float* op_ms, int32_t cap);
/* Device pointers of the last forward's results (valid until the next call on this handle) and
 * the engine's cudaStream_t, so a caller can hand them to NCCL without a host round trip.       */
typedef struct ctd_device_outputs {
  void* stream;      /* cudaStream_t                                  */
  void* mask_u8;     /* u8  [n][h][w]                                 */
  void* det;         /* f32 [n][300][6]                               */
  void* det_count;   /* i32 [n]                                       */
  void* bitmap;      /* u8  [n][h][w]                                 */
  void* labels;      /* i32 [n][h][w]                                 */
  void* n_labels;    /* i32 [n]                                       */
  void* line_boxes;  /* i16 [n][1000][4][2]                           */
  void* line_scores; /* f32 [n][1000]                                 */
  void* line_count;  /* i32 [n]                                       */
  void* results_base;   /* mask_u8 | det | det_count | n_labels | line_* live in ONE allocation sized for
                           max_batch, so a single NCCL gather moves a rank's results          */
  size_t results_bytes;
} ctd_device_outputs;
CTD_API int ctd_get_device_outputs(ctd_handle* h, ctd_device_outputs* out);

/* ---- stand-alone array kernels (stage-isolated parity; same kernels the pipeline uses) --
 * cv2.connectedComponentsWithStats(img, connectivity=8, ltype=CV_32S) as the reference
 * effectively calls it (utils/textmask.py:93,113,138; SURVEY App. D #16).
 * img u8 [h][w] (non-zero = foreground), HOST pointers.  labels i32 [h][w];
 * stats i32 [n_labels][5] = x,y,w,h,area (row 0 = background); returns count in *n_labels.
 * `stats_cap` = rows available in `stats`.                                                 */
CTD_API int ctd_connected_components(ctd_handle* h, const uint8_t* img, int32_t ih, int32_t iw, int32_t* labels,
                             int32_t* stats, int32_t stats_cap, int32_t* n_labels);

/* Stage-isolated form of the above on a caller-supplied probability map (HOST f32 [ih][iw]):
 * binarize(pred > thresh) -> contours -> boxes/scores, as `SegDetectorRepresenter(thresh).__call__`
 * would return for one image.  boxes i16 [1000][4][2], scores f32 [1000], *count = rows used.       */
CTD_API int ctd_seg_represent(ctd_handle* h, const float* pred, int32_t ih, int32_t iw, float thresh, int16_t* boxes,
                              float* scores, int32_t* count);

/* `refine_mask(img, pred_mask, blk_list, refine_mode)` (utils/textmask.py:159-169): img HOST u8 [ih][iw][3]
 * BGR, mask HOST u8 [ih][iw], windows HOST i32 [n_win][4] = `expand_textwindow(img.shape, blk.xyxy, 16)` of
 * every block (python slice semantics), refine_mode 0 = REFINEMASK_INPAINT, 1 = REFINEMASK_ANNOTATION.
 * out HOST u8 [ih][iw] = mask_refined.  Windows follow python slice semantics (negative bounds wrap).          */
CTD_API int ctd_refine_mask(ctd_handle* h, const uint8_t* img, const uint8_t* mask, int32_t ih, int32_t iw,
                            const int32_t* windows, int32_t n_win, int32_t refine_mode, uint8_t* out);

/* ---- line -> block grouping (host C++, no GPU needed) ---------------------------------------------
 * `group_output(blks, lines, im_w, im_h, mask, sort_blklist)` (utils/textblock.py:421-508) with its callees
 * examine_textblk / split_textblk / try_merge_textline / merge_textlines / sort_textblk_list (267-419) and
 * TextBlock.adjust_bbox / sort_lines (87-105).  One record per resulting TextBlock, field for field
 * (utils/textblock.py:12-85; only the fields group_output assigns are carried).                      */
typedef struct ctd_block {
  int32_t xyxy[4];       /* TextBlock.xyxy                                                  */
  int32_t language;      /* index into LANG_LIST = ['eng', 'ja', 'unknown'] (textblock.py:9) */
  int32_t vertical;      /* TextBlock.vertical                                              */
  int32_t angle;         /* TextBlock.angle (degrees)                                       */
  int32_t merged;        /* TextBlock.merged                                                */
  int32_t n_lines;       /* len(TextBlock.lines); rows line_off .. line_off+n_lines-1 of `lines_out` */
  int32_t line_off;
  int32_t n_dist;        /* len(TextBlock.distance) (differs from n_lines for split blocks: the reference
                            deep-copies the parent's distance array, textblock.py:397,412)   */
  int32_t dist_off;
  int32_t font_is_float; /* python type of font_size: int until try_merge_textline averages it */
  int32_t reserved;
  double font_size;      /* TextBlock.font_size                                             */
  double vec[2];         /* TextBlock.vec                                                   */
  double norm;           /* TextBlock.norm                                                  */
  double weight;         /* TextBlock.weight (reading-order key, -1 when sort_blklist = 0)  */
} ctd_block;

/* Capacity of one page's block section in the result arena / of ctd_detect_page's outputs: the reference produces
 * at most max_det (300) detector blocks + one block per text line left over (<= 1000 lines, db_utils.py max_candidates). */
#define CTD_MAX_BLOCKS 1300
#define CTD_MAX_BLOCK_DIST 8192
/* header of a page's block section (see ctd_results_layout); flags bit 0: the distance arrays did not fit and were
 * dropped (n_dist = 0 in every record), bit 1: group_output failed for the page (n_blocks = 0).                 */
typedef struct ctd_page_blocks {
  int32_t n_blocks, n_lines, n_dist, flags;
} ctd_page_blocks;

/* blk_xyxy i32 [n_blk][4], blk_cls i32 [n_blk]: the detector rows after postprocess_yolo (inference.py:101-114);
 * lines i32 [n_lines][4][2]: the kept text-line quads in page coordinates; mask u8 [im_h][im_w] or NULL.
 * Results: blocks_out[*n_blocks], lines_out i32 [..][4][2], dist_out f64 [..].  Returns CTD_E_CAPACITY (with
 * *n_blocks set) when an output array is too small: blocks <= n_blk + n_lines, lines <= n_lines + n_blk,
 * distances <= (n_lines + n_blk) * max lines per block.  Pure host code, thread-safe, needs no handle. */
CTD_API int ctd_group_output(const int32_t* blk_xyxy, const int32_t* blk_cls, int32_t n_blk, const int32_t* lines,
                             int32_t n_lines, int32_t im_w, int32_t im_h, const uint8_t* mask, int32_t sort_blklist,
                             ctd_block* blocks_out, int32_t blocks_cap, int32_t* lines_out, int32_t lines_cap,
                             double* dist_out, int32_t dist_cap, int32_t* n_blocks);
/* `expand_textwindow(img.shape, xyxy, expand_r)` (utils/imgproc_utils.py:151-161) followed by the index
 * normalisation of the python slice `img[y1:y2, x1:x2]` (negative bounds wrap, then clamp): win = x1,y1,x2,y2.  */
CTD_API void ctd_expand_textwindow(int32_t im_w, int32_t im_h, const int32_t* xyxy, int32_t expand_r, int32_t* win);

/* ---- the whole of `TextDetector.__call__` (inference.py:141-178) ---------------------------------------------
 * One page of any size: letterbox + forward + post-processing on the GPU, postprocess_yolo casts / box_thresh /
 * group_output / expand_textwindow on the host (C++), refine_mask (and, with keep_undetected != 0,
 * refine_undetected_mask, textmask.py:135-156) on the GPU with the page and its mask resident in HBM.
 * page HOST u8 [ih][iw][3] BGR; net_h x net_w = the detector's input_size (<= the engine's max shape, multiples of
 * 64); mask_out / mask_refined_out HOST u8 [ih][iw] (mask_out is the page-sized mask, modified in place by
 * refine_undetected_mask exactly like the reference's); blocks / lines_out / dist_out as ctd_group_output.
 * Blocking.  Returns CTD_E_CAPACITY with *n_blocks set when an output array is too small (CTD_MAX_BLOCKS blocks and
 * lines, CTD_MAX_BLOCK_DIST distances always suffice).                                                     */
CTD_API int ctd_detect_page(ctd_handle* h, const uint8_t* page, int32_t ih, int32_t iw, int32_t net_h, int32_t net_w,
                            int32_t refine_mode, int32_t keep_undetected, uint8_t* mask_out, uint8_t* mask_refined_out,
                            ctd_block* blocks, int32_t blocks_cap, int32_t* lines_out, int32_t lines_cap, double* dist_out,
                            int32_t dist_cap, int32_t* n_blocks);

/* Batches of NET-SIZED pages through the same chain, two batches in flight per handle (throughput form of the
 * above; supersedes ctd_submit for callers that want blocks and mask_refined).  ctd_submit_full returns at once:
 * the forward + device post-processing are enqueued, a worker thread of the handle runs the host stage when their
 * results arrive and enqueues refine_mask; ctd_collect(h, slot) blocks until `results_host` is complete.
 * results_host: HOST (pinned) buffer of ctd_results_layout().total_bytes:
 *   [0, phase_a_bytes)  mask_u8 | det | det_count | n_labels | line_boxes | line_scores | line_count (as ctd_submit)
 *   mask_refined        u8 [n][ph][pw]
 *   blocks + i*blocks_stride   page i: ctd_page_blocks header, ctd_block[CTD_MAX_BLOCKS] at +blk_records_off,
 *                       i32 lines [..][4][2] at +blk_lines_off, f64 distances at +blk_dist_off
 * pages: HOST (pinned) pointer, or with pages_on_device != 0 a DEVICE pointer that must stay valid until the slot
 * is collected (refine_mask reads the pages in place).  The same bytes exist on the device (ctd_device_arena) once
 * the slot is collected, so a multi-GPU caller can gather a rank's complete results with one NCCL call.    */
typedef struct ctd_results_layout_t {
  int32_t max_batch, max_h, max_w, reserved;
  size_t total_bytes, phase_a_bytes;
  size_t mask_u8, det, det_count, n_labels, line_boxes, line_scores, line_count;  /* sized for max_batch x max_h x max_w */
  size_t mask_refined, blocks, blocks_stride, blk_records_off, blk_lines_off, blk_dist_off;
} ctd_results_layout_t;
CTD_API int ctd_results_layout(ctd_handle* h, ctd_results_layout_t* out);
CTD_API int ctd_submit_full(ctd_handle* h, int32_t slot, const uint8_t* pages, int32_t n, int32_t ph, int32_t pw,
                            int32_t pages_on_device, int32_t refine_mode, void* results_host);
/* Device copy of slot `slot`'s complete results (same layout) and the stream its last writes were enqueued on.   */
CTD_API int ctd_device_arena(ctd_handle* h, int32_t slot, void** base, void** post_stream);

/* ---- text-line crops for OCR (SURVEY 8f row f4) -----------------------------------------------------------------
 * `TextBlock.get_transformed_region(img, idx, textheight)` (utils/textblock.py:162-194) for many lines in one call:
 * quad expansion by font_size / 3 and clip to [0, im_w] x [0, im_h] (flags bit CTD_REGION_EXPAND), aspect ratio of
 * the quad's mid-lines, output size (h = int(textheight), w = round-half-even(textheight / ratio) for horizontal lines;
 * w = int(textheight), h = round(textheight * ratio) for vertical ones), `cv2.findHomography(src, dst, RANSAC, 5.0)`
 * (4 points: normalised DLT), `cv2.warpPerspective(img, M, (w, h))` (INTER_LINEAR, BORDER_CONSTANT 0, OpenCV's
 * fixed-point arithmetic) and, for vertical lines, `cv2.rotate(.., ROTATE_90_COUNTERCLOCKWISE)`.  Bit-exact with
 * OpenCV 4.x; csrc/regions.cu.  A w or h of 0 gives a crop of the page's size (OpenCV's empty dsize);
 * a line the reference cannot crop gets a non-zero status and no bytes.                                         */
#define CTD_REGION_EXPAND 1          /* flags bit 0: language 'eng', or 'unknown' and not vertical (textblock.py:168) */
#define CTD_REGION_VERTICAL 2        /* flags bit 1: TextBlock.vertical                                            */
#define CTD_REGION_OK 0
#define CTD_REGION_E_RATIO 1         /* ratio 0, inf or nan: the reference's round() raises OverflowError / ValueError */
#define CTD_REGION_E_HOMOGRAPHY 2    /* w or h is 1, or the quad has no extent along x or y: findHomography returns
                                        None and warpPerspective raises cv2.error                                   */
#define CTD_REGION_E_SIZE 3          /* the crop would exceed 2^31 bytes                                            */
typedef struct ctd_region {
  int32_t status;        /* CTD_REGION_*                                                                     */
  int32_t out_h, out_w;  /* crop shape after the rotation of vertical lines (times `channels` bytes per pixel) */
  int32_t w, h;          /* the reference's w, h (dst corners (w-1, h-1))                                    */
  int32_t reserved;
  size_t offset;         /* byte offset of the crop in the packed output (crops follow each other, no padding) */
  size_t bytes;          /* out_h * out_w * channels (0 when status != 0)                                    */
  double M[9];           /* forward homography, row-major: filled by ctd_transform_regions                   */
} ctd_region;
/* Host-only planning (no handle, thread-safe): quads f64 [n][4][2], flags i32 [n], font_size f64 [n] -> regions[n]
 * (status, shape, offset, bytes; M = 0) and *total_bytes of the packed output.  CTD_E_INVALID for channels
 * not in {1, 3}.                                                                                                 */
CTD_API int ctd_plan_regions(const double* quads, const int32_t* flags, const double* font_size, int32_t n, int32_t im_w,
                             int32_t im_h, int32_t channels, double textheight, ctd_region* regions, size_t* total_bytes);
/* All crops of one page in one call on the handle's stream (blocking): img u8 [ih][iw][channels] (HOST, uploaded once
 * into the handle's grow-on-demand scratch, or with img_on_device != 0 a DEVICE pointer, read in place); out receives
 * the packed crops (HOST, or with out_on_device != 0 a DEVICE pointer) and must hold the planned total
 * (CTD_E_CAPACITY otherwise, with regions[] planned).  regions[] as ctd_plan_regions plus the forward M of every
 * line with status 0.                                                                                            */
CTD_API int ctd_transform_regions(ctd_handle* h, const uint8_t* img, int32_t ih, int32_t iw, int32_t channels,
                                  int32_t img_on_device, const double* quads, const int32_t* flags, const double* font_size,
                                  int32_t n, double textheight, ctd_region* regions, uint8_t* out, int32_t out_on_device,
                                  size_t out_bytes);

/* utils/yolov5_utils.py:124-218 on a caller-supplied prediction tensor (HOST f32
 * [rows][5+nc]); output as ctd_get_detections for one page.                                */
CTD_API int ctd_nms(ctd_handle* h, const float* pred, int32_t rows, float conf_thresh, float iou_thresh, float* det,
            int32_t* det_count);

#ifdef __cplusplus
}
#endif
#endif /* CTD_B200_H_ */
