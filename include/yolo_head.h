/*
 * yolo_head.h -- C ABI of libyolohead.so, the B200 (sm_100a) implementation of the YOLOv4 detection-head hot
 * path of zjykzj/YOLOv4.  The reference is pure Python and has no FFI of its own (SURVEY.md 8(b)): the
 * reference-side boundary is the Python call surface of three symbols, and this header is what the Python
 * shim (yolov4_b200/_cabi.py, ctypes) binds to replace each of them.  Every entry point cites the
 * reference interface it replaces.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only; no torch / C++ types.
 *   - every function returns int: 0 = YL_OK, 1..99 = argument errors, 1000+e = cudaError_t e.  Never throws.
 *   - all device-pointer functions are stream-ordered on `stream` (a cudaStream_t passed as void*), do not
 *     allocate, do not synchronise, and are CUDA-graph capturable.
 *   - fp32 everywhere (the reference trains and evaluates with apex O0, README.md:106,112), except the head tensors of the
 *     fused detection path (yl_filter_raw_typed, yl_context_create_typed) and of the fused loss (yl_loss_forward_typed,
 *     yl_loss_forward_chained_typed, yl_loss_backward_typed), which may also be fp16 or bf16 as a model run with .half(), under
 *     autocast or apex O1/O2 produces them: they are widened exactly to fp32 and the fp32 spec applies from there; the loss
 *     gradient is then written in the head's element type.
 *   - sigmoid / exp / log are the "spec math" of DESIGN.md section 4 (fixed IEEE op sequences), so results are
 *     bit-reproducible and identical to the CPU oracle.
 */
#ifndef YOLO_HEAD_H_
#define YOLO_HEAD_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YL_OK 0
#define YL_ERR_ARG 1          /* null pointer / non-positive size / unsupported shape */
#define YL_ERR_CLASSES 2      /* more classes than the candidate bitmask supports (YL_MAX_CLASSES) */
#define YL_ERR_WORKSPACE 3    /* workspace smaller than yl_post_workspace_bytes() */
#define YL_ERR_CAPACITY 4     /* yl_detect_host: a class segment overflowed cap_seg; recreate the context larger */
#define YL_ERR_CUDA_BASE 1000 /* 1000 + cudaError_t */

#define YL_MAX_CLASSES 128
#define YL_ABI_VERSION 1

/* element type of the head tensors of the fused detection path and of the fused loss */
#define YL_DTYPE_F32 0
#define YL_DTYPE_F16 1
#define YL_DTYPE_BF16 2

typedef void *yl_stream_t; /* cudaStream_t */

int yl_abi_version(void);
/* Hash of the sources the library was compiled from (build.py:source_hash); the loader refuses a stale library. */
const char *yl_source_hash(void);
const char *yl_error_string(int code);
/* Self-test of the library's spec math (no reference counterpart): the bounded reciprocal used by the sigmoid against the
 * IEEE quotient for every float in [1, 2^125]; *bad_dev (device u64) receives the number of mismatches. */
int yl_selftest_rcp(unsigned long long *bad_dev, yl_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * A2  YOLOLayer.forward, eval branch                       replaces yolo/model/yololayer.py:88-120,146-166
 *   raw   [B, 3*(5+C), F, F] contiguous device fp32 (head conv output, yolov4.py:235-251)
 *   anch_grid[6] = masked anchors / stride, (w0,h0,w1,h1,w2,h2)               (yololayer.py:73-76)
 *   out   rows of (5+C) floats; box (b,a,y,x) -> row b*rows_per_image + row_offset + a*F*F + y*F + x, so the
 *         three layers can write straight into the torch.cat((x1,x2,x3),1) buffer of yolov4.py:324.
 * The reference's in-place overwrite of `raw` (a side effect nobody reads) is not reproduced.
 * --------------------------------------------------------------------------------------------------------- */
int yl_decode_dense(const float *raw, int B, int F, int C, const float *anch_grid, float stride,
                    float *out, long rows_per_image, long row_offset, yl_stream_t stream);
/* yl_decode_dense with YOLOv4's grid-sensitivity decode (darknet's scale_x_y; DESIGN.md section 1).  With s = scale_x_y and
 * beta = fl32(-0.5 * (s - 1)) evaluated in float64, the box centre of cell (i, j) is
 *   cx = fl(fl(fl(sigmoid(tx) * s) + beta) + i),  bx = fl(cx * stride)           (cy, by likewise with j)
 * every operation one fp32 rounding in this order; w, h, objectness and classes are unchanged, and nothing is clamped (a centre
 * may leave its cell).  s = 1 is yl_decode_dense (the same launch, the same bytes; yl_decode_dense is this call with 1), s = 2
 * is the 2 sigmoid - 0.5 centre of YOLOv5 / Scaled-YOLOv4.  A NaN, infinite or non-positive s returns YL_ERR_ARG before any
 * CUDA call. */
int yl_decode_dense_ex(const float *raw, int B, int F, int C, const float *anch_grid, float stride, float scale_x_y,
                       float *out, long rows_per_image, long row_offset, yl_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * A3  YOLOLayer.forward, train branch                      replaces yolo/model/yololayer.py:122-145
 *   output_planar [B,3,5+C,F,F]: sigmoid on xy/obj/cls, raw wh.  The reference's dict['output'] is the
 *                 permute(0,1,3,4,2) view of this storage (strides (255F^2, 85F^2, F, 1, F^2)).
 *   pred_planar   [B,3,4,F,F]: grid-unit boxes (no *stride); dict['pred'] is its permuted view.
 * yl_decode_train_backward: grad_raw = grad_out * d(output)/d(raw) (sigmoid' on xy/obj/cls, 1 on wh), for
 * the autograd.Function that keeps `output` differentiable (yololoss.py:402-432 back-props through it).
 * --------------------------------------------------------------------------------------------------------- */
int yl_decode_train(const float *raw, int B, int F, int C, const float *anch_grid,
                    float *output_planar, float *pred_planar, yl_stream_t stream);
int yl_decode_train_backward(const float *output_planar, const float *grad_out_planar, int B, int F, int C,
                             float *grad_raw, yl_stream_t stream);
/* The same gradient from the RAW head tensor (sigmoid recomputed with the bits of the forward pass).  This is the form the
 * autograd node uses: the reference's YOLOLoss.forward multiplies dict['output'] by its masks in place
 * (yololoss.py:402-408), so the tensor the forward returned cannot be the one kept for the backward pass. */
int yl_decode_train_backward_raw(const float *raw, const float *grad_out_planar, int B, int F, int C,
                                 float *grad_raw, yl_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * A4+A5  postprocess(prediction, num_classes, conf_thre, nms_thre)   replaces yolo/util/utils.py:92-223
 *        (and nms, utils.py:32-89, which it calls per (image, class))
 *
 * Two front ends fill the same candidate workspace, one back end consumes it:
 *   yl_filter_raw     fused decode + confidence filter straight from the three raw head tensors (the 495 MB
 *                     dense [B,M,5+C] tensor is never materialised)          yololayer.py:88-166 + utils.py:117-184
 *   yl_filter_dense   confidence filter of an already decoded [B,M,5+C] tensor -- the literal
 *                     postprocess(prediction, ...) entry                      utils.py:117-184
 *   yl_nms            per (image,class) sort (score desc, box index desc) + greedy NMS (drop at IoU >= thr)
 *                     + class-ascending concatenation                        utils.py:32-89, :191-220
 *
 * Workspace: one device buffer of yl_post_workspace_bytes(B, M, C, cap_seg) bytes.  cap_seg = capacity of one
 * (image,class) candidate segment.  Counting is always exact; a segment that receives more than cap_seg
 * candidates is reported through meta[] and the caller re-runs with a larger cap_seg (the shim does).
 *
 * Output: out_rows [B, cap_out, 7] = (x1,y1,x2,y2,obj_conf,cls_conf,cls_idx), image b's K_b rows first;
 *         meta [3*B] int32: meta[b] = K_b (true count, may exceed cap_out -> rows truncated),
 *                            meta[B+b] = max candidates seen in any class segment of image b,
 *                            meta[2B+b] = total candidates of image b.
 * --------------------------------------------------------------------------------------------------------- */
size_t yl_post_workspace_bytes(int B, long M, int C, int cap_seg);

/* Zeroes the per-run counters.  Must precede yl_filter_* on the same stream. */
int yl_post_reset(void *ws, size_t ws_bytes, int B, long M, int C, int cap_seg, yl_stream_t stream);

/* raw[l] = [B, 3*(5+C), F[l], F[l]], l = 0..n_layers-1 (n_layers <= 3), strides 8/16/32 (yololayer.py:54);
 * anchors_px[18] and anchor_mask[9] are cfg MODEL.ANCHORS / ANCHOR_MASK.  M must equal sum 3*F[l]^2.  Any grid sizes F[l] >= 1
 * work (odd and even, in any mix), at any element-aligned base and any batch size (above 21845 images the kernels are launched
 * in slices of images).
 * img_first/img_count select a contiguous image range (used to pipeline image groups on several streams). */
int yl_filter_raw(const float *const *raw, const int *F, int n_layers, int B, int C,
                  const float *anchors_px, const int *anchor_mask, float conf_thre,
                  void *ws, size_t ws_bytes, long M, int cap_seg, int img_first, int img_count,
                  yl_stream_t stream);

/* The two kernels of yl_filter_raw run separately (measurement / pipelining): stages bit 0 = streaming flag kernel
 * (reads every raw byte once, writes 16 B per box), bit 1 = emit kernel (resolves the flagged pairs exactly).
 * Bit 2 (with bit 0 or 1): the call also resets the workspace counters, i.e. it replaces yl_post_reset -- inside the flag
 * kernel where that exists, so a step has one graph node less; only for the first (or only) image group of a step. */
int yl_filter_raw_stage(const float *const *raw, const int *F, int n_layers, int B, int C,
                        const float *anchors_px, const int *anchor_mask, float conf_thre,
                        void *ws, size_t ws_bytes, long M, int cap_seg, int img_first, int img_count,
                        int stages, yl_stream_t stream);

/* yl_filter_raw_stage for head tensors of element type `dtype` (YL_DTYPE_*).  A 16-bit value is widened exactly to fp32 (every
 * fp16 / bf16 value, subnormals, +-0, +-inf and NaN included, has an exact fp32 image), so the candidates are bit for bit those of
 * yl_filter_raw_stage on the widened tensors; the workspace and everything after this call are unchanged.  16-bit input takes the
 * register-staged flag kernel (k_flag_raw) on every scale.  yl_filter_raw and yl_filter_raw_stage are this call with
 * YL_DTYPE_F32.  An unknown dtype returns YL_ERR_ARG before any CUDA call. */
int yl_filter_raw_typed(const void *const *raw, int dtype, const int *F, int n_layers, int B, int C,
                        const float *anchors_px, const int *anchor_mask, float conf_thre, void *ws, size_t ws_bytes,
                        long M, int cap_seg, int img_first, int img_count, int stages, yl_stream_t stream);

/* yl_filter_raw_typed with YOLOv4's grid-sensitivity decode: scale_x_y[l] is head l's scale (the centre of yl_decode_dense_ex),
 * NULL = every scale 1.  Only the boxes of the candidates change; which (box, class) pairs pass the threshold does not depend
 * on the box.  NULL, or every scale exactly 1, is yl_filter_raw_typed (the same launches, the same bytes; yl_filter_raw_typed
 * is this call with NULL).  A NaN, infinite or non-positive scale returns YL_ERR_ARG before any CUDA call. */
int yl_filter_raw_ex(const void *const *raw, int dtype, const int *F, int n_layers, int B, int C,
                     const float *anchors_px, const int *anchor_mask, float conf_thre, const float *scale_x_y /* [n_layers] */,
                     void *ws, size_t ws_bytes, long M, int cap_seg, int img_first, int img_count, int stages, yl_stream_t stream);

/* pred [B, M, 5+C] decoded (cx,cy,w,h,obj,cls...), not modified (the reference's in-place xyxy overwrite,
 * utils.py:126, is an unobserved side effect).  num_classes <= C limits the row pre-filter (utils.py:139). */
int yl_filter_dense(const float *pred, int B, long M, int C, int num_classes, float conf_thre,
                    void *ws, size_t ws_bytes, int cap_seg, int img_first, int img_count, yl_stream_t stream);

int yl_nms(void *ws, size_t ws_bytes, int B, long M, int C, int cap_seg, float nms_thre,
           float *out_rows, long cap_out, int *meta, int img_first, int img_count, yl_stream_t stream);

/* yl_nms with a per-image detection cap (max_det; the max_det / detections_per_img option of other detectors).  Let K_b be
 * image b's uncapped row count and s = fl32(obj_conf * cls_conf) (rows' columns 4 x 5, -0 counted as +0).  When K_b > max_det,
 * the kept rows are the first max_det of a STABLE descending sort of the uncapped rows by s (equal scores keep the uncapped
 * order: lower class first, then the order inside the class), emitted in the uncapped order (class ascending, score
 * descending), so every consumer of yl_nms output takes them unchanged.  Within a class the uncapped rows are already in
 * score order, so the cap keeps a prefix of every (image, class) segment: one extra kernel (k_select_topk, one CTA per
 * image, radix select of the max_det-th largest score) lowers the per-class counts before the concatenation.
 *   max_det   0 = no cap (exactly yl_nms: same launches, no extra kernel); 1 <= max_det <= cap_out caps every image;
 *             anything else returns YL_ERR_ARG before any CUDA call
 *   meta[b]   = rows written = min(K_b, max_det); meta[B+b], meta[2B+b] as for yl_nms
 *   uncapped  device int32 [B] receiving K_b for the images of this call, or NULL
 * The workspace is that of yl_post_workspace_bytes(); yl_nms is this call with max_det = 0 and uncapped = NULL. */
int yl_nms_topk(void *ws, size_t ws_bytes, int B, long M, int C, int cap_seg, float nms_thre, int max_det,
                float *out_rows, long cap_out, int *meta, int *uncapped, int img_first, int img_count, yl_stream_t stream);

/* yl_nms_topk with class-agnostic NMS (the agnostic / --agnostic-nms option of other YOLO code bases).  The candidates of an
 * image are the (box, class) pairs of the filter, unchanged; s = fl32(obj_conf * cls_conf), -0 counted as +0.
 *   order        s descending, then class ascending, then box row descending (the stable descending sort by s of the
 *                class-ascending concatenation of the per-class orders: the tie rule of max_det)
 *   suppression  walking that order, a candidate is dropped when IoU >= nms_thre (the literal NaN-propagating formula of
 *                utils.py:71-77) with any earlier kept candidate, whatever either class is
 *   output       the kept candidates as ordinary rows, classes ascending, then s descending, then row descending; max_det then
 *                caps the agnostic rows as stated for yl_nms_topk
 * So a box keeps at most one label, its best-scoring passing class -- except a degenerate box (NaN, zero or negative extent,
 * overflowing area), whose self-IoU is below nms_thre: it keeps every copy, as the literal algorithm does.
 *   agnostic   0 = yl_nms_topk (same launches, same bytes); 1 = class-agnostic; anything else returns YL_ERR_ARG before any
 *              CUDA call.  With 1, ws must hold yl_post_workspace_bytes_ex(B, M, C, cap_seg, 1) bytes, M < 2^25 and
 *              C * cap_seg < 2^32 (else YL_ERR_ARG).  meta[b] is the agnostic row count (capped by max_det), meta[B+b] and
 *              meta[2B+b] are as for yl_nms; uncapped receives the agnostic count before the cap.
 * Image groups (img_first / img_count) use only their own images' slices of the workspace. */
int yl_nms_ex(void *ws, size_t ws_bytes, int B, long M, int C, int cap_seg, float nms_thre, int max_det, int agnostic,
              float *out_rows, long cap_out, int *meta, int *uncapped, int img_first, int img_count, yl_stream_t stream);
/* yl_nms_ex with DIoU-NMS (Zheng et al., AAAI 2020; the DIoU-NMS of the YOLOv4 paper).  The candidates, their order, the rows,
 * their order in the output, max_det and the capacity protocol are those of yl_nms_ex (per class, or agnostic with
 * agnostic = 1); only the suppression decision changes.  A candidate a is dropped by an earlier kept box b (both x1,y1,x2,y2)
 * when, every operation one fp32 rounding in this order and max / min propagating NaN:
 *   iou = the literal NaN-propagating IoU of utils.py:71-77 (the decision of yl_nms)
 *   dx  = (a.x1 + a.x2) * 0.5 - (b.x1 + b.x2) * 0.5        dy = (a.y1 + a.y2) * 0.5 - (b.y1 + b.y2) * 0.5
 *   cw  = max(a.x2, b.x2) - min(a.x1, b.x1)                 ch = max(a.y2, b.y2) - min(a.y1, b.y1)
 *   pen = (dx*dx + dy*dy) / (cw*cw + ch*ch)
 *   suppress  <=>  (iou - pen) >= nms_thre
 * ">=" is the paper's rule and the reference's rule for IoU (darknet's diounms uses ">" and an exponent beta_nms, which this
 * call does not have).  pen >= 0 or NaN, so a pair the IoU rule keeps apart is never suppressed here: a NaN penalty (c^2 = 0,
 * inf / inf) decides "keep", and a degenerate box (NaN, zero or negative extent) never suppresses anything at nms_thre > 0,
 * itself included.  With nms_thre <= 0, boxes that do not overlap can suppress each other, as they do under IoU.
 *   diou   0 = yl_nms_ex (same launches, same bytes); 1 = DIoU-NMS; anything else returns YL_ERR_ARG before any CUDA call.
 * The workspace is that of yl_nms_ex (yl_post_workspace_bytes_ex with the same agnostic). */
int yl_nms_ex2(void *ws, size_t ws_bytes, int B, long M, int C, int cap_seg, float nms_thre, int max_det, int agnostic, int diou,
               float *out_rows, long cap_out, int *meta, int *uncapped, int img_first, int img_count, yl_stream_t stream);
/* Workspace bytes for yl_nms_ex: agnostic = 0 is yl_post_workspace_bytes(); 1 adds 8 bytes per candidate slot
 * (B * C * cap_seg) of scratch for images whose survivors exceed shared memory; anything else returns 0. */
size_t yl_post_workspace_bytes_ex(int B, long M, int C, int cap_seg, int agnostic);

/* ---------------------------------------------------------------------------------------------------------
 * A6+A7  YOLOLoss.build_target(output, pred, layer_no, labels)      replaces yolo/model/yololoss.py:118-371
 *        (and bboxes_iou, yololoss.py:16-91, which it calls twice per image)
 *   pred          element (b,a,j,i,k) at pred[b*ps[0] + a*ps[1] + j*ps[2] + i*ps[3] + k*ps[4]] (floats); the
 *                 reference passes a non-contiguous view with strides (255F^2, 85F^2, F, 1, F^2)
 *   labels        [B,K,5] fp32 (xc,yc,w,h,cls) in input pixels, zero padded (transform.py:464-471)
 *   outputs       dense contiguous fp32: target [B,3,F,F,5+C], obj_mask [B,3,F,F], tgt_mask [B,3,F,F,4+C],
 *                 tgt_scale [B,3,F,F,2]  (yololoss.py:156-167)
 *   status        device int32[1], set non-zero if a matched GT indexes outside the grid (the reference
 *                 raises IndexError there); may be NULL.
 * --------------------------------------------------------------------------------------------------------- */
int yl_build_target(const float *pred, const long *pred_strides, const float *labels, int B, int F, int K,
                    int C, int layer_no, const float *anchors_px, const int *anchor_mask3, float ignore_thre,
                    float *target, float *obj_mask, float *tgt_mask, float *tgt_scale, int *status,
                    yl_stream_t stream);
/* The same for up to three scales in ONE pair of launches (the form YOLOLoss.forward uses, yololoss.py:381-393 loops over the
 * layers): the small grids' latency-bound CTAs run next to the 76x76 ones.  pred[l] / target[l] / ... per scale as above,
 * ps15 = the n_layers stride quintuples back to back, F[l] the grid sizes, layer_no[l] the scale numbers, anchor_mask = the
 * full 3x3 mask table (row layer_no[l] is used).  Results are identical to n_layers calls of yl_build_target. */
int yl_build_target3(const float *const *pred, const long *ps15, const float *labels, int B, const int *F, int K,
                     int C, int n_layers, const int *layer_no, const float *anchors_px, const int *anchor_mask,
                     float ignore_thre, float *const *target, float *const *obj_mask, float *const *tgt_mask,
                     float *const *tgt_scale, int *status, yl_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * N1 (SURVEY.md 8f)  per-detection epilogue of the reference's callers
 *   mode 0: validate()  yolo/engine/build.py:146-164 + yolobox2xywh (yolo/util/utils.py:281-309), float64 like the Python loop
 *           out row = (image_id, category_id, x, y, w, h, score = obj_conf*cls_conf)
 *   mode 1: detect.parse_info()  detect.py:171-179 + yolobox2yxyx (utils.py:312-340), fp32 box arithmetic
 *           out row = (image_id, category_id, y1, x1, y2, x2, cls_conf)
 *   rows [K,7] fp32 (postprocess output rows back to back), row_image [K] image index of each row,
 *   img_info [n_img,4] = (src_h, src_w, dst_h, dst_w) float64, image_ids [n_img] int64, class_ids [n_classes] int32 (all device)
 * --------------------------------------------------------------------------------------------------------- */
int yl_coco_rows(const float *rows, const int *row_image, long K, const double *img_info, const long long *image_ids,
                 const int *class_ids, int n_classes, int mode, double *out, yl_stream_t stream);
/* The same epilogue straight on the padded device output of yl_nms (rows [B, cap_out, 7] + counts [B] = meta[0..B)): one launch
 * for the whole batch, no concatenation and no per-image index tensor; out is compact, [sum counts, 7], image b's rows at the
 * exclusive prefix of the counts. */
int yl_coco_rows_padded(const float *rows, const int *counts, int B, long cap_out, const double *img_info,
                        const long long *image_ids, const int *class_ids, int n_classes, int mode, double *out,
                        yl_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * N2 (SURVEY.md 8f)  YOLOLoss.forward for one layer, fused            replaces yolo/model/yololoss.py:390-432
 *                    (with the train-mode YOLOLayer, yololayer.py:122-145, and build_target, :118-371, it consumes)
 *   raw        [B, 3*(5+C), F, F] raw head tensor of the layer (device fp32)
 *   labels     [B,K,5] fp32 as for yl_build_target
 *   loss4      device float64[4], ACCUMULATED into: loss_xy (:421), loss_wh (:423), loss_obj (:425), loss_cls (:427);
 *              the layer's loss is their sum (:432); zero it before the first layer
 *   saved for yl_loss_backward: gobj [B,3,F,F] fp32 (d loss / d raw objectness), tcell_all / mcell int32 [B,K],
 *              mgrad [B,K,4+C] fp32 (d loss / d raw xy,wh,classes of the matched cells)
 *   status     device int32[1] (caller zeroes it), set non-zero when a matched GT indexes outside the grid or carries a
 *              class id outside [0, C) (the reference raises IndexError / writes another channel there); may be NULL
 * yl_loss_backward: grad_raw [B, 3*(5+C), F, F] = upstream[0] * d loss / d raw (upstream: device fp32 scalar).
 * None of the reference's dense output / pred / target / mask tensors is materialised: 5 of the 5+C planes are read.
 * Aliasing rule: calls for different layers issued back to back on one stream (yl_loss_forward_chained) overlap on the device
 * (programmatic dependent launch: the next layer's matching runs in the tail of this layer's objectness kernel), so gobj / tcell_all /
 * mcell / mgrad of consecutive calls must be distinct buffers (one set per layer, as yl_loss_backward needs anyway);
 * loss4 and status are shared and only accumulated into.  YL_PDL=0 restores plain stream order.
 * --------------------------------------------------------------------------------------------------------- */
int yl_loss_forward(const float *raw, const float *labels, int B, int F, int K, int C, int layer_no,
                    const float *anchors_px, const int *anchor_mask3, float ignore_thre,
                    double *loss4, float *gobj, int *tcell_all, int *mcell, float *mgrad, int *status,
                    yl_stream_t stream);
/* The same call for the SECOND and later layers of one loss evaluation, issued directly behind the previous layer's
 * yl_loss_forward[_chained] on the same stream: its matching kernel is launched programmatically and starts in the tail of
 * the previous layer's objectness kernel.  It reads raw / labels and accumulates into loss4 / status before it waits for
 * that kernel, which is safe only because its predecessor is this library's own kernel; behind anything else (the
 * producer of raw or labels, the fill that zeroes loss4) use yl_loss_forward, a normal, fully ordered launch. */
int yl_loss_forward_chained(const float *raw, const float *labels, int B, int F, int K, int C, int layer_no,
                    const float *anchors_px, const int *anchor_mask3, float ignore_thre,
                    double *loss4, float *gobj, int *tcell_all, int *mcell, float *mgrad, int *status,
                    yl_stream_t stream);
int yl_loss_backward(const float *gobj, const int *mcell, const float *mgrad, const float *upstream,
                     int B, int F, int K, int C, float *grad_raw, yl_stream_t stream);
/* The three loss calls for head tensors of element type `dtype` (YL_DTYPE_*); yl_loss_forward, yl_loss_forward_chained and
 * yl_loss_backward are these calls with YL_DTYPE_F32.  An unknown dtype returns YL_ERR_ARG before any CUDA call.
 *   forward    raw [B, 3*(5+C), F, F] of that type.  Every fp16 / bf16 value (subnormals, +-0, +-inf and NaN included) has an
 *              exact fp32 image: each element is widened on load and the fp32 loss of the fp32 call applies unchanged, so loss4
 *              equals that of the fp32 call on the widened tensor up to the order of the fp64 sums.  The saved tables (gobj,
 *              tcell_all, mcell, mgrad) stay fp32 with the same shapes, and the aliasing rule above is unchanged.
 *   backward   grad_raw [B, 3*(5+C), F, F] of that type: every element is the fp32 call's value fl32(d * upstream[0]), rounded
 *              once to nearest-even into the type (so a large loss scale overflows to +-inf where the rounded value does).
 * This is not the reference's own half-precision arithmetic; it is the fp32 loss of the widened heads. */
int yl_loss_forward_typed(const void *raw, int dtype, const float *labels, int B, int F, int K, int C, int layer_no,
                          const float *anchors_px, const int *anchor_mask3, float ignore_thre,
                          double *loss4, float *gobj, int *tcell_all, int *mcell, float *mgrad, int *status,
                          yl_stream_t stream);
int yl_loss_forward_chained_typed(const void *raw, int dtype, const float *labels, int B, int F, int K, int C, int layer_no,
                                  const float *anchors_px, const int *anchor_mask3, float ignore_thre,
                                  double *loss4, float *gobj, int *tcell_all, int *mcell, float *mgrad, int *status,
                                  yl_stream_t stream);
int yl_loss_backward_typed(const float *gobj, const int *mcell, const float *mgrad, const float *upstream,
                           int B, int F, int K, int C, void *grad_raw, int dtype, yl_stream_t stream);

/* IoU box regression in the fused loss (YOLOv4's CIoU, darknet's iou_loss = giou / diou / ciou).  yl_loss_forward_ex is the
 * forward call of all of the above: yl_loss_forward[_typed] is it with iou_loss = YL_IOU_LOSS_NONE, iou_normalizer = 1,
 * chained = 0, and yl_loss_forward_chained[_typed] the same with chained = 1 (chained = 1: the PDL launch and its rule above).
 *   iou_loss NONE   the loss above, bit for bit
 *   GIOU/DIOU/CIOU  the xy BCE and wh MSE of every matched cell are replaced by iou_normalizer * L(p, g): torchvision's
 *            generalized_ / distance_ / complete_box_iou_loss (eps = 1e-7) of the train-mode predicted box p (grid units, the
 *            fp32 bits of the decode) and the cell's last matched GT g (label / stride), on the xyxy corners x +- w / 2.  No
 *            tgt_scale weighting.  loss4[0] accumulates the box term, loss4[1] receives nothing, loss4[2] / loss4[3] and the
 *            objectness / class gradients are those of YL_IOU_LOSS_NONE.  mgrad[..., 0:4] holds iou_normalizer * d L / d raw
 *            (CIoU's alpha held constant, ties of the min / max split evenly; fp32, see DESIGN.md section 1 for the bound);
 *            a NaN term gives NaN in the cell's four entries.
 * An unknown iou_loss, a negative, NaN or infinite iou_normalizer, or an unknown dtype returns YL_ERR_ARG before any CUDA
 * call.  The saved tables, the aliasing rule and yl_loss_backward[_typed] are unchanged. */
#define YL_IOU_LOSS_NONE 0
#define YL_IOU_LOSS_GIOU 1
#define YL_IOU_LOSS_DIOU 2
#define YL_IOU_LOSS_CIOU 3
int yl_loss_forward_ex(const void *raw, int dtype, const float *labels, int B, int F, int K, int C, int layer_no,
                       const float *anchors_px, const int *anchor_mask3, float ignore_thre, int iou_loss, float iou_normalizer,
                       int chained, double *loss4, float *gobj, int *tcell_all, int *mcell, float *mgrad, int *status,
                       yl_stream_t stream);
/* yl_loss_forward_ex with YOLOv4's grid-sensitivity decode of the layer (darknet's scale_x_y, which yolov4.cfg pairs with
 * iou_loss = ciou).  The train-mode predicted box p of the ignore test and of the IoU box term takes the centre
 * fl(fl(fl(sigmoid(tx) * s) + beta) + i) (beta as for yl_decode_dense_ex; cy likewise), and d px / d tx = s sigmoid (1 - sigmoid):
 * mgrad[..., 0:2] = fl(fl(fl(iou_normalizer * d L / d px) * s) * sigmoid) * (1 - sigmoid).  w / h, the objectness and class
 * terms and yl_loss_backward[_typed] are unchanged.  s = 1 is yl_loss_forward_ex (the same launches, the same bytes;
 * yl_loss_forward_ex is this call with 1).  A NaN, infinite or non-positive s, or s != 1 with YL_IOU_LOSS_NONE (the BCE xy
 * term has no scaled form), returns YL_ERR_ARG before any CUDA call. */
int yl_loss_forward_ex2(const void *raw, int dtype, const float *labels, int B, int F, int K, int C, int layer_no,
                        const float *anchors_px, const int *anchor_mask3, float ignore_thre, int iou_loss, float iou_normalizer,
                        float scale_x_y, int chained, double *loss4, float *gobj, int *tcell_all, int *mcell, float *mgrad,
                        int *status, yl_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * Host-buffer entry (what a non-Python caller binds; also the bench's end-to-end leg): raw head tensors in
 * HOST memory -> detections in HOST memory.  The context owns device staging buffers, workspace, streams and
 * pinned bounce buffers; H2D copies, kernels and the D2H of rows/counts are all inside the call.
 *   raw_host[l] [B, 3*(5+C), F[l], F[l]] host (pinned or pageable), elements of the context's dtype: fp32 for yl_context_create;
 *               for yl_context_create_typed with YL_DTYPE_F16 / YL_DTYPE_BF16, 16-bit elements (IEEE binary16 / bfloat16 bit
 *               patterns), which halves the bytes uploaded
 *   out_rows_host [B, cap_out, 7] fp32, counts_host [B]
 * Returns YL_OK; counts_host[b] > cap_out means image b was truncated.
 * --------------------------------------------------------------------------------------------------------- */
typedef struct yl_context yl_context;
int yl_context_create(yl_context **ctx, int device, int B, const int *F, int n_layers, int C,
                      const float *anchors_px, const int *anchor_mask, int cap_seg, long cap_out);
/* yl_context_create for head tensors of element type `dtype` (YL_DTYPE_*); the device staging buffers hold that type.
 * An unknown dtype returns YL_ERR_ARG before any CUDA call. */
int yl_context_create_typed(yl_context **ctx, int device, int B, const int *F, int n_layers, int C, int dtype,
                            const float *anchors_px, const int *anchor_mask, int cap_seg, long cap_out);
int yl_context_destroy(yl_context *ctx);
int yl_detect_host(yl_context *ctx, const float *const *raw_host, float conf_thre, float nms_thre,
                   float *out_rows_host, int *counts_host);
/* yl_detect_host with a per-image detection cap (yl_nms_topk): counts_host[b] = min(K_b, max_det) and only those rows are
 * copied back.  max_det = 0 is no cap (yl_detect_host is this call with 0); 1 <= max_det <= the context's cap_out, anything
 * else returns YL_ERR_ARG before any CUDA call. */
int yl_detect_host_topk(yl_context *ctx, const float *const *raw_host, float conf_thre, float nms_thre, int max_det,
                        float *out_rows_host, int *counts_host);
/* yl_detect_host_topk with class-agnostic NMS (yl_nms_ex): agnostic = 0 is yl_detect_host_topk, 1 is class-agnostic, anything
 * else returns YL_ERR_ARG before any CUDA call.  The first agnostic call enlarges the context's workspace to
 * yl_post_workspace_bytes_ex(..., 1). */
int yl_detect_host_ex(yl_context *ctx, const float *const *raw_host, float conf_thre, float nms_thre, int max_det, int agnostic,
                      float *out_rows_host, int *counts_host);
/* yl_detect_host_ex with DIoU-NMS (yl_nms_ex2): a candidate a is dropped by an earlier kept box b when
 * fl(iou - pen) >= nms_thre, pen = (dx*dx + dy*dy) / (cw*cw + ch*ch) with the centre distances dx, dy and the enclosing box's
 * extents cw, ch, each operation one fp32 rounding as stated for yl_nms_ex2.  diou = 0 is yl_detect_host_ex, 1 is DIoU-NMS,
 * anything else returns YL_ERR_ARG before any CUDA call. */
int yl_detect_host_ex2(yl_context *ctx, const float *const *raw_host, float conf_thre, float nms_thre, int max_det, int agnostic,
                       int diou, float *out_rows_host, int *counts_host);
/* yl_detect_host_ex2 with YOLOv4's grid-sensitivity decode (yl_filter_raw_ex): scale_x_y[l] is head l's scale, NULL = every
 * scale 1 (yl_detect_host_ex2 is this call with NULL).  A NaN, infinite or non-positive scale returns YL_ERR_ARG before any
 * CUDA call. */
int yl_detect_host_ex3(yl_context *ctx, const float *const *raw_host, float conf_thre, float nms_thre, int max_det, int agnostic,
                       int diou, const float *scale_x_y /* [n_layers] */, float *out_rows_host, int *counts_host);

/* ---------------------------------------------------------------------------------------------------------
 * (e) Multi-GPU: the final exchange of the image-sharded path            (SURVEY.md 8(e); no reference counterpart: the
 *     reference validates on rank 0 only, yolo/engine/build.py:110-190, main_amp.py:175,207)
 * One process per GPU; rank r owns B images and ends up with the detections of all world*B images (rank-major).  Each rank
 * owns one device window (rows / counts / flags) that the peers map through CUDA IPC over NVLink; yl_xchg_push copies
 * exactly counts[b] rows per image into every rank's window with one bulk store per peer (no collective, no host
 * synchronisation), yl_xchg_wait blocks the stream until every rank's rows of that slot have landed, yl_xchg_release
 * hands the slot back (a peer's next push into it waits for that).  All three are graph-capturable, so the exchange of
 * step i runs under the kernels of step i+1 (double-buffered `slots`).
 *   create   cap_out % 4 == 0 (row runs stay 16-byte aligned); slots in [1, 8]
 *   handle   yl_xchg_handle_bytes() opaque bytes of this rank's window, to be all-gathered by the host (torch.distributed)
 *   connect  handles = world * yl_xchg_handle_bytes() bytes, rank-major
 *   push     rows [B, cap_out, 7] fp32 and counts [B] i32 as written by yl_nms (device, rows 16-byte aligned)
 *   rows/counts  device pointers to THIS rank's gathered [world*B, cap_out, 7] / [world*B] of a slot
 *   status   device int32: 0 ok, 1 = a push timed out waiting for a reader, 2 = a wait timed out waiting for a source
 * --------------------------------------------------------------------------------------------------------- */
typedef struct yl_xchg yl_xchg;
int yl_xchg_create(yl_xchg **out, int device, int rank, int world, int B, long cap_out, int slots);
int yl_xchg_destroy(yl_xchg *x);
/* The same object over windows the CALLER owns: `windows[p]` = rank p's window as mapped into this process (all of
 * yl_xchg_window_bytes() bytes, 256-byte aligned; e.g. torch symmetric memory), `multicast` = an NVSwitch multicast mapping of the
 * same windows or NULL.  With a multicast mapping yl_xchg_push issues one bulk store to the multicast mapping and the switch
 * replicates it into every window (a rank sends 1/world of the bytes of the per-peer stores).  No CUDA IPC; yl_xchg_destroy
 * leaves the windows alone.  The caller synchronises the ranks between creation and the first push. */
size_t yl_xchg_window_bytes(int world, int B, long cap_out, int slots);
int yl_xchg_create_external(yl_xchg **out, int device, int rank, int world, int B, long cap_out, int slots,
                            void *const *windows, void *multicast);
size_t yl_xchg_handle_bytes(void);
int yl_xchg_local_handle(yl_xchg *x, void *handle);
int yl_xchg_connect(yl_xchg *x, const void *handles);
int yl_xchg_push(yl_xchg *x, const float *rows, const int *counts, int slot, yl_stream_t stream);
int yl_xchg_wait(yl_xchg *x, int slot, yl_stream_t stream);
int yl_xchg_release(yl_xchg *x, int slot, yl_stream_t stream);
void *yl_xchg_rows(yl_xchg *x, int slot);
void *yl_xchg_counts(yl_xchg *x, int slot);
void *yl_xchg_status(yl_xchg *x);

#ifdef __cplusplus
}
#endif
#endif /* YOLO_HEAD_H_ */
