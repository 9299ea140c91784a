"""postprocess -- drop-in for yolo/util/utils.py:92-223 (and the nms() it calls, :32-89), plus the fused entry.

  postprocess(prediction, num_classes, conf_thre, nms_thre)        the reference's exact call surface
  detect_raw(head_outputs, num_classes, conf_thre, nms_thre, ...)  fused: raw head tensors -> detections,
                                                                   never materialising the dense [B,M,5+C] tensor
  HeadPostprocessor                                                fixed-shape, sync-free, CUDA-graph replayable

All compute runs in libyolohead.so (hand-written sm_100a kernels) through the C ABI; there is no eager fallback.
"""
import threading

import numpy as np
import torch

from . import _cabi

ANCHORS_PX = [[12, 16], [19, 36], [40, 28], [36, 75], [76, 55], [72, 146], [142, 110], [192, 243], [459, 401]]
ANCHOR_MASK = [[0, 1, 2], [3, 4, 5], [6, 7, 8]]

_DEFAULT_CAP_SEG = 1024
_DEFAULT_CAP_OUT = 16384

# head tensor dtypes of the fused path -> YL_DTYPE_* (include/yolo_head.h)
_DTYPE_CODES = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}


def _f32(x):
    """Python-float thresholds are compared in fp32 by torch / NumPy (SURVEY.md 7-4)."""
    return float(np.float32(x))


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _next_pow2(n):
    p = 1
    while p < n:
        p <<= 1
    return p


class _Workspace:
    """Device scratch for one (device, stream, thread, B, M, C, cap_seg): calls of the same shape on different CUDA streams
    or host threads may run concurrently and must not share candidate buffers and counters."""

    _cache = {}

    def __init__(self, device, B, M, C, cap_seg, agnostic=False):
        self.B, self.M, self.C, self.cap_seg = B, M, C, cap_seg
        self.nbytes = _cabi.lib().yl_post_workspace_bytes_ex(B, M, C, cap_seg, int(agnostic))
        if self.nbytes == 0:
            raise _cabi.YoloHeadError("invalid postprocess shape B=%d M=%d C=%d" % (B, M, C))
        self.buf = torch.empty(self.nbytes, dtype=torch.uint8, device=device)

    @classmethod
    def get(cls, device, B, M, C, cap_seg, agnostic=False):
        # agnostic workspaces carry extra scratch (yl_post_workspace_bytes_ex) and are kept apart from the others
        key = (str(device), int(torch.cuda.current_stream(device).cuda_stream), threading.get_ident(), B, M, C, agnostic, cap_seg)
        ws = cls._cache.get(key)
        if ws is None:
            # keep one workspace per (device, stream, thread, B, M, C, agnostic): drop smaller-capacity predecessors
            for k in [k for k in cls._cache if k[:7] == key[:7]]:
                del cls._cache[k]
            ws = cls._cache[key] = cls(device, B, M, C, cap_seg, agnostic)
        return ws

    def ptr(self):
        return self.buf.data_ptr()


_cap_hint = {}    # (B, M, C) -> (cap_seg, cap_out) that were last sufficient


def _check_max_det(max_det):
    """None (no cap) or an int >= 1; checked before any CUDA work."""
    if max_det is None:
        return None
    if isinstance(max_det, bool) or not isinstance(max_det, (int, np.integer)) or int(max_det) < 1:
        raise ValueError("max_det must be None or an int >= 1, got %r" % (max_det,))
    return int(max_det)


def _check_agnostic(agnostic):
    """A bool; checked before any CUDA work."""
    if not isinstance(agnostic, bool):
        raise TypeError("agnostic must be a bool, got %r" % (agnostic,))
    return agnostic


def _check_diou(diou):
    """A bool; checked before any CUDA work."""
    if not isinstance(diou, bool):
        raise TypeError("diou must be a bool, got %r" % (diou,))
    return diou


def _scale_value(v):
    """One scale_x_y value as the fp32 the kernels use: a real number, finite and > 0 in fp32."""
    if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, float, np.integer, np.floating)):
        raise TypeError("scale_x_y values must be real numbers, got %r" % (v,))
    with np.errstate(over="ignore"):
        f = np.float32(v)
    if not np.isfinite(f) or not f > 0:
        raise ValueError("scale_x_y values must be finite and > 0 (in float32), got %r" % (v,))
    return float(f)


def _check_scale_x_y(scale_x_y, n_heads):
    """scale_x_y for n_heads head tensors: None, one real number for every head, or a sequence of one real number per head in
    head order.  Returns None when every scale is 1 (the unscaled decode, bit for bit) and otherwise a list of n_heads fp32
    values.  Raises TypeError / ValueError before any CUDA work."""
    if scale_x_y is None:
        return None
    if isinstance(scale_x_y, (str, bytes)) or not hasattr(scale_x_y, "__len__"):
        vals = [_scale_value(scale_x_y)] * n_heads
    else:
        vals = [_scale_value(v) for v in scale_x_y]
        if len(vals) != n_heads:
            raise ValueError("scale_x_y needs one value per head tensor (%d), got %d" % (n_heads, len(vals)))
    return None if all(v == 1.0 for v in vals) else vals


def _round4(n):
    return (n + 3) // 4 * 4


def _split(rows, meta_host, B, out_device, out_dtype):
    out = []
    for b in range(B):
        k = int(meta_host[b])
        if k == 0:
            out.append(None)                         # utils.py:132,159-160
        else:
            r = rows[b, :k]
            if r.device != out_device or r.dtype != out_dtype:
                r = r.to(device=out_device, dtype=out_dtype)
            out.append(r)
    return out


def _run(front_end, device, B, M, C, nms_thre, max_det=None, agnostic=False, diou=False):
    """Runs front end + NMS, growing cap_seg / cap_out and re-running when the device reports an overflow.  With a cap the
    output holds max_det rows per image (rounded up to a multiple of 4), which no image can exceed; the capacities a capped,
    agnostic or DIoU call settles on are kept apart from those of plain calls."""
    L = _cabi.lib()
    plain = max_det is None and not agnostic and not diou
    hint_key = (B, M, C) if plain else (B, M, C, max_det, agnostic, diou)
    cap_seg, cap_out = _cap_hint.get(hint_key, (_DEFAULT_CAP_SEG, _DEFAULT_CAP_OUT))
    if max_det is not None:
        cap_out = _round4(max_det)
    cap_seg = min(cap_seg, _next_pow2(M))
    while True:
        ws = _Workspace.get(device, B, M, C, cap_seg, agnostic)
        rows = torch.empty((B, cap_out, 7), dtype=torch.float32, device=device)
        meta = torch.empty((3 * B,), dtype=torch.int32, device=device)
        _cabi.check(L.yl_post_reset(ws.ptr(), ws.nbytes, B, M, C, cap_seg, _stream()))
        front_end(ws, cap_seg)
        _cabi.check(L.yl_nms_ex2(ws.ptr(), ws.nbytes, B, M, C, cap_seg, _f32(nms_thre), max_det or 0, int(agnostic), int(diou),
                                 rows.data_ptr(), cap_out, meta.data_ptr(), None, 0, B, _stream()))
        mh = meta.cpu().numpy()                      # the one D2H sync the list-of-tensors contract requires
        max_seg, max_rows = int(mh[B:2 * B].max()), int(mh[:B].max())
        if max_seg > cap_seg:
            cap_seg = _next_pow2(max_seg)
            if max_det is None:
                cap_out = max(cap_out, _next_pow2(int(mh[2 * B:].max())))
            continue
        if max_rows > cap_out:
            cap_out = _next_pow2(max_rows)
            continue
        _cap_hint[hint_key] = (cap_seg, cap_out)
        return rows, mh


def postprocess(prediction, num_classes, conf_thre=0.7, nms_thre=0.45, *, max_det=None, agnostic=False, diou=False):
    """Same contract as the reference's postprocess (yolo/util/utils.py:92).

    prediction: [B, M, 5+C] decoded (cx, cy, w, h, obj, cls...), fp32, on a CUDA device (a CPU tensor, as
    detect.py:115-118 passes, is moved to the current CUDA device and the results are moved back).
    Returns a list of B entries: Tensor[K_i, 7] = (x1, y1, x2, y2, obj_conf, cls_conf, cls_idx), classes
    ascending then score descending, or None for images without detections.
    Differences from the reference, none observable by its callers: `prediction[:, :, :4]` is not overwritten
    in place with the corner form (utils.py:126), and score ties are ordered (score desc, box index desc),
    the order of a stable argsort, where NumPy's default sort leaves them unspecified (utils.py:58).
    num_classes limits the row pre-filter to the first num_classes classes; a value above C means C, as the reference's slice.
    max_det (keyword only, not part of the reference signature): keep at most this many detections per image, those with the
    highest obj_conf * cls_conf (equal scores keep the order above), still listed classes ascending then score descending.
    agnostic (keyword only, not part of the reference signature): class-agnostic NMS, see detect_raw.
    diou (keyword only, not part of the reference signature): DIoU-NMS, see detect_raw.
    """
    max_det = _check_max_det(max_det)
    agnostic = _check_agnostic(agnostic)
    diou = _check_diou(diou)
    if prediction.dim() != 3 or prediction.shape[2] < 6:
        raise ValueError("prediction must be [B, M, 5+C]")
    if prediction.dtype != torch.float32:
        raise TypeError("prediction must be float32 (the reference path runs fp32 / apex O0)")
    in_device = prediction.device
    pred = prediction if prediction.is_cuda else prediction.cuda()
    pred = pred.contiguous()
    B, M, nch = pred.shape
    C = nch - 5
    if B == 0:
        return []
    num_classes = min(int(num_classes), C)           # the reference's slice image_pred[:, 5:5 + num_classes] clamps
    L = _cabi.lib()
    with torch.cuda.device(pred.device):
        def front(ws, cap_seg):
            _cabi.check(L.yl_filter_dense(pred.data_ptr(), B, M, C, num_classes, _f32(conf_thre), ws.ptr(), ws.nbytes,
                                          cap_seg, 0, B, _stream()))
        rows, mh = _run(front, pred.device, B, M, C, nms_thre, max_det, agnostic, diou)
    return _split(rows, mh, B, in_device, prediction.dtype)


def _check_raws(head_outputs, num_classes):
    # the library takes the scale of a head tensor from its position (stride 8 << l, anchor_mask[l]; yololayer.py:54,60):
    # a caller with fewer heads passes them in the reference's order starting at the stride-8 head
    if len(head_outputs) < 1 or len(head_outputs) > 3:
        raise ValueError("expected 1..3 head tensors (stride 8, 16, 32 in this order)")
    if any(head_outputs[i].shape[2] < head_outputs[i + 1].shape[2] for i in range(len(head_outputs) - 1)):
        raise ValueError("head tensors must be ordered stride 8, 16, 32 (largest grid first; yolov4.py:324)")
    B = head_outputs[0].shape[0]
    Fs = []
    raws = []
    for r in head_outputs:
        if r.dim() != 4 or r.shape[0] != B or r.shape[1] != 3 * (5 + num_classes) or r.shape[2] != r.shape[3]:
            raise ValueError("head tensor must be [B, 3*(5+C), F, F], got %s" % (tuple(r.shape),))
        if r.dtype not in _DTYPE_CODES or not r.is_cuda:
            raise TypeError("head tensors must be float32, float16 or bfloat16 CUDA tensors")
        if r.dtype != head_outputs[0].dtype:
            raise TypeError("head tensors must share one dtype, got %s and %s" % (head_outputs[0].dtype, r.dtype))
        raws.append(r.contiguous())
        Fs.append(int(r.shape[2]))
    return raws, B, Fs, _DTYPE_CODES[raws[0].dtype]


def detect_raw(head_outputs, num_classes, conf_thre=0.7, nms_thre=0.45, anchors=ANCHORS_PX, anchor_mask=ANCHOR_MASK, max_det=None,
               agnostic=False, diou=False, scale_x_y=None):
    """Fused YOLOLayer eval decode (yololayer.py:88-166) + postprocess (utils.py:92-223).

    head_outputs: the three raw head conv outputs [B, 3*(5+C), F_l, F_l] (stride 8, 16, 32; yolov4.py:235-251).
    Equivalent to postprocess(torch.cat([YOLOLayer_l(x_l)], 1), num_classes, conf_thre, nms_thre) but reads the
    raw tensors once and never writes the dense decoded tensor.

    The heads may be float32, float16 or bfloat16 (all of one dtype), as a model run with .half() or under
    torch.autocast produces them.  A 16-bit head is widened exactly to float32 and the float32 computation follows, so
    the result is bit for bit detect_raw([h.float() for h in head_outputs], ...).  This is not the reference's own
    half-precision arithmetic, which rounds every sigmoid, exp and product to fp16.  Rows are float32 for every input
    dtype: this entry is not a reference call surface, and float32 rows are what the exact widening produces.

    max_det: keep at most this many detections per image, those with the highest obj_conf * cls_conf; ties keep the
    uncapped order (lower class first, then the order inside the class).  The kept rows stay in the uncapped order, classes
    ascending then score descending.  None (the default) keeps every detection.

    agnostic: class-agnostic NMS.  One greedy NMS per image over all its (box, class) candidates, in the order score
    descending, class ascending, box index descending; a candidate is dropped at IoU >= nms_thre with any earlier kept
    candidate, whatever the classes.  A box then keeps at most one label, its best-scoring passing class (a degenerate box --
    NaN, zero or negative extent, overflowing area -- never suppresses itself and keeps all its labels).  The kept rows are
    listed as usual, classes ascending then score descending; max_det applies to them.  Default False: per-class NMS.

    diou: DIoU-NMS (Zheng et al., AAAI 2020; the DIoU-NMS of the YOLOv4 paper).  Candidates, order, rows and max_det are as
    without it, per class or agnostic; only the suppression decision changes.  A candidate a is dropped by an earlier kept box
    b when fl32(iou - pen) >= nms_thre, with the literal IoU above and pen = (dx*dx + dy*dy) / (cw*cw + ch*ch): dx, dy the
    distances of the box centres ((x1 + x2) * 0.5), cw, ch the extents of the smallest box enclosing both, every operation
    one fp32 rounding, max / min propagating NaN.  A NaN penalty keeps the pair apart, and pen >= 0, so DIoU never suppresses
    a pair IoU keeps apart: boxes far apart that overlap enough for IoU survive as separate detections.  darknet's diounms
    compares with > and an exponent beta_nms; this is the paper's >= with no exponent.  Default False: IoU.

    scale_x_y: YOLOv4's grid-sensitivity decode (darknet's scale_x_y; yolov4.cfg sets 1.2, 1.1, 1.05 for the stride 8, 16,
    32 heads).  With s the head's scale and beta = fl32(-0.5 * (s - 1)) (evaluated in float64), a box centre of cell i is
    fl(fl(fl(sigmoid(tx) * s) + beta) + i) grid units before the stride, every operation one fp32 rounding; nothing is
    clamped.  One real number applies to every head, a sequence gives one value per head tensor in head order.  Only the boxes
    change: the scores, and so which pairs pass conf_thre, do not depend on the scale.  None (the default), 1.0 or all ones is
    the plain decode, bit for bit.  A bool or non-real raises TypeError; a non-finite or non-positive value or a wrong length
    raises ValueError, before any CUDA work.
    """
    max_det = _check_max_det(max_det)
    agnostic = _check_agnostic(agnostic)
    diou = _check_diou(diou)
    sxy = _check_scale_x_y(scale_x_y, len(head_outputs))
    raws, B, Fs, dt = _check_raws(head_outputs, num_classes)
    C = int(num_classes)
    M = sum(3 * f * f for f in Fs)
    L = _cabi.lib()
    dev = raws[0].device
    anch = _cabi.floats([v for wh in anchors for v in wh])
    mask = _cabi.ints([v for m in anchor_mask for v in m])
    rp = _cabi.ptrs([r.data_ptr() for r in raws])
    fs = _cabi.ints(Fs)
    sp = None if sxy is None else _cabi.floats(sxy)
    with torch.cuda.device(dev):
        def front(ws, cap_seg):
            _cabi.check(L.yl_filter_raw_ex(rp, dt, fs, len(raws), B, C, anch, mask, _f32(conf_thre), sp, ws.ptr(), ws.nbytes,
                                           M, cap_seg, 0, B, 3, _stream()))
        rows, mh = _run(front, dev, B, M, C, nms_thre, max_det, agnostic, diou)
    return _split(rows, mh, B, dev, torch.float32)


class HeadPostprocessor:
    """Fixed-shape fused decode + filter + NMS with no host synchronisation: the serving / benchmark form.

    run(head_outputs) enqueues the whole chain on the current stream and returns (rows [B,cap_out,7], meta [3B])
    device tensors owned by this object (overwritten by the next run).  The filter (flag + emit) of every image group runs
    on the current stream and its NMS on a side stream, so with n_groups > 1 the NMS of group g runs next to the filter of
    group g+1; on B200 one group is fastest because every kernel already fills the machine.  capture() records the chain into
    a CUDA graph bound to the given input tensors; replay() launches it.  The head tensors may be float32, float16 or
    bfloat16 (see detect_raw); each run takes the dtype from the tensors it is given.

    max_det caps the detections of every image as in detect_raw; cap_out then defaults to max_det rounded up to a multiple
    of 4, so the output (and a DetectionExchange built with hp.cap_out) is sized by the cap.  uncapped is a device int32 [B]
    with every image's uncapped count, refreshed by every run and replay: meta[b] < uncapped[b] means image b was capped.
    Without a cap uncapped is the view meta[:B].  agnostic selects class-agnostic NMS as in detect_raw (uncapped then counts
    the agnostic rows), and diou DIoU-NMS as in detect_raw.  scale_x_y (one number, or one per grid size) is the
    grid-sensitivity decode of detect_raw, fixed at construction for run / capture / replay.
    """

    def __init__(self, batch, grid_sizes, num_classes, conf_thre, nms_thre, device=None, cap_seg=_DEFAULT_CAP_SEG,
                 cap_out=None, n_groups=1, anchors=ANCHORS_PX, anchor_mask=ANCHOR_MASK, max_det=None, agnostic=False, diou=False,
                 scale_x_y=None):
        self.max_det = _check_max_det(max_det)
        self.agnostic = _check_agnostic(agnostic)
        self.diou = _check_diou(diou)
        self.scale_x_y = _check_scale_x_y(scale_x_y, len(grid_sizes))
        self._sxy = None if self.scale_x_y is None else _cabi.floats(self.scale_x_y)
        if cap_out is None:
            cap_out = _DEFAULT_CAP_OUT if self.max_det is None else _round4(self.max_det)
        if self.max_det is not None and self.max_det > int(cap_out):
            raise ValueError("max_det %d exceeds cap_out %d" % (self.max_det, int(cap_out)))
        self.L = _cabi.lib()
        self.device = torch.device(device if device is not None else "cuda")
        self.B, self.Fs, self.C = int(batch), [int(f) for f in grid_sizes], int(num_classes)
        self.M = sum(3 * f * f for f in self.Fs)
        self.conf, self.nms = _f32(conf_thre), _f32(nms_thre)
        self.cap_seg, self.cap_out = int(cap_seg), int(cap_out)
        self.n_groups = max(1, min(int(n_groups), self.B))
        self.anch = _cabi.floats([v for wh in anchors for v in wh])
        self.mask = _cabi.ints([v for m in anchor_mask for v in m])
        self.fs = _cabi.ints(self.Fs)
        with torch.cuda.device(self.device):
            self.ws = _Workspace(self.device, self.B, self.M, self.C, self.cap_seg, self.agnostic)
            self.rows = torch.empty((self.B, self.cap_out, 7), dtype=torch.float32, device=self.device)
            self.meta = torch.zeros((3 * self.B,), dtype=torch.int32, device=self.device)
            self.uncapped = self.meta[:self.B] if self.max_det is None else torch.zeros((self.B,), dtype=torch.int32, device=self.device)
            self.side = torch.cuda.Stream(device=self.device)
        self.graph = None
        # kernels launched per run(): per group flag + emit + segment NMS + fix-up (+ 1 memset node)
        self.launches_per_run = self.n_groups * 5

    def run(self, head_outputs):
        L, B, C, M = self.L, self.B, self.C, self.M
        raws, Bc, Fs, dt = _check_raws(head_outputs, C)  # shape / dtype / device checked, non-contiguous inputs copied
        if Bc != B or Fs != self.Fs:
            raise ValueError("shape mismatch with the configured postprocessor")
        self._live_inputs = raws                         # a contiguous copy must outlive the enqueued kernels
        rp = _cabi.ptrs([r.data_ptr() for r in raws])
        main = torch.cuda.current_stream(self.device)
        G = self.n_groups
        fold_reset = G == 1                              # one group: the flag kernel zeroes the counters itself
        if not fold_reset:
            _cabi.check(L.yl_post_reset(self.ws.ptr(), self.ws.nbytes, B, M, C, self.cap_seg, main.cuda_stream))
        for g in range(G):
            i0, i1 = B * g // G, B * (g + 1) // G
            _cabi.check(L.yl_filter_raw_ex(rp, dt, self.fs, len(self.Fs), B, C, self.anch, self.mask, self.conf, self._sxy,
                                           self.ws.ptr(), self.ws.nbytes, M, self.cap_seg, i0, i1 - i0, 7 if fold_reset else 3,
                                           main.cuda_stream))
            self.side.wait_stream(main)
            _cabi.check(L.yl_nms_ex2(self.ws.ptr(), self.ws.nbytes, B, M, C, self.cap_seg, self.nms, self.max_det or 0,
                                     int(self.agnostic), int(self.diou), self.rows.data_ptr(), self.cap_out, self.meta.data_ptr(),
                                     None if self.max_det is None else self.uncapped.data_ptr(), i0, i1 - i0, self.side.cuda_stream))
        main.wait_stream(self.side)
        return self.rows, self.meta

    def capture(self, head_outputs):
        raws, B, Fs, _ = _check_raws(head_outputs, self.C)
        if B != self.B or Fs != self.Fs:
            raise ValueError("shape mismatch with the configured postprocessor")
        self._captured_inputs = raws
        with torch.cuda.device(self.device):
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self.run(raws)                       # warm-up outside capture
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self.run(raws)
        return self

    def replay(self):
        self.graph.replay()
        return self.rows, self.meta

    def results(self):
        """Host-side view of the last run: list of [K_i,7] tensors / None (one D2H sync)."""
        mh = self.meta.cpu().numpy()
        if int(mh[self.B:2 * self.B].max()) > self.cap_seg or int(mh[:self.B].max()) > self.cap_out:
            raise _cabi.YoloHeadError("capacity exceeded (max segment %d / cap_seg %d, max rows %d / cap_out %d)" % (
                int(mh[self.B:2 * self.B].max()), self.cap_seg, int(mh[:self.B].max()), self.cap_out))
        return _split(self.rows, mh, self.B, self.device, torch.float32)
