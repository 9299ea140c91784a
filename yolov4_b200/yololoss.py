"""YOLOLoss -- drop-in for yolo/model/yololoss.py: build_target runs in libyolohead.so (yl_build_target).

build_target(output, pred, layer_no, labels) -> (target, obj_mask, tgt_mask, tgt_scale)      (yololoss.py:118-371)
forward(outputs, targets) restates the reference's loss arithmetic (yololoss.py:373-443) in plain torch so the
class can replace the reference's criterion as a whole, dense tensors and all.
fused_yolo_loss(head_outputs, padded_labels, cfg, ignore_thresh) is SURVEY.md's "next" row N2: the same loss value and
its gradient with respect to the raw head tensors from yl_loss_forward / yl_loss_backward, without materialising
output / pred / target / masks; the padded labels are cast and uploaded once for the three scales (row N4).  The fused loss
also takes fp16 / bf16 head tensors (autocast, apex O1/O2): widened exactly to fp32 inside the kernels, gradients in the
head's dtype.
"""
import numpy as np
import torch
from torch import nn

from . import _cabi
from .postprocess import _check_scale_x_y


def _stream():
    return torch.cuda.current_stream().cuda_stream


# head tensor dtypes of the fused loss -> YL_DTYPE_* (include/yolo_head.h)
_DTYPE_CODES = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}


def _head_dtype_code(raws):
    """YL_DTYPE_* of the fused loss's head tensors: float32, float16 or bfloat16 CUDA tensors, all of one dtype.  Raises
    TypeError before any CUDA work."""
    for r in raws:
        if not isinstance(r, torch.Tensor) or not r.is_cuda or r.dtype not in _DTYPE_CODES:
            raise TypeError("fused YOLO loss needs float32, float16 or bfloat16 CUDA head tensors; there is no CPU fallback")
        if r.dtype != raws[0].dtype:
            raise TypeError("fused YOLO loss head tensors must share one dtype, got %s and %s" % (raws[0].dtype, r.dtype))
    return _DTYPE_CODES[raws[0].dtype]


class _LabelUploader:
    """N4 (SURVEY.md 8f): the padded labels [B,K,5] of a step (float64 on the host as the loader collates them,
    yolo/data/transform.py:464-471) are cast to fp32 once on the host, staged in pinned memory and uploaded with ONE
    asynchronous copy that the three scales share -- the reference clones, uploads and casts them once per layer
    (yololoss.py:392, :129).  One staging buffer per (shape, device); an event guards its reuse."""

    _stage = {}

    @classmethod
    def upload(cls, labels, device):
        device = torch.device(device)
        if labels.is_cuda:
            return labels.to(device=device, dtype=torch.float32).contiguous()
        key = (tuple(labels.shape), str(device))
        ent = cls._stage.get(key)
        if ent is None:
            ent = cls._stage[key] = [torch.empty(tuple(labels.shape), dtype=torch.float32).pin_memory(), None]
        buf, ev = ent
        if ev is not None:
            ev.synchronize()                       # the previous step's copy out of this buffer has finished
        buf.copy_(labels)                          # host cast float64 -> fp32 (the value yololoss.py:129 computes)
        with torch.cuda.device(device):
            dev = buf.to(device, non_blocking=True)
            ent[1] = torch.cuda.Event()
            ent[1].record()
        return dev


def upload_labels(labels, device):
    """One pinned fp32 upload of the padded labels, to be shared by the three scales (row N4)."""
    return _LabelUploader.upload(labels, device)


def build_target(output, pred, layer_no, labels, anchors, anchor_mask, ignore_thresh, n_classes, strict=False):
    """Functional form.  output: only shape/dtype/device are used (as in the reference); pred [B,3,F,F,4] any strides;
    labels [B,K,5] (xc,yc,w,h,cls) in input pixels, zero padded, any float dtype (cast to fp32 like yololoss.py:129).
    strict=True synchronises and raises IndexError when a matched GT falls outside the grid, as the reference does."""
    if not pred.is_cuda or pred.dtype != torch.float32:
        raise TypeError("build_target (B200) needs float32 CUDA tensors; there is no CPU fallback")
    B, A, F = int(output.shape[0]), int(output.shape[1]), int(output.shape[2])
    n_ch = 5 + n_classes
    assert output.shape[-1] == n_ch and A == 3
    dev = pred.device
    lab = upload_labels(labels, dev)
    K = int(lab.shape[1])
    target = torch.empty((B, 3, F, F, n_ch), dtype=torch.float32, device=dev)
    obj_mask = torch.empty((B, 3, F, F), dtype=torch.float32, device=dev)
    tgt_mask = torch.empty((B, 3, F, F, 4 + n_classes), dtype=torch.float32, device=dev)
    tgt_scale = torch.empty((B, 3, F, F, 2), dtype=torch.float32, device=dev)
    status = torch.empty((1,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().yl_build_target(
            pred.data_ptr(), _cabi.longs(pred.stride()), lab.data_ptr(), B, F, K, n_classes, int(layer_no),
            _cabi.floats([v for wh in anchors for v in wh]), _cabi.ints(anchor_mask[layer_no]),
            float(np.float32(ignore_thresh)), target.data_ptr(), obj_mask.data_ptr(), tgt_mask.data_ptr(),
            tgt_scale.data_ptr(), status.data_ptr(), _stream()))
    if strict and int(status.item()) != 0:
        raise IndexError("a matched ground-truth box indexes outside the %dx%d grid" % (F, F))
    return target, obj_mask, tgt_mask, tgt_scale


def build_targets3(outputs, preds, layer_nos, labels, anchors, anchor_mask, ignore_thresh, n_classes):
    """build_target for up to three scales with ONE pair of launches (yl_build_target3): the list of
    (target, obj_mask, tgt_mask, tgt_scale) tuples that per-layer build_target calls return, bit for bit.  This is the form
    YOLOLoss.forward uses; the per-layer method stays for callers of the reference's own API (yololoss.py:393)."""
    if not 1 <= len(preds) <= 3 or len(outputs) != len(preds) or len(layer_nos) != len(preds):
        raise ValueError("1..3 scales, one output / pred / layer number each")
    dev = preds[0].device
    n_ch = 5 + n_classes
    lab = upload_labels(labels, dev)
    B, K = int(lab.shape[0]), int(lab.shape[1])
    res, Fs, strides_all = [], [], []
    for o, p in zip(outputs, preds):
        if not p.is_cuda or p.dtype != torch.float32 or p.device != dev:
            raise TypeError("build_target (B200) needs float32 CUDA tensors on one device; there is no CPU fallback")
        F = int(o.shape[2])
        assert o.shape[-1] == n_ch and int(o.shape[1]) == 3 and int(o.shape[0]) == B
        res.append((torch.empty((B, 3, F, F, n_ch), dtype=torch.float32, device=dev),
                    torch.empty((B, 3, F, F), dtype=torch.float32, device=dev),
                    torch.empty((B, 3, F, F, 4 + n_classes), dtype=torch.float32, device=dev),
                    torch.empty((B, 3, F, F, 2), dtype=torch.float32, device=dev)))
        Fs.append(F)
        strides_all += list(p.stride())
    status = torch.empty((1,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().yl_build_target3(
            _cabi.ptrs([p.data_ptr() for p in preds]), _cabi.longs(strides_all), lab.data_ptr(), B, _cabi.ints(Fs), K, n_classes,
            len(preds), _cabi.ints(layer_nos), _cabi.floats([v for wh in anchors for v in wh]),
            _cabi.ints([v for m in anchor_mask for v in m]), float(np.float32(ignore_thresh)),
            _cabi.ptrs([r[0].data_ptr() for r in res]), _cabi.ptrs([r[1].data_ptr() for r in res]),
            _cabi.ptrs([r[2].data_ptr() for r in res]), _cabi.ptrs([r[3].data_ptr() for r in res]), status.data_ptr(), _stream()))
    return res


class YOLOLoss(nn.Module):
    strides = [8, 16, 32]

    def __init__(self, cfg, ignore_thresh=0.7, device=None):
        super().__init__()
        self.cfg = cfg
        self.ignore_thresh = ignore_thresh
        self.device = device
        self.anchors = cfg['ANCHORS']
        self.n_classes = cfg['N_CLASSES']
        self.l2_loss = nn.MSELoss(reduction="sum").to(device)
        self.bce_loss = nn.BCELoss(reduction="sum").to(device)

    def build_target(self, output, pred, layer_no, labels):
        # side-effect attributes of the reference (yololoss.py:133-150); nothing reads them afterwards
        self.anch_mask = self.cfg['ANCHOR_MASK'][layer_no]
        self.n_anchors = len(self.anch_mask)
        self.stride = self.strides[layer_no]
        self.all_anchors_grid = [(w / self.stride, h / self.stride) for w, h in self.anchors]
        self.masked_anchors = [self.all_anchors_grid[i] for i in self.anch_mask]
        return build_target(output, pred, layer_no, labels, self.anchors, self.cfg['ANCHOR_MASK'], self.ignore_thresh,
                            self.n_classes)

    def forward(self, outputs, targets):
        assert isinstance(outputs, list) and isinstance(targets, dict)
        total = 0
        outs = [od['output'].to(self.device) for od in outputs]
        preds = [od['pred'].to(self.device) for od in outputs]
        layer_nos = [int(od['layer_no']) for od in outputs]
        labels = upload_labels(targets['padded_labels'], preds[0].device)          # once for the three layers (N4)
        if 1 <= len(outputs) <= 3:
            # one pair of launches for all scales (the reference loops: yololoss.py:381-393); same tensors, bit for bit
            built = build_targets3(outs, preds, layer_nos, labels, self.anchors, self.cfg['ANCHOR_MASK'], self.ignore_thresh,
                                   self.n_classes)
        else:
            built = [self.build_target(o, p, l, labels) for o, p, l in zip(outs, preds, layer_nos)]
        for output, (target, obj_mask, tgt_mask, tgt_scale) in zip(outs, built):
            n_ch = output.shape[-1]
            sel = np.r_[0:4, 5:n_ch]
            # yololoss.py:402-414 (written out of place; same values)
            out_m = output.clone()
            out_m[..., 4] = output[..., 4] * obj_mask
            out_m[..., sel] = output[..., sel] * tgt_mask
            out_m[..., 2:4] = out_m[..., 2:4] * tgt_scale
            target[..., 4] *= obj_mask
            target[..., sel] *= tgt_mask
            target[..., 2:4] *= tgt_scale
            bce_w = nn.BCELoss(weight=tgt_scale * tgt_scale, reduction="sum")
            loss_xy = bce_w(out_m[..., :2], target[..., :2])
            loss_wh = self.l2_loss(out_m[..., 2:4], target[..., 2:4]) / 2
            loss_obj = self.bce_loss(out_m[..., 4], target[..., 4])
            loss_cls = self.bce_loss(out_m[..., 5:], target[..., 5:])
            total = total + loss_xy + loss_wh + loss_obj + loss_cls
        return total


# iou_loss= of the fused loss -> YL_IOU_LOSS_* (include/yolo_head.h)
_IOU_LOSS_CODES = {None: 0, "giou": 1, "diou": 2, "ciou": 3}


def _iou_args(iou_loss, iou_normalizer):
    """(YL_IOU_LOSS_* code, fp32 normalizer) of the fused loss's box-term keywords; raises before any CUDA work."""
    if not (iou_loss is None or isinstance(iou_loss, str)) or iou_loss not in _IOU_LOSS_CODES:
        raise ValueError("iou_loss must be None, 'giou', 'diou' or 'ciou', got %r" % (iou_loss,))
    if isinstance(iou_normalizer, (bool, np.bool_)) or not isinstance(iou_normalizer, (int, float, np.integer, np.floating)):
        raise TypeError("iou_normalizer must be a real number, got %r" % (iou_normalizer,))
    norm = float(iou_normalizer)
    if not np.isfinite(norm) or norm < 0.0 or norm > float(np.finfo(np.float32).max):
        raise ValueError("iou_normalizer must be finite and >= 0, got %r" % (iou_normalizer,))
    if iou_loss is None and norm != 1.0:
        raise ValueError("iou_normalizer weights the IoU box term only: it needs iou_loss='giou', 'diou' or 'ciou'")
    return _IOU_LOSS_CODES[iou_loss], float(np.float32(norm))


def _scale_args(scale_x_y, n_heads, iou_code):
    """One fp32 scale_x_y per head tensor (all 1.0 without scales); raises before any CUDA work."""
    sxy = _check_scale_x_y(scale_x_y, n_heads)
    if sxy is not None and iou_code == 0:
        raise ValueError("scale_x_y moves the predicted centre of the IoU box term: it needs iou_loss='giou', 'diou' or 'ciou' "
                         "(the BCE xy term has no scaled form)")
    return sxy or [1.0] * n_heads


class _FusedYoloLoss(torch.autograd.Function):
    """N2: raw head tensors + padded labels -> the reference's YOLOLoss.forward value, gradient straight to the raw tensors
    (in the heads' dtype: fp32, fp16 or bf16)."""

    @staticmethod
    def forward(ctx, labels, anchors, anchor_mask, ignore_thresh, n_classes, iou_code, iou_norm, sxy, *raws):
        L = _cabi.lib()
        C = int(n_classes)
        dtype = _head_dtype_code(raws)
        for r in raws:
            if r.dim() != 4 or r.shape[1] != 3 * (5 + C) or r.shape[0] != labels.shape[0]:
                raise TypeError("fused YOLO loss needs CUDA head tensors [B, 3*(5+C), F, F]; there is no CPU fallback")
        dev = raws[0].device
        lab = upload_labels(labels, dev)
        B, K = int(lab.shape[0]), int(lab.shape[1])
        anch = _cabi.floats([v for wh in anchors for v in wh])
        saved, keep = [], []
        with torch.cuda.device(dev):
            loss4 = torch.zeros(4, dtype=torch.float64, device=dev)
            status = torch.zeros(1, dtype=torch.int32, device=dev)
            calls = []
            for l, r in enumerate(raws):
                rc = r.detach().contiguous()
                F = int(rc.shape[2])
                gobj = torch.empty((B, 3, F, F), dtype=torch.float32, device=dev)
                tcell = torch.empty((B, K), dtype=torch.int32, device=dev)
                mcell = torch.empty((B, K), dtype=torch.int32, device=dev)
                mgrad = torch.empty((B, K, 4 + C), dtype=torch.float32, device=dev)
                calls.append((rc, F, l, gobj, tcell, mcell, mgrad))
                saved += [gobj, mcell, mgrad]
                keep += [rc, tcell]         # see yl_loss_forward: the scales' kernels overlap, their buffers must not alias
            # every foreign kernel (contiguous copies, the fills of loss4 / status) is enqueued by now: the calls below are back
            # to back on the stream, so the second and later ones may be launched programmatically behind their predecessor
            for i, (rc, F, l, gobj, tcell, mcell, mgrad) in enumerate(calls):
                _cabi.check(L.yl_loss_forward_ex2(rc.data_ptr(), dtype, lab.data_ptr(), B, F, K, C, l, anch,
                                                  _cabi.ints(anchor_mask[l]), float(np.float32(ignore_thresh)), iou_code,
                                                  iou_norm, sxy[i], int(i > 0), loss4.data_ptr(), gobj.data_ptr(), tcell.data_ptr(),
                                                  mcell.data_ptr(), mgrad.data_ptr(), status.data_ptr(), _stream()))
        ctx.save_for_backward(*saved)
        ctx.shapes = [tuple(r.shape) for r in raws]
        ctx.dtype, ctx.dtype_code = raws[0].dtype, dtype
        ctx.K, ctx.C = K, C
        ctx.status = status
        ctx.loss4 = loss4
        return loss4.sum().to(torch.float32)          # the reference returns a float32 scalar

    @staticmethod
    def backward(ctx, grad_out):
        L = _cabi.lib()
        saved = ctx.saved_tensors
        up = grad_out.detach().to(torch.float32).reshape(1).contiguous()
        grads = []
        with torch.cuda.device(up.device):
            for l, shp in enumerate(ctx.shapes):
                gobj, mcell, mgrad = saved[3 * l:3 * l + 3]
                B, _, F, _ = shp
                g = torch.empty(shp, dtype=ctx.dtype, device=up.device)        # written in the head's dtype, no fp32 copy
                _cabi.check(L.yl_loss_backward_typed(gobj.data_ptr(), mcell.data_ptr(), mgrad.data_ptr(), up.data_ptr(), B, F, ctx.K,
                                                     ctx.C, g.data_ptr(), ctx.dtype_code, _stream()))
                grads.append(g)
        return (None, None, None, None, None, None, None, None) + tuple(grads)


def fused_yolo_loss(head_outputs, padded_labels, cfg, ignore_thresh=0.7, iou_loss=None, iou_normalizer=1.0, scale_x_y=None):
    """N2 (SURVEY.md 8f): the value of `YOLOLoss(cfg, ignore_thresh)([YOLOLayer_l.train()(x_l)], {'padded_labels': labels})`
    (yolo/model/yololoss.py:373-443 on top of yololayer.py:122-145) computed from the three raw head tensors without
    materialising output / pred / target / masks; differentiable with respect to the head tensors.
    Loss and gradient agree with the reference within 1e-5 / 2e-5 relative (not bit-exact: reduction order).

    The heads may be float32, float16 or bfloat16 CUDA tensors of one dtype (a model under torch.autocast or apex O1/O2); the
    loss is always a float32 scalar.  A 16-bit head is widened exactly to fp32 inside the kernels, so the loss is that of
    `[h.float() for h in head_outputs]` up to the order of the fp64 sums, and its gradient has the head's dtype: bit for bit
    the fp32 path's gradient on the widened heads (with the same upstream gradient, e.g. a GradScaler's scale) rounded to
    nearest-even, overflow to +-inf included.  This is not the reference's own half-precision arithmetic.  Mixed dtypes,
    float64 and CPU heads raise TypeError before any CUDA work.

    iou_loss='giou' / 'diou' / 'ciou' (YOLOv4's CIoU box regression, darknet's iou_loss option) replaces the xy BCE and wh MSE
    of every matched cell by iou_normalizer * torchvision's generalized_ / distance_ / complete_box_iou_loss (eps 1e-7) of the
    train-mode predicted box and the cell's last GT, in grid units, without tgt_scale weighting; objectness and class terms
    are unchanged (DESIGN.md section 1).  iou_normalizer (a finite real >= 0) weights the box term only; with iou_loss=None
    it must stay 1.  A bad keyword raises ValueError (TypeError for a bool normalizer) before any CUDA work.

    scale_x_y (YOLOv4's grid-sensitivity decode, darknet's scale_x_y; yolov4.cfg pairs 1.2 / 1.1 / 1.05 with iou_loss='ciou'):
    None, one real number for every head, or one per head tensor in head order.  The train-mode predicted box of the IoU box
    term and of the ignore test takes the centre fl(fl(fl(sigmoid(t) * s) + beta) + cell), beta = fl32(-0.5 * (s - 1)), and
    d centre / d t = s * sigmoid * (1 - sigmoid); w / h, objectness and class terms are unchanged.  None or all ones is the
    loss without it, bit for bit.  A scale other than 1 needs an IoU box term (iou_loss=None raises ValueError: the BCE xy
    term has no scaled form); a bool or non-real raises TypeError, a non-finite or non-positive value or a wrong length
    ValueError, before any CUDA work."""
    iou_code, iou_norm = _iou_args(iou_loss, iou_normalizer)
    sxy = _scale_args(scale_x_y, len(head_outputs), iou_code)
    return _FusedYoloLoss.apply(padded_labels, cfg['ANCHORS'], cfg['ANCHOR_MASK'], ignore_thresh, cfg['N_CLASSES'], iou_code,
                                iou_norm, sxy, *head_outputs)


def fused_yolo_loss_components(head_outputs, padded_labels, cfg, ignore_thresh=0.7, layers=None, iou_loss=None,
                               iou_normalizer=1.0, scale_x_y=None):
    """The four sums (loss_xy, loss_wh, loss_obj, loss_cls; yololoss.py:421-427) over the given layers as a float64[4] device
    tensor, no autograd.  `layers[i]` is the layer number of head_outputs[i] (default 0, 1, 2).  The heads may be float32,
    float16 or bfloat16 CUDA tensors of one dtype: a 16-bit head gives the components of its widened fp32 copy (up to the order
    of the fp64 sums); mixed dtypes, float64 and CPU heads raise TypeError before any CUDA work.  iou_loss / iou_normalizer as
    for fused_yolo_loss: with an IoU box term, component 0 is that term and component 1 is 0.  scale_x_y as for
    fused_yolo_loss, one value per head tensor (not per layer number)."""
    iou_code, iou_norm = _iou_args(iou_loss, iou_normalizer)
    sxy = _scale_args(scale_x_y, len(head_outputs), iou_code)
    L = _cabi.lib()
    dtype = _head_dtype_code(head_outputs)
    dev = head_outputs[0].device
    lab = upload_labels(padded_labels, dev)
    B, K = int(lab.shape[0]), int(lab.shape[1])
    C = int(cfg['N_CLASSES'])
    anch = _cabi.floats([v for wh in cfg['ANCHORS'] for v in wh])
    layers = list(range(len(head_outputs))) if layers is None else layers
    keep = []                   # the scales' kernels overlap on the device (yl_loss_forward): no buffer is reused between them
    with torch.cuda.device(dev):
        loss4 = torch.zeros(4, dtype=torch.float64, device=dev)
        calls = []
        for l, r in zip(layers, head_outputs):
            rc = r.detach().contiguous()
            F = int(rc.shape[2])
            gobj = torch.empty((B, 3, F, F), dtype=torch.float32, device=dev)
            tcell = torch.empty((B, K), dtype=torch.int32, device=dev)
            mcell = torch.empty((B, K), dtype=torch.int32, device=dev)
            mgrad = torch.empty((B, K, 4 + C), dtype=torch.float32, device=dev)
            calls.append((rc, F, int(l), gobj, tcell, mcell, mgrad))
            keep += [rc, gobj, tcell, mcell, mgrad]
        for i, (rc, F, l, gobj, tcell, mcell, mgrad) in enumerate(calls):     # back to back: see _FusedYoloLoss.forward
            _cabi.check(L.yl_loss_forward_ex2(rc.data_ptr(), dtype, lab.data_ptr(), B, F, K, C, l, anch,
                                              _cabi.ints(cfg['ANCHOR_MASK'][l]), float(np.float32(ignore_thresh)), iou_code,
                                              iou_norm, sxy[i], int(i > 0), loss4.data_ptr(), gobj.data_ptr(), tcell.data_ptr(),
                                              mcell.data_ptr(), mgrad.data_ptr(), None, _stream()))
    return loss4
