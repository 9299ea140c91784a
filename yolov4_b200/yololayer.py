"""YOLOLayer -- drop-in for yolo/model/yololayer.py (same constructor, attributes, forward outputs).

eval:  forward(x[B, 3*(5+C), F, F]) -> Tensor[B, 3*F*F, 5+C]                              (yololayer.py:146-166)
train: forward(x) -> {'layer_no', 'output': [B,3,F,F,5+C] view, 'pred': [B,3,F,F,4] view}   (yololayer.py:122-145)

The module has no parameters or buffers, exactly like the reference's (`masked_anchors` is a plain attribute),
so checkpoints load unchanged with strict=True (val.py:82-83).
"""
import numpy as np
import torch
from torch import nn

from . import _cabi
from .postprocess import _check_scale_x_y, _scale_value


def _stream():
    return torch.cuda.current_stream().cuda_stream


class _DecodeTrain(torch.autograd.Function):
    """`output` of the train branch stays differentiable w.r.t. the head conv output (yololoss.py:402-432
    back-propagates through it).  `pred` only feeds IoU comparisons in build_target and carries no gradient."""

    @staticmethod
    def forward(ctx, raw, anch, n_classes):
        raw = raw.contiguous()
        B, _, F, _ = raw.shape
        nch = 5 + n_classes
        out = torch.empty((B, 3, nch, F, F), dtype=raw.dtype, device=raw.device)
        pred = torch.empty((B, 3, 4, F, F), dtype=raw.dtype, device=raw.device)
        with torch.cuda.device(raw.device):
            _cabi.check(_cabi.lib().yl_decode_train(raw.data_ptr(), B, F, n_classes, anch, out.data_ptr(), pred.data_ptr(),
                                                    _stream()))
        # The RAW tensor is what the backward pass keeps, not `out`: the reference's YOLOLoss.forward multiplies
        # dict['output'] (a view of `out`) by its masks in place (yololoss.py:402-408), which would bump the version of a
        # saved `out` and make loss.backward() raise.  The backward kernel recomputes sigmoid(raw) (same bits).
        ctx.save_for_backward(raw)
        ctx.n_classes = n_classes
        ctx.mark_non_differentiable(pred)
        return out, pred

    @staticmethod
    def backward(ctx, grad_out, _grad_pred):
        (raw,) = ctx.saved_tensors
        B, _, F, _ = raw.shape
        nch = 5 + ctx.n_classes
        g = grad_out.contiguous()
        grad_raw = torch.empty_like(raw)
        with torch.cuda.device(raw.device):
            _cabi.check(_cabi.lib().yl_decode_train_backward_raw(raw.data_ptr(), g.data_ptr(), B, F, ctx.n_classes,
                                                                 grad_raw.data_ptr(), _stream()))
        return grad_raw, None, None


class YOLOLayer(nn.Module):
    strides = [8, 16, 32]

    def __init__(self, cfg, layer_no, device=None, *, scale_x_y=None):
        """scale_x_y (keyword only, not part of the reference signature): YOLOv4's grid-sensitivity decode of this head, one
        real number s (darknet's scale_x_y).  The eval output's centres become fl(fl(fl(fl(sigmoid(t) * s) + beta) + cell)
        * stride), beta = fl32(-0.5 * (s - 1)); None or 1 is the reference's decode, bit for bit.  The train branch feeds the
        reference's BCE loss, which has no scaled form: in training mode a scale other than 1 raises ValueError (train with
        fused_yolo_loss(..., iou_loss=..., scale_x_y=...)).  A plain attribute, so the state_dict stays empty."""
        super().__init__()
        self.scale_x_y = 1.0 if scale_x_y is None else _scale_value(scale_x_y)
        self.stride = self.strides[layer_no]
        self.layer_no = layer_no
        self.anchors = cfg['ANCHORS']
        self.anchor_mask = cfg['ANCHOR_MASK'][layer_no]
        self.n_anchors = len(self.anchor_mask)
        if self.n_anchors != 3:
            raise ValueError("libyolohead supports 3 anchors per scale (the reference's configs)")
        # yololayer.py:73-76: Python doubles, cast to the input dtype at use
        self.all_anchors_grid = [(w / self.stride, h / self.stride) for w, h in self.anchors]
        self.masked_anchors = [self.all_anchors_grid[i] for i in self.anchor_mask]
        self.masked_anchors = torch.from_numpy(np.array(self.masked_anchors))
        self.n_classes = cfg['N_CLASSES']
        self.device = device
        self._anch = _cabi.floats(self.masked_anchors.to(torch.float32).reshape(-1).tolist())

    def forward(self, output):
        if output.dim() != 4 or output.shape[1] != self.n_anchors * (5 + self.n_classes) or output.shape[2] != output.shape[3]:
            raise ValueError("expected [B, %d, F, F], got %s" % (self.n_anchors * (5 + self.n_classes), tuple(output.shape)))
        if not output.is_cuda or output.dtype != torch.float32:
            raise TypeError("YOLOLayer (B200) needs a float32 CUDA tensor; there is no CPU fallback")
        B, _, F, _ = output.shape
        n_ch = 5 + self.n_classes
        if self.training:
            if self.scale_x_y != 1.0:
                raise ValueError("YOLOLayer with scale_x_y=%r has no train branch (the reference's BCE xy loss has no scaled "
                                 "form): train with fused_yolo_loss(..., iou_loss=..., scale_x_y=...)" % (self.scale_x_y,))
            out_planar, pred_planar = _DecodeTrain.apply(output, self._anch, self.n_classes)
            return dict({
                'layer_no': self.layer_no,
                'output': out_planar.permute(0, 1, 3, 4, 2),     # strides (255F^2, 85F^2, F, 1, F^2) as in the reference
                'pred': pred_planar.permute(0, 1, 3, 4, 2),
            })
        raw = output.detach().contiguous()
        res = torch.empty((B, self.n_anchors * F * F, n_ch), dtype=raw.dtype, device=raw.device)
        with torch.cuda.device(raw.device):
            _cabi.check(_cabi.lib().yl_decode_dense_ex(raw.data_ptr(), B, F, self.n_classes, self._anch, float(self.stride),
                                                       self.scale_x_y, res.data_ptr(), self.n_anchors * F * F, 0, _stream()))
        return res


def decode_dense_cat(head_outputs, cfg, *, scale_x_y=None):
    """The three eval-mode YOLOLayer outputs written straight into one [B, sum 3F^2, 5+C] tensor: the value of
    `torch.cat((x1, x2, x3), 1)` at yolov4.py:324 without the three intermediate tensors and the cat copy.
    scale_x_y: None, one real number or one per head tensor in head order, the grid-sensitivity decode of
    YOLOLayer(..., scale_x_y=s) (detect_raw states it); checked before any CUDA work."""
    sxy = _check_scale_x_y(scale_x_y, len(head_outputs)) or [1.0] * len(head_outputs)
    C = int(cfg['N_CLASSES'])
    B = int(head_outputs[0].shape[0])
    Fs = [int(r.shape[2]) for r in head_outputs]
    M = sum(3 * f * f for f in Fs)
    dev = head_outputs[0].device
    out = torch.empty((B, M, 5 + C), dtype=torch.float32, device=dev)
    off = 0
    with torch.cuda.device(dev):
        for l, r in enumerate(head_outputs):
            if not r.is_cuda or r.dtype != torch.float32 or r.shape[1] != 3 * (5 + C):
                raise TypeError("head tensors must be float32 CUDA tensors [B, 3*(5+C), F, F]")
            s = YOLOLayer.strides[l]
            anch = _cabi.floats([v / s for i in cfg['ANCHOR_MASK'][l] for v in cfg['ANCHORS'][i]])
            raw = r.detach().contiguous()
            _cabi.check(_cabi.lib().yl_decode_dense_ex(raw.data_ptr(), B, Fs[l], C, anch, float(s), sxy[l], out.data_ptr(), M, off,
                                                       _stream()))
            off += 3 * Fs[l] * Fs[l]
    return out
