"""YOLOv4's grid-sensitivity decode (`scale_x_y=`) stated in NumPy from the oracle's fp32 spec math (DESIGN.md section 1):

  beta             fl32(-0.5 * (s - 1)) evaluated in float64 from the fp32 s (darknet's scal_add bias)
  centre           fl(fl(fl(sigmoid(t) * s) + beta) + cell), each step one fp32 rounding
  decode_eval      orc.decode_eval with the scaled centres: bx = fl(cx * stride); w, h, objectness and classes unchanged
  decode_train     orc.decode_train with the scaled centres in `pred` (grid units); `output` unchanged
  layer_spec       one layer of the fused loss with an IoU box term: iou_loss_spec.layer_spec on the scaled `pred`, with the
                   ignore mask of orc.build_target on that `pred`, and d px / d tx = s sigmoid (1 - sigmoid)
  obj_grad_fp32    the objectness gradient plane as the kernel forms it in fp32 (bit for bit)
"""
import numpy as np

import iou_loss_spec
from oracle import oracle as orc

f32 = np.float32


def beta(s):
    return f32(-0.5 * (float(f32(s)) - 1.0))


def centre(t, cell, s):
    """fl(fl(fl(sigmoid(t) * s) + beta) + cell) of fp32 logits t and integer cells (broadcast)."""
    s = f32(s)
    with np.errstate(all="ignore"):
        return ((orc.sigmoidf(t) * s).astype(f32) + beta(s)).astype(f32) + np.asarray(cell).astype(f32)


def _grid(F):
    j, i = np.meshgrid(np.arange(F), np.arange(F), indexing="ij")
    return i, j


def decode_eval(raw, layer_no, C, s, anchors=orc.ANCHORS_PX, mask=orc.ANCHOR_MASK):
    """raw [B, 3(5+C), F, F] -> [B, 3F^2, 5+C] of YOLOLayer(..., scale_x_y=s) in eval mode."""
    raw = np.ascontiguousarray(raw, f32)
    out = orc.decode_eval(raw, layer_no, C, anchors, mask)
    B, _, F, _ = raw.shape
    i, j = _grid(F)
    stride = f32(orc.STRIDES[layer_no])
    nch = 5 + C
    for a in range(3):
        rows = slice(a * F * F, (a + 1) * F * F)
        with np.errstate(all="ignore"):
            out[:, rows, 0] = (centre(raw[:, a * nch], i, s) * stride).reshape(B, -1)
            out[:, rows, 1] = (centre(raw[:, a * nch + 1], j, s) * stride).reshape(B, -1)
    return out


def decode_eval_cat(raws, C, scales, anchors=orc.ANCHORS_PX, mask=orc.ANCHOR_MASK):
    return np.concatenate([decode_eval(r, l, C, scales[l], anchors, mask) for l, r in enumerate(raws)], axis=1)


def decode_train(raw, layer_no, C, s, anchors=orc.ANCHORS_PX, mask=orc.ANCHOR_MASK):
    """(output [B,3,F,F,5+C], pred [B,3,F,F,4]) with the scaled centres in pred (grid units)."""
    raw = np.ascontiguousarray(raw, f32)
    output, pred = orc.decode_train(raw, layer_no, C, anchors, mask)
    pred = np.array(pred)
    F = raw.shape[2]
    i, j = _grid(F)
    nch = 5 + C
    for a in range(3):
        pred[:, a, :, :, 0] = centre(raw[:, a * nch], i, s)
        pred[:, a, :, :, 1] = centre(raw[:, a * nch + 1], j, s)
    return output, pred


def matched_pairs(raw, labels, layer_no, C, s, anchors=orc.ANCHORS_PX, mask=orc.ANCHOR_MASK):
    """iou_loss_spec.matched_pairs with the scaled train-mode box p."""
    output, pred = decode_train(raw, layer_no, C, s, anchors, mask)
    owner = iou_loss_spec.last_gt_per_cell(labels, layer_no, pred.shape[2], anchors, mask)
    cells = np.array(sorted(owner), np.int64).reshape(-1, 4)
    tb = (np.asarray(labels, f32)[..., :4] / f32(orc.STRIDES[layer_no])).astype(f32)
    p = np.array([pred[b, a, j, i] for b, a, j, i in cells], f32).reshape(-1, 4)
    g = np.array([tb[b, owner[(b, a, j, i)]] for b, a, j, i in cells], f32).reshape(-1, 4)
    sg = np.array([output[b, a, j, i, :2] for b, a, j, i in cells], f32).reshape(-1, 2)
    return cells, p, g, sg


def raw_chain(dp, p, sg, s):
    """d / d p -> d / d raw with the scale: s sigmoid (1 - sigmoid) for x, y, pw, ph for w, h (float64)."""
    return iou_loss_spec.raw_chain(dp, p, sg) * np.array([float(f32(s)), float(f32(s)), 1.0, 1.0])


def raw_grad_fp32(kind, p, g, sg, s, norm=1.0):
    """The kernel's mgrad[..., 0:4]: fp32 ((n d) * s) * sigmoid * (1 - sigmoid) for x, y; (n d) * pw, ph for w, h."""
    _, d = iou_loss_spec.box_loss_fp32(kind, p, g)
    with np.errstate(all="ignore"):
        dn = d * f32(norm)
        sg = np.asarray(sg, f32)
        out = np.empty_like(dn)
        out[:, :2] = ((dn[:, :2] * f32(s)) * sg) * (f32(1) - sg)
        out[:, 2:] = dn[:, 2:] * np.asarray(p, f32)[:, 2:]
    return out


def obj_grad_fp32(raw, labels, layer_no, C, thr, s, anchors=orc.ANCHORS_PX, mask=orc.ANCHOR_MASK):
    """(objectness component float64, d loss / d raw objectness [B, 3, F, F] fp32 as k_loss_obj forms it): the ignore mask is
    orc.build_target's on the scaled pred; matched cells have target 1 and are never ignored."""
    output, pred = decode_train(raw, layer_no, C, s, anchors, mask)
    target, obj_mask, _, _ = orc.build_target(pred, np.asarray(labels, f32), layer_no, C, thr, anchors, mask)
    x = np.ascontiguousarray(output[..., 4], f32)
    t = (target[..., 4] * obj_mask).astype(f32)
    keep = obj_mask != 0
    one = f32(1)
    with np.errstate(all="ignore"):
        g = ((x - t) / np.maximum((one - x) * x, f32(1e-12))).astype(f32)
        g = ((g * x) * (one - x)).astype(f32)
        lx = np.maximum(np.log(x), f32(-100)).astype(np.float64)
        l1x = np.maximum(np.log(one - x), f32(-100)).astype(np.float64)
    g = np.where(keep, g, f32(0)).astype(f32)
    term = np.where(keep, np.where(t == 1, -lx, -l1x), 0.0)
    return term.sum(), g, obj_mask


def layer_spec(raw, labels, layer_no, C, thr, kind, s, norm=1.0, anchors=orc.ANCHORS_PX, mask=orc.ANCHOR_MASK):
    """One layer with the scale: (components float64 [4], per-cell (cells, term, d term / d raw, p), objectness gradient
    plane fp32 [B, 3, F, F], obj_mask).  Components 1 and 3 are iou_loss_spec.layer_spec's (0 and the class term, which does
    not depend on the box); 0 is the IoU term of the scaled p, 2 the objectness term under the scaled ignore mask."""
    comps, _, _ = iou_loss_spec.layer_spec(raw, labels, layer_no, C, thr, kind, norm, anchors, mask)
    cells, p, g, sg = matched_pairs(raw, labels, layer_no, C, s, anchors, mask)
    term, dp = iou_loss_spec.box_loss(kind, p, g)
    with np.errstate(invalid="ignore", over="ignore"):
        graw = norm * raw_chain(dp, p, sg, s)
    obj, gobj, obj_mask = obj_grad_fp32(raw, labels, layer_no, C, thr, s, anchors, mask)
    comps = np.array([norm * term.sum(), 0.0, obj, comps[3]])
    return comps, (cells, norm * term, graw, p, g, sg), gobj, obj_mask
