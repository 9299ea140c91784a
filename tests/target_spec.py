"""YOLOLoss.build_target for one layer (yolo/model/yololoss.py:196-369) stated literally in NumPy: the reading the C oracle's
hand-written scatter and both CUDA paths (build_target, the fused loss) are checked against.

  nlabel       number of label rows whose sum (fp32, left to right) is > 0; the FIRST nlabel rows are used, zero rows and
               rows with a sum <= 0 among them included (:196-219)
  assignment   best anchor = first maximum of the nine (0, 0, w, h) IoUs, NaN counting as the maximum (torch.argmax); the GT
               belongs to the layer when the best anchor is in its mask; the anchor slot is best_n % 3, used as given for
               the cell and for the wh target's anchor (:249-265, :257)
  cell         i, j = int16 truncation of the grid-unit centre (:206-207), indexed with Python's rules
  scatter      one Python loop over the GTs in order, writing obj_mask / tgt_mask / tgt_scale / target[..., 0:5] and then
               target[b, a, j, i, 5 + cls] = 1 with cls the int16 truncation of the class id (:304-369): NumPy indexing
               gives the negative-index wrap, and raises IndexError exactly where the reference does
The arithmetic is the oracle's own (orc.logf, orc.bboxes_iou, fp32 NumPy operations), so results compare bit for bit.
"""
import numpy as np

from oracle import oracle as orc


def build_target(pred, labels, layer_no, n_classes, ignore_thre=0.7, anchors=orc.ANCHORS_PX, mask=orc.ANCHOR_MASK):
    """pred [B,3,F,F,4] fp32, labels [B,K,5] (xc, yc, w, h, cls) in pixels -> (target, obj_mask, tgt_mask, tgt_scale).
    Raises IndexError where the reference's indexing does."""
    pred = np.asarray(pred, np.float32)
    labels = np.asarray(labels, np.float32)
    B, _, F, _, _ = pred.shape
    nch = 5 + n_classes
    stride = np.float32(orc.STRIDES[layer_no])
    ref_anchors = np.zeros((9, 4), np.float32)                                       # :139-150
    ref_anchors[:, 2:] = np.array([[w / float(stride), h / float(stride)] for w, h in anchors], np.float64).astype(np.float32)
    masked = ref_anchors[mask[layer_no], 2:]
    target = np.zeros((B, 3, F, F, nch), np.float32)                                 # :156-167
    obj_mask = np.ones((B, 3, F, F), np.float32)
    tgt_mask = np.zeros((B, 3, F, F, 4 + n_classes), np.float32)
    tgt_scale = np.zeros((B, 3, F, F, 2), np.float32)

    s = labels[:, :, 0]
    for c in range(1, 5):
        s = s + labels[:, :, c]
    nlabel = (s > 0).sum(1)                                                          # :219
    tx, ty, tw, th = (labels[:, :, c] / stride for c in range(4))                    # :196-202
    with np.errstate(invalid="ignore"):
        ti_all, tj_all = tx.astype(np.int16), ty.astype(np.int16)                    # :206-207
    fF = np.float32(F)
    for b in range(B):
        n = int(nlabel[b])
        if n == 0:                                                                   # :225-227
            continue
        truth_box = np.zeros((n, 4), np.float32)
        truth_box[:, 2], truth_box[:, 3] = tw[b, :n], th[b, :n]
        best_n_all = np.argmax(orc.bboxes_iou(truth_box, ref_anchors, xyxy=True), axis=1)   # first max, NaN is the max
        best_n = best_n_all % 3
        in_layer = np.isin(best_n_all, mask[layer_no])
        truth_box[:, 0], truth_box[:, 1] = tx[b, :n], ty[b, :n]
        ious = orc.bboxes_iou(pred[b].reshape(-1, 4), truth_box, xyxy=False)         # :276-286
        best = np.max(ious, axis=1)                                                  # propagates NaN like torch.max
        obj_mask[b] = (~(best > np.float32(ignore_thre))).reshape(3, F, F).astype(np.float32)
        for t in range(n):                                                           # :304-369
            if not in_layer[t]:
                continue
            i, j, a = int(ti_all[b, t]), int(tj_all[b, t]), int(best_n[t])
            obj_mask[b, a, j, i] = 1
            tgt_mask[b, a, j, i, :] = 1
            with np.errstate(invalid="ignore"):
                tgt_scale[b, a, j, i, :] = np.sqrt(np.float32(2) - tw[b, t] * th[b, t] / fF / fF)
            target[b, a, j, i, 0] = tx[b, t] - np.float32(ti_all[b, t])
            target[b, a, j, i, 1] = ty[b, t] - np.float32(tj_all[b, t])
            target[b, a, j, i, 2] = orc.logf(tw[b, t] / masked[a, 0] + np.float32(1e-16))
            target[b, a, j, i, 3] = orc.logf(th[b, t] / masked[a, 1] + np.float32(1e-16))
            target[b, a, j, i, 4] = 1
            target[b, a, j, i, 5 + int(np.float32(labels[b, t, 4]).astype(np.int16))] = 1
    return target, obj_mask, tgt_mask, tgt_scale
