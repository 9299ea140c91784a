"""Class-agnostic NMS stated in NumPy: the literal algorithm the library's agnostic mode is checked against.

The candidates of an image are the (box, class) pairs the reference's filter emits (utils.py:117-184, restated operation for
operation in fp32 as oracle/yolo_head_oracle.c does), s = fl32(obj_conf * cls_conf) with -0 == +0.
  order        s descending, then class ascending, then box row descending
  suppression  walking that order, a candidate is dropped when IoU >= thr with any earlier kept candidate, whatever either
               class is; IoU is the literal NaN-propagating fp32 formula of utils.py:71-77
  output       the kept candidates as 7-float rows (x1, y1, x2, y2, obj_conf, cls_conf, cls), classes ascending, then s
               descending, then row descending
Greedy runs over ALL candidates: the first-copy reduction the CUDA kernel relies on is checked against this, not assumed.
"""
import numpy as np

from oracle import oracle as orc


def candidates(pred, num_classes, conf_thre):
    """pred [M, 5+C] decoded (cx, cy, w, h, obj, cls...) of one image -> dict of per-candidate arrays in the filter's order
    (box ascending, class ascending): box [n,4] xyxy, obj, conf, cls, row, s."""
    pred = np.asarray(pred, dtype=np.float32)
    C = pred.shape[1] - 5
    conf = np.float32(conf_thre)
    obj = pred[:, 4]
    with np.errstate(invalid="ignore", over="ignore"):
        mx = np.max(pred[:, 5:5 + num_classes], axis=1)           # torch.max propagates NaN (utils.py:139-141)
        pre = obj * mx >= conf                                     # utils.py:145-148
        ok = (pred[:, 5:] * obj[:, None] >= conf) & pre[:, None]   # utils.py:170
    row, cls = np.nonzero(ok)
    p = pred[row]
    hw, hh = p[:, 2] / np.float32(2), p[:, 3] / np.float32(2)      # utils.py:117-126
    with np.errstate(invalid="ignore", over="ignore"):
        box = np.stack([p[:, 0] - hw, p[:, 1] - hh, p[:, 0] + hw, p[:, 1] + hh], 1).astype(np.float32)
        s = (p[:, 4] * pred[row, 5 + cls]).astype(np.float32)
    return {"box": box, "obj": p[:, 4].copy(), "conf": pred[row, 5 + cls].copy(), "cls": cls.astype(np.int64),
            "row": row.astype(np.int64), "s": s}


def iou_ge(box_i, area_i, boxes, areas, thr):
    """The literal decision IoU(i, k) >= thr of utils.py:71-77 for one box against many, fp32, NaN-propagating."""
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        tlx = np.maximum(box_i[0], boxes[:, 0])
        tly = np.maximum(box_i[1], boxes[:, 1])
        brx = np.minimum(box_i[2], boxes[:, 2])
        bry = np.minimum(box_i[3], boxes[:, 3])
        en = ((tlx < brx) & (tly < bry)).astype(np.float32)
        inter = ((brx - tlx) * (bry - tly)) * en
        iou = inter / ((area_i + areas) - inter)
        return iou >= np.float32(thr)


def areas(box):
    with np.errstate(invalid="ignore", over="ignore"):
        return ((box[:, 2] - box[:, 0]) * (box[:, 3] - box[:, 1])).astype(np.float32)


def greedy(box, thr):
    """Greedy NMS over boxes already in order: indices of the kept ones."""
    ar = areas(box)
    kept = np.empty(len(box), np.int64)
    nk = 0
    for i in range(len(box)):
        if nk and iou_ge(box[i], ar[i], box[kept[:nk]], ar[kept[:nk]], thr).any():
            continue
        kept[nk] = i
        nk += 1
    return kept[:nk]


def image_order(cand):
    """Image-wide order: s descending (-0 == +0), class ascending, row descending."""
    return np.lexsort((-cand["row"], cand["cls"], -cand["s"]))


def rows_of(cand, idx):
    """Rows of the candidates idx, classes ascending, then s descending, then row descending; None when empty."""
    if len(idx) == 0:
        return None
    idx = np.asarray(idx)[np.lexsort((-cand["row"][idx], -cand["s"][idx], cand["cls"][idx]))]
    return np.concatenate([cand["box"][idx], cand["obj"][idx, None], cand["conf"][idx, None],
                           cand["cls"][idx, None].astype(np.float32)], 1).astype(np.float32)


def agnostic_kept(cand, thr):
    """Indices (into cand) of the candidates agnostic NMS keeps, in image-wide order."""
    order = image_order(cand)
    return order[greedy(cand["box"][order], thr)]


def per_class_kept(cand, thr):
    """Indices of the candidates per-class NMS keeps (utils.py:191-220 with the stable tie order): used to check candidates()
    against the C oracle."""
    order = image_order(cand)
    out = []
    for c in np.unique(cand["cls"]):
        oc = order[cand["cls"][order] == c]
        out.append(oc[greedy(cand["box"][oc], thr)])
    return np.concatenate(out) if out else np.zeros((0,), np.int64)


def postprocess(prediction, num_classes, conf_thre, nms_thre, agnostic=True):
    """prediction [B, M, 5+C] -> list of [K_i, 7] float32 arrays or None."""
    out = []
    for p in np.asarray(prediction, dtype=np.float32):
        cand = candidates(p, num_classes, conf_thre)
        kept = agnostic_kept(cand, nms_thre) if agnostic else per_class_kept(cand, nms_thre)
        out.append(rows_of(cand, kept))
    return out


def detect(raws, n_classes, conf_thre, nms_thre, agnostic=True):
    """Raw head tensors (numpy or CPU / CUDA tensors) -> the oracle's decode, then postprocess() above."""
    arrs = [r.detach().float().cpu().numpy() if hasattr(r, "detach") else np.asarray(r, np.float32) for r in raws]
    return postprocess(orc.decode_eval_cat(arrs, n_classes), n_classes, conf_thre, nms_thre, agnostic)
