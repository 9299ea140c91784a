"""DIoU-NMS stated in NumPy: the literal algorithm the library's diou mode is checked against.

The candidates, their order and the output rows are those of per-class NMS (the C oracle's postprocess) or, with agnostic, of
agnostic_spec; only the suppression decision changes.  A candidate a is dropped by an earlier kept box b (both xyxy) when
    iou = the literal NaN-propagating fp32 IoU of utils.py:71-77 (agnostic_spec.iou_ge)
    dx  = (a.x1 + a.x2) * 0.5 - (b.x1 + b.x2) * 0.5        dy = (a.y1 + a.y2) * 0.5 - (b.y1 + b.y2) * 0.5
    cw  = max(a.x2, b.x2) - min(a.x1, b.x1)                 ch = max(a.y2, b.y2) - min(a.y1, b.y1)
    pen = (dx*dx + dy*dy) / (cw*cw + ch*ch)
    suppress  <=>  (iou - pen) >= thr
every operation one fp32 rounding in the order written, max / min propagating NaN.  Greedy runs over all candidates.
"""
import numpy as np

from agnostic_spec import areas, candidates, image_order, rows_of
from oracle import oracle as orc


def iou_and_penalty(box_a, area_a, boxes, areas_b):
    """(iou, pen) of one candidate box_a against many earlier boxes, fp32, NaN-propagating."""
    f = np.float32
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        tlx = np.maximum(box_a[0], boxes[:, 0])
        tly = np.maximum(box_a[1], boxes[:, 1])
        brx = np.minimum(box_a[2], boxes[:, 2])
        bry = np.minimum(box_a[3], boxes[:, 3])
        en = ((tlx < brx) & (tly < bry)).astype(f)
        inter = ((brx - tlx) * (bry - tly)) * en
        iou = inter / ((area_a + areas_b) - inter)
        h = f(0.5)
        dx = (box_a[0] + box_a[2]) * h - (boxes[:, 0] + boxes[:, 2]) * h
        dy = (box_a[1] + box_a[3]) * h - (boxes[:, 1] + boxes[:, 3]) * h
        cw = np.maximum(box_a[2], boxes[:, 2]) - np.minimum(box_a[0], boxes[:, 0])
        ch = np.maximum(box_a[3], boxes[:, 3]) - np.minimum(box_a[1], boxes[:, 1])
        pen = (dx * dx + dy * dy) / (cw * cw + ch * ch)
    return iou.astype(f), pen.astype(f)


def diou_ge(box_a, area_a, boxes, areas_b, thr):
    """The DIoU decision fl(iou - pen) >= thr of candidate box_a against each of boxes."""
    iou, pen = iou_and_penalty(box_a, area_a, boxes, areas_b)
    with np.errstate(invalid="ignore"):
        return (iou - pen) >= np.float32(thr)


def greedy(box, thr):
    """Greedy DIoU-NMS over boxes already in order: indices of the kept ones."""
    ar = areas(box)
    kept = np.empty(len(box), np.int64)
    nk = 0
    for i in range(len(box)):
        if nk and diou_ge(box[i], ar[i], box[kept[:nk]], ar[kept[:nk]], thr).any():
            continue
        kept[nk] = i
        nk += 1
    return kept[:nk]


def kept(cand, thr, agnostic=False):
    """Indices (into cand) of the candidates DIoU-NMS keeps: per class, or over the whole image with agnostic."""
    order = image_order(cand)
    if agnostic:
        return order[greedy(cand["box"][order], thr)]
    out = []
    for c in np.unique(cand["cls"]):
        oc = order[cand["cls"][order] == c]
        out.append(oc[greedy(cand["box"][oc], thr)])
    return np.concatenate(out) if out else np.zeros((0,), np.int64)


def postprocess(prediction, num_classes, conf_thre, nms_thre, agnostic=False):
    """prediction [B, M, 5+C] -> list of [K_i, 7] float32 arrays or None."""
    out = []
    for p in np.asarray(prediction, dtype=np.float32):
        cand = candidates(p, num_classes, conf_thre)
        out.append(rows_of(cand, kept(cand, nms_thre, agnostic)))
    return out


def detect(raws, n_classes, conf_thre, nms_thre, agnostic=False):
    """Raw head tensors (numpy or CPU / CUDA tensors) -> the oracle's decode, then postprocess() above."""
    arrs = [r.detach().float().cpu().numpy() if hasattr(r, "detach") else np.asarray(r, np.float32) for r in raws]
    return postprocess(orc.decode_eval_cat(arrs, n_classes), n_classes, conf_thre, nms_thre, agnostic)
