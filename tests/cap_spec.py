"""The per-image detection cap (max_det) stated in NumPy: the function the capped outputs of the library are checked against."""
import numpy as np


def cap_detections(rows_list, max_det):
    """Per-image detection cap applied to uncapped results (list of [n, 7] arrays / tensors or None): an image with more
    than max_det rows keeps the first max_det of a stable descending sort by the fp32 score obj_conf * cls_conf (columns
    4 x 5; -0 == +0), emitted in the original order.  Returns numpy arrays / None."""
    out = []
    for r in rows_list:
        if r is None:
            out.append(None)
            continue
        r = np.asarray(r.detach().cpu().numpy() if hasattr(r, "detach") else r, dtype=np.float32)
        if r.shape[0] > max_det:
            s = r[:, 4] * r[:, 5]                                # fp32 product
            keep = np.sort(np.argsort(-s, kind="stable")[:max_det])
            r = r[keep]
        out.append(r)
    return out
