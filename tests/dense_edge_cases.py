"""Decoded [B, M, 5+C] inputs for the dense front end (postprocess / yl_filter_dense) at its special values, and NumPy models
of its row filter.

The reference's row filter (utils.py:139-148) is literal: a row survives when obj * max(cls[:num_classes]) >= conf, the max
propagating NaN; every class column c of a surviving row with obj * cls[c] >= conf is a candidate (utils.py:170).
"""
import numpy as np

F32 = np.float32
INF, NAN = F32(np.inf), F32(np.nan)
TINY = np.array([1], np.uint32).view(np.float32)[0]                    # smallest subnormal, 1.4e-45
FLT_MAX = np.finfo(np.float32).max

TABLE_OBJ = [-INF, F32(-1), F32(-0.0), F32(0), TINY, F32(1e-30), F32(0.5), F32(1), FLT_MAX, INF, NAN]
TABLE_MAX = [-INF, F32(-1), F32(-0.0), F32(0), F32(0.5), F32(1), INF, NAN]
TABLE_CONF = [-INF, F32(-1), F32(0), TINY, F32(1e-4), F32(0.5), F32(1), INF, NAN]
TABLE_C, TABLE_NUM_CLASSES = 4, 2


def _companion(mx):
    """A second class inside num_classes that keeps mx the maximum: a finite one where mx allows, negative where mx <= 0."""
    if np.isnan(mx):
        return F32(0.25)
    if mx == -INF:
        return -INF
    return F32(0.25) if mx > 0 else F32(mx - 1) if mx < 0 else F32(-0.5)


def truth_table():
    """One image, one row per (obj, class max): classes [max, companion, 0.25, -1] with num_classes = 2, so the max is
    exactly the table value and every row also carries a finite and a negative class outside the max.  The 8x8 boxes sit on
    a 20-pixel grid and never overlap, so per-class NMS keeps every candidate.  Returns [M, 5+C] float32."""
    rows = []
    for obj in TABLE_OBJ:
        for mx in TABLE_MAX:
            i = len(rows)
            rows.append([10 + 20 * (i % 16), 10 + 20 * (i // 16), 8, 8, obj, mx, _companion(mx), 0.25, -1])
    return np.array(rows, np.float32)


def _per_class(pred, conf):
    with np.errstate(invalid="ignore", over="ignore"):
        return pred[:, 5:] * pred[:, 4:5] >= F32(conf)


def literal_pairs(pred, num_classes, conf):
    """[M, C] candidate mask of the reference's filter (what agnostic_spec.candidates selects)."""
    with np.errstate(invalid="ignore", over="ignore"):
        row = pred[:, 4] * np.max(pred[:, 5:5 + num_classes], axis=1) >= F32(conf)
    return _per_class(pred, conf) & row[:, None]


def shortcut_pairs(pred, num_classes, conf, use_shortcut):
    """[M, C] candidate mask of a filter that, where use_shortcut(obj) holds, replaces the max by 'one of the first num_classes
    classes passes the per-class test and none of them is NaN', and elsewhere is literal."""
    per = _per_class(pred, conf)
    short = per[:, :num_classes].any(1) & ~np.isnan(pred[:, 5:5 + num_classes]).any(1)
    with np.errstate(invalid="ignore"):
        sc = use_shortcut(pred[:, 4])
    return np.where(sc[:, None], per & short[:, None], literal_pairs(pred, num_classes, conf))


def shortcut_before_fix(obj):
    """The condition the unaligned kernel once took the shortcut on."""
    return obj >= 0


def shortcut_fixed(obj):
    """Finite positive objectness: fl(obj * x) is monotone in x and never NaN for a non-NaN x."""
    return (obj > 0) & (obj < INF)
