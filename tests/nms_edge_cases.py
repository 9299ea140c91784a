"""Decoded [B, M, 5+C] inputs for the NMS back end (yl_nms / yl_nms_ex2 after yl_filter_dense) at its exact decisions, its bin
shortcuts and its routing boundaries, and NumPy restatements of the small tier's planting rules.

Every planted row has obj = 1 and its score in one class column (every other class 0), and the filter runs at a tiny positive
conf, so each (image, class) segment holds exactly the planted boxes in the planted score order.  Boxes are given as x1, y1,
x2, y2 with dyadic values for which the filter's cx -+ w/2 gives those corners back exactly (xyxy_to_xywh checks it).

The restatements (area_bin_gap, small_tier_queues) follow yl_nms.cu operation for operation.  They are used to plant pairs on
either side of a shortcut's boundary and to say which segments the small tier must pass on to the big tier; the result of
every case is checked against the literal fp32 NMS, never against them.
"""
import math

import numpy as np

import agnostic_spec as spec

F32 = np.float32
TINY = np.array([1], np.uint32).view(np.float32)[0]                    # smallest subnormal, 1.4e-45
CONF = F32(2.0 ** -60)                                                  # below every planted score, above 0
NBIN, SMALL_R, SMALL_THREADS, QCAP_W, SMEM_R = 48, 256, 128, 512, 1024
AREA_BIN_OFF = (127 + 4) << 2
THRESHOLDS = [TINY, F32(1e-6), F32(0.45), F32(0.999), F32(1), F32(1.5), F32(np.inf), F32(0.0), F32(-0.0), F32(-0.5),
              F32(np.nan)]


def nextf(x, d):
    return np.nextafter(F32(x), F32(d))


# ------------------------------------------------------------------------------------------------ case assembly
def xyxy_to_xywh(box):
    """(cx, cy, w, h) whose corners in the filter's fp32 arithmetic are exactly box (asserted)."""
    x1, y1, x2, y2 = (F32(v) for v in box)
    w, h = F32(x2 - x1), F32(y2 - y1)
    cx, cy = F32(x1 + w / F32(2)), F32(y1 + h / F32(2))
    back = (F32(cx - w / F32(2)), F32(cy - h / F32(2)), F32(cx + w / F32(2)), F32(cy + h / F32(2)))
    assert back == (x1, y1, x2, y2), (box, back)
    return cx, cy, w, h


def make_pred(images, C, seed=0, xywh=False):
    """images: list (per image) of {class: (boxes [n, 4], scores [n])}, boxes xyxy (or cx, cy, w, h with xywh=True or a third
    tuple item).  The rows of an image are shuffled (the filter's record order and the box rows then differ from the score
    order), images padded with rows no class passes.  Returns pred [B, M, 5+C] float32."""
    rng = np.random.RandomState(seed)
    per = []
    for segs in images:
        rows = []
        for c, seg in sorted(segs.items()):
            as_xywh = xywh or len(seg) > 2                              # (boxes, scores, "xywh"): given as cx, cy, w, h
            for bx, s in zip(seg[0], seg[1]):
                r = np.zeros(5 + C, np.float32)
                r[:4] = bx if as_xywh else xyxy_to_xywh(bx)
                r[4], r[5 + c] = 1.0, s
                rows.append(r)
        per.append(np.array(rows, np.float32).reshape(-1, 5 + C)[rng.permutation(len(rows))])
    M = max(1, max(len(p) for p in per))
    pred = np.zeros((len(images), M, 5 + C), np.float32)
    for b, p in enumerate(per):
        pred[b, :len(p)] = p
    return pred


def descending_scores(n, top=0.75):
    """n distinct scores, descending, exact in fp32."""
    return (F32(top) - np.arange(n, dtype=np.float32) * F32(2.0 ** -14)).astype(np.float32)


# ------------------------------------------------------------------------------------------------ exact-decision pairs
U22, U19 = 2.0 ** -22, 2.0 ** -19
# name -> (kept box A, candidate B, anchors): A scores above B; anchors (lowest scores, touching nothing) fix the segment's
# coordinate range, so that for "edge_*" a bin edge of the small tier's coordinate tables (48 bins over [0, 192]) sits at x = 16
BASE_PAIRS = {
    "partial": ((0, 0, 10, 10), (3, 4, 13, 14), ()),
    "contained": ((0, 0, 16, 16), (2, 3, 9, 12), ()),
    "identical": ((1, 1, 7, 5), (1, 1, 7, 5), ()),
    "touching": ((0, 0, 8, 8), (8, 0, 16, 8), ()),
    "ulp_overlap": ((0, 0, 3, 2), (3 - U22, 0, 3.5 - U22, 2), ()),
    "ratio_045": ((0, 0, 20, 20), (1, 1, 13, 16), ()),
    "ratio_0999": ((0, 0, 1000, 1000), (0, 0, 999, 1000), ()),
    "edge_touch": ((16, 8, 24, 24), (12, 8, 16, 24), ((0, 0, 1, 1), (191, 191, 192, 192))),
    "edge_ulp": ((16, 8, 24, 24), (12 + U19, 8, 16 + U19, 24), ((0, 0, 1, 1), (191, 191, 192, 192))),
}
SCALES = list(range(-80, 68))                                           # coordinates times 2^k
FILLER = {"small": 0, "big": 300 - 2, "global": 1100 - 2}               # records added to reach each tier


def literal_iou(a, b):
    """fl32 IoU of two xyxy boxes, the literal NaN-propagating formula (agnostic_spec.iou_ge's arithmetic)."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)[None]
    with np.errstate(invalid="ignore", over="ignore", divide="ignore", under="ignore"):
        aa, ab = spec.areas(a[None])[0], spec.areas(b)[0]
        tlx, tly = np.maximum(a[0], b[0, 0]), np.maximum(a[1], b[0, 1])
        brx, bry = np.minimum(a[2], b[0, 2]), np.minimum(a[3], b[0, 3])
        en = F32((tlx < brx) & (tly < bry))
        inter = F32(F32(F32(brx - tlx) * F32(bry - tly)) * en)
        return F32(inter / F32(F32(aa + ab) - inter)), inter, F32(F32(aa + ab) - inter), aa, ab


def pair_threshold(name):
    """q = the literal IoU of the pair at scale 1, and the three thresholds q, q one ulp down, q one ulp up."""
    a, b, _ = BASE_PAIRS[name]
    q = literal_iou(a, b)[0]
    return q, {"q": q, "below": nextf(q, -np.inf), "above": nextf(q, np.inf)}


def scaled(box, k):
    return tuple(F32(v) * F32(2.0 ** k) for v in box)


def filler_boxes(n):
    """n non-overlapping 2x2 boxes in a band far from every base pair (x, y >= 1200)."""
    i = np.arange(n)
    x, y = 1200 + 4 * (i % 64), 1200 + 4 * (i // 64)
    return [(float(a), float(c), float(a + 2), float(c + 2)) for a, c in zip(x, y)]


def pair_images(name, tier="small"):
    """One copy of the pair per segment, at every scale of SCALES: image 0 holds the scales below 2^-6 (class = position in
    its half), image 1 the others.  tier adds filler records (lowest scores) so that each segment has more than 256 records
    (big tier in shared memory) or more than 1024 (big tier in global memory).  Returns (images, C, {(b, c): k})."""
    a, b, anchors = BASE_PAIRS[name]
    extra = list(anchors) + filler_boxes(FILLER[tier])
    half = [k for k in SCALES if k < -6], [k for k in SCALES if k >= -6]
    images, where = [], {}
    for img, ks in enumerate(half):
        segs = {}
        for c, k in enumerate(ks):
            boxes = [scaled(a, k), scaled(b, k)] + [scaled(e, k) for e in extra]
            segs[c] = (boxes, descending_scores(len(boxes)))
            where[(img, c)] = k
        images.append(segs)
    return images, max(len(h) for h in half), where


# ------------------------------------------------------------------------------------------------ area bins
def area_bin_gap(thr):
    """yl_nms.cu area_bin_gap, restated for planting: the smallest area-bin gap at which suppresses_pos's area test alone
    already rules a pair out."""
    thr = float(thr)
    if not thr > 0:
        return NBIN + 1
    need = 1.0 / (0.999 * thr) * 1.001
    for K in range(1, NBIN + 1):
        worst = 1e300
        for p in range(4):
            hi, lo = p + K, p + 1
            worst = min(worst, math.ldexp(1.0 + (hi & 3) * 0.25, hi >> 2) / math.ldexp(1.0 + (lo & 3) * 0.25, lo >> 2))
        if worst >= need:
            return K
    return NBIN + 1


def area_bin(area):
    """Area bin of the small tier: float bits >> 21 (four bins per octave) from 16 px^2, clamped to [0, NBIN)."""
    bits = np.asarray(area, np.float32).view(np.uint32).astype(np.int64)
    return np.clip((bits >> 21) - AREA_BIN_OFF, 0, NBIN - 1)


def gap_change_thresholds():
    """Thresholds on both sides of every change of area_bin_gap between K = 2 and K = 12: the largest fp32 threshold with
    the smaller K and the next float."""
    out = []
    lo_bits = np.array([F32(0.05)]).view(np.uint32)[0]
    hi_bits = np.array([F32(1.0)]).view(np.uint32)[0]
    f = lambda u: np.array([u], np.uint32).view(np.float32)[0]          # noqa: E731
    for K in range(2, 13):
        # area_bin_gap is non-increasing in thr: find the last threshold whose gap is still > K - 1 ... bisection on the bits
        a, b = int(lo_bits), int(hi_bits)
        if not (area_bin_gap(f(a)) >= K > area_bin_gap(f(b))):
            continue
        while b - a > 1:
            m = (a + b) // 2
            if area_bin_gap(f(m)) >= K:
                a = m
            else:
                b = m
        out += [f(a), f(b)]
    return out


def area_gap_pair(base_bin, gap):
    """Contained pair (A outside, B inside, both from the origin, one height) whose areas sit at the tightest spot of a bin
    gap: area(B) the largest float of bin base_bin, area(A) the smallest float of bin base_bin + gap.  Its IoU is the
    largest a pair with that bin gap can have at this in-octave position."""
    amin = np.array([((base_bin + 1 + AREA_BIN_OFF) << 21) - 1], np.uint32).view(np.float32)[0]
    amax = np.array([(base_bin + gap + AREA_BIN_OFF) << 21], np.uint32).view(np.float32)[0]
    h = F32(4.0)
    A, Bx = (0.0, 0.0, float(amax / h), float(h)), (0.0, 0.0, float(amin / h), float(h))
    assert spec.areas(np.array([A], np.float32))[0] == amax and spec.areas(np.array([Bx], np.float32))[0] == amin
    return A, Bx


AREA_BASE_BINS = (8, 9, 10, 11)                                         # the four in-octave positions (areas 64 .. 128)


def gap_pair_thresholds(gaps=range(1, 9)):
    """The IoU of the tightest pair of each gap and in-octave position: at that threshold the pair is suppressed, and its gap
    is below area_bin_gap (often exactly K - 1, where a gap one too small would wrongly rule it out)."""
    return sorted({literal_iou(*area_gap_pair(p, g))[0] for g in gaps for p in AREA_BASE_BINS})


def area_gap_images(thr):
    """At thr (K = area_bin_gap(thr)): one segment per (gap in K-1, K, K+1) x in-octave position.  Returns (images, C,
    {(0, c): (gap, base_bin)})."""
    K = area_bin_gap(thr)
    segs, where = {}, {}
    for gap in (K - 1, K, K + 1):
        for p in AREA_BASE_BINS:
            if gap < 1:
                continue
            c = len(segs)
            segs[c] = (list(area_gap_pair(p, gap)), descending_scores(2))
            where[(0, c)] = (gap, p)
    return [segs], len(segs), where


# ------------------------------------------------------------------------------------------------ routing
def sorted_segment(pred_b, C, c):
    """Boxes of the (image, class) segment in the small tier's order (score desc, box row desc) as the literal filter makes
    them."""
    cand = spec.candidates(pred_b, C, CONF)
    sel = np.nonzero(cand["cls"] == c)[0]
    o = sel[np.lexsort((-cand["row"][sel], -cand["s"][sel]))]
    return cand["box"][o]


def _coord_bin(v, lo, scale):
    with np.errstate(invalid="ignore", over="ignore"):
        x = F32(F32(v - lo) * scale)
    q = np.where(np.isnan(x), 0.0, np.floor(np.clip(np.nan_to_num(x, nan=0.0, posinf=3e9, neginf=-3e9), -3e9, 3e9)))
    return np.clip(q, 0, NBIN - 1).astype(np.int64)


def small_tier_queues(box, thr):
    """Candidate pairs per warp queue of k_segment_nms_bins for a segment already in its sorted order (steps 1-4 of the
    kernel: coordinate range clamped to +-1e6, 48 coordinate bins, area bins, the six exclusion tests).  Returns [4] counts."""
    box = np.asarray(box, np.float32)
    n = len(box)
    with np.errstate(invalid="ignore"):
        valid = (box[:, 0] < box[:, 2]) & (box[:, 1] < box[:, 3])
    lo, hi = F32(np.inf), F32(-np.inf)
    if valid.any():
        v = box[valid]
        lo, hi = F32(min(v[:, 0].min(), v[:, 1].min())), F32(max(v[:, 2].max(), v[:, 3].max()))
    lo, hi = max(lo, F32(-1e6)), min(hi, F32(1e6))
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        scale = F32(F32(NBIN) / F32(hi - lo))
    if not (scale > 0 and scale < F32(3e38)):
        scale = F32(0)
    bx1, by1, bx2, by2 = (_coord_bin(box[:, i], lo, scale) for i in (0, 1, 2, 3))
    with np.errstate(over="ignore", invalid="ignore"):
        ab = area_bin(spec.areas(box))
    K = area_bin_gap(thr)
    q = np.zeros(SMALL_THREADS // 32, np.int64)
    for j in range(n):
        if not valid[j]:
            continue
        i = np.arange(j)
        ok = valid[:j] & ~((bx1[:j] > bx2[j]) | (bx2[:j] < bx1[j]) | (by1[:j] > by2[j]) | (by2[:j] < by1[j]) |
                           (ab[:j] - K >= ab[j]) | (ab[:j] + K <= ab[j]))
        q[(j % SMALL_THREADS) // 32] += int(ok[i].sum())
    return q


def must_go_big(box, thr, cap_seg):
    """Whether k_segment_nms_bins passes the segment on: more than 256 records, !(thr > 0) or a warp queue over 512 pairs.
    None for a segment that takes no NMS at all (empty, or over cap_seg)."""
    n = len(box)
    if n == 0 or n > cap_seg:
        return None
    if n > SMALL_R or not thr > 0:
        return True
    return bool(small_tier_queues(box, thr).max() > QCAP_W)


def site_boxes(sites):
    """Boxes on the 48 x-bins of a [0, 192] range (bin width 4): a box at site s spans x in [4s+1, 4s+3] and the full height, so
    boxes at one site are candidates of each other and of nothing else."""
    return [(4.0 * s + 1, 0.0, 4.0 * s + 3, 192.0) for s in sites]


def queue_cluster(extra_pairs):
    """A segment whose warp-0 queue holds 496 + 15 + extra_pairs pairs: sorted rows 0..31 at site 0 (496 pairs), rows 32..127
    on sites 1..40 (queues of warps 1-3), rows 128..133 at site 41 (15 pairs), then extra_pairs pairs of rows on sites
    42, 43, ... (one pair each).  Returns (boxes in score order, scores)."""
    sites = [0] * 32 + [1 + (i % 40) for i in range(96)] + [41] * 6
    for e in range(extra_pairs):
        sites += [42 + e, 42 + e]
    boxes = site_boxes(sites)
    return boxes, descending_scores(len(boxes))


def routing_segment(n, seed):
    """n boxes of 8..24 px scattered over a 600 px square: overlapping neighbours, few candidate pairs per warp."""
    rng = np.random.RandomState(seed)
    xy = np.floor(rng.rand(n, 2) * 576) + 8
    wh = 8 + 2 * np.floor(rng.rand(n, 2) * 8)
    boxes = [(float(x), float(y), float(x + w), float(y + h)) for (x, y), (w, h) in zip(xy, wh)]
    return boxes, descending_scores(n, top=0.9)


def tie_segment(n, seed):
    """n boxes in overlapping pairs (IoU 0.6) whose two boxes share a score; every score is shared by a pair and pairs sit
    all along the order, 128 included, so only the (score, row) re-rank separates them."""
    rng = np.random.RandomState(seed)
    boxes, scores = [], []
    for i in range(n // 2):
        x, y = 8 + 40 * (i % 14), 8 + 40 * (i // 14)
        boxes += [(float(x), float(y), float(x + 16), float(y + 16)), (float(x + 4), float(y), float(x + 20), float(y + 16))]
        s = F32(0.5) + F32(rng.randint(0, 3)) * F32(2.0 ** -20) if i % 3 else F32(0.5)   # many pairs tie with other pairs too
        scores += [s, s]
    return boxes, np.array(scores, np.float32)


def invalid_segment():
    """Only boxes no pair test can see: NaN coordinates, zero width, zero height, negative extents (xywh form)."""
    nan = np.nan
    return ([(nan, 10, 8, 8), (20, nan, 8, 8), (30, 30, nan, 8), (40, 40, 8, nan), (50, 50, 0, 8), (60, 60, 8, 0),
             (70, 70, -4, 8), (80, 80, 8, -4), (90, 90, -0.0, 8)], descending_scores(9), "xywh")


def identical_segment(n, where):
    """n identical boxes: at tiny coordinates (the bin scale 48 / range overflows: one bin), or beyond 1e6 (the clamped
    range is empty: one bin)."""
    box = (2.0 ** -124, 2.0 ** -124, 2.0 ** -123, 2.0 ** -123) if where == "tiny" else (2e6, 2e6, 2e6 + 64, 2e6 + 32)
    return [box] * n, descending_scores(n)


def layout(B, M, C, cap_seg):
    """post_layout of yl_common.cuh: byte offsets of the workspace arrays."""
    al = lambda x: (x + 255) // 256 * 256                               # noqa: E731
    M4 = (M + 3) // 4 * 4
    L, o = {}, 0
    for name, nbytes in (("seg_count", 4 * B * C), ("kept_count", 4 * B * C), ("big_count", 4 * B), ("tile_count", 8 * B)):
        L[name] = o
        o += al(nbytes)
    L["counters_bytes"] = o
    for name, nbytes in (("big_list", 4 * B * C), ("cand", 32 * B * C * cap_seg), ("obj", 4 * B * M4),
                         ("flags", 4 * ((C + 31) // 32) * B * M4)):
        L[name] = o
        o += al(nbytes)
    L["kept_scratch"] = o
    if cap_seg > SMEM_R:
        o += al(4 * B * C * cap_seg)
    L["total"] = o
    return L
