"""The builders of the NMS back end's edge cases (nms_edge_cases.py), checked without a GPU: every exact-decision pair decides
at its threshold q and flips one ulp beyond, the scaled copies reach every fp32 regime they are planted for, the area-gap pairs
straddle area_bin_gap, the planted queue cluster holds 512 / 513 pairs, the restated workspace layout matches the library, and
yl_nms_ex2 rejects bad arguments before any CUDA work."""
from fractions import Fraction

import numpy as np
import pytest

import agnostic_spec as spec
import nms_edge_cases as nec

F32 = np.float32


def _exact_iou(a, b):
    """The true IoU of two boxes with exact rational arithmetic (no rounding anywhere), or None without an overlap."""
    a, b = [Fraction(float(v)) for v in a], [Fraction(float(v)) for v in b]
    w, h = min(a[2], b[2]) - max(a[0], b[0]), min(a[3], b[3]) - max(a[1], b[1])
    if w <= 0 or h <= 0:
        return None
    inter = w * h
    return inter / ((a[2] - a[0]) * (a[3] - a[1]) + (b[2] - b[0]) * (b[3] - b[1]) - inter)


@pytest.mark.parametrize("name", list(nec.BASE_PAIRS))
def test_pair_decides_at_q_and_flips_one_ulp_above(name):
    """In the literal fp32 formula B is suppressed at q and one ulp below it and kept one ulp above; the exact IoU says on which
    side of q the true value sits (fl(inter / uni) is within half an ulp of it)."""
    a, b, anchors = nec.BASE_PAIRS[name]
    for box in (a, b) + tuple(anchors):
        nec.xyxy_to_xywh(box)
    q, thr = nec.pair_threshold(name)
    boxes = np.array([b], np.float32)
    ar = spec.areas(np.array([a], np.float32))[0]
    for side, want in (("q", True), ("below", True), ("above", False)):
        assert bool(spec.iou_ge(np.array(a, np.float32), ar, boxes, spec.areas(boxes), thr[side])[0]) == want, side
    exact = _exact_iou(a, b)
    if exact is None:
        assert q == 0
    else:
        assert abs(Fraction(float(q)) - exact) <= Fraction(float(np.spacing(q))) / 2
        assert Fraction(float(thr["above"])) > exact


def test_scaled_copies_reach_every_regime():
    """Over all pairs and scales: areas in area bin 0 and bin 47, subnormal areas and intersections, overflowing areas, a
    union that overflows from finite areas, coordinates beyond +-1e6, and decisions at scale 2^k that differ from scale 1."""
    seen = set()
    for name, (a, b, _) in nec.BASE_PAIRS.items():
        q = nec.pair_threshold(name)[0]
        for k in nec.SCALES:
            A, B = nec.scaled(a, k), nec.scaled(b, k)
            nec.xyxy_to_xywh(A), nec.xyxy_to_xywh(B)
            iou, inter, uni, aa, ab = nec.literal_iou(A, B)
            for ar in (aa, ab):
                if 0 < ar < np.finfo(np.float32).tiny:
                    seen.add("subnormal area")
                if np.isinf(ar):
                    seen.add("area overflows")
                if np.isfinite(ar) and ar > 0:
                    seen.add("bin %d" % nec.area_bin(ar) if nec.area_bin(ar) in (0, nec.NBIN - 1) else "bin inside")
            if 0 < inter < np.finfo(np.float32).tiny:
                seen.add("subnormal inter")
            if np.isfinite(aa) and np.isfinite(ab) and np.isinf(uni):
                seen.add("union overflows")
            if max(abs(v) for v in A + B) > 1e6:
                seen.add("beyond 1e6")
            if not iou == q:
                seen.add("scale changes the IoU")
    want = {"subnormal area", "area overflows", "bin 0", "bin 47", "bin inside", "subnormal inter", "union overflows",
            "beyond 1e6", "scale changes the IoU"}
    assert want <= seen, want - seen


def test_area_gap_pairs_straddle_the_gap():
    """At every planted threshold: each pair's bins differ by exactly its gap, every pair whose gap reaches K = area_bin_gap(thr)
    has IoU < thr (the exclusion the small tier's area tables make is exact), and at the pair-IoU thresholds pairs at gap
    K - 1 do reach the threshold (a gap one too small would drop their suppression)."""
    biting = 0
    for thr in nec.gap_change_thresholds() + nec.gap_pair_thresholds():
        images, _, where = nec.area_gap_images(thr)
        K = nec.area_bin_gap(thr)
        for (b, c), (gap, p) in where.items():
            A, Bx = images[b][c][0]
            ar = spec.areas(np.array([A, Bx], np.float32))
            assert nec.area_bin(ar[0]) - nec.area_bin(ar[1]) == gap and nec.area_bin(ar[1]) == p
            iou = nec.literal_iou(A, Bx)[0]
            if gap >= K:
                assert iou < thr, (thr, gap, p)
            elif gap == K - 1 and iou >= thr:
                biting += 1
    assert biting >= 8
    assert len(nec.gap_change_thresholds()) >= 16


def test_gap_change_thresholds_change_the_gap():
    ts = nec.gap_change_thresholds()
    for lo, hi in zip(ts[0::2], ts[1::2]):
        assert np.nextafter(lo, F32(np.inf)) == hi and nec.area_bin_gap(lo) == nec.area_bin_gap(hi) + 1


@pytest.mark.parametrize("extra,pairs", [(1, 512), (2, 513)])
def test_queue_cluster_holds_512_and_513_pairs(extra, pairs):
    boxes, scores = nec.queue_cluster(extra)
    q = nec.small_tier_queues(boxes, F32(0.45))
    assert q[0] == pairs and q[1:].max() < 512 and len(boxes) <= nec.SMALL_R
    assert nec.must_go_big(boxes, F32(0.45), 256) == (pairs > 512)


@pytest.mark.parametrize("n", (1, 2, 63, 64, 65, 127, 128, 129, 255, 256))
def test_routing_sizes_stay_in_the_small_tier(n):
    """The scattered segments of the size tests never overflow a pair queue: n alone decides their tier."""
    boxes, _ = nec.routing_segment(n, n)
    assert nec.small_tier_queues(boxes, F32(0.45)).max() <= 64


def test_degenerate_segments():
    """Identical boxes at a tiny range or beyond 1e6 leave a bin scale of 0 (every pair a candidate, 496 + 284 pairs per warp
    queue at most); invalid boxes are no candidates at all."""
    for where in ("tiny", "huge"):
        boxes, _ = nec.identical_segment(40, where)
        b = np.array(boxes, np.float32)
        lo, hi = max(F32(min(b[:, 0].min(), b[:, 1].min())), F32(-1e6)), min(F32(max(b[:, 2].max(), b[:, 3].max())), F32(1e6))
        with np.errstate(over="ignore"):
            scale = F32(F32(48) / F32(hi - lo))
        assert not (scale > 0 and scale < F32(3e38)), where
        assert nec.small_tier_queues(boxes, F32(0.45)).tolist() == [496, 284, 0, 0]
    xywh, scores, _ = nec.invalid_segment()
    pred = nec.make_pred([{0: (xywh, scores, "xywh")}], 1)
    box = spec.candidates(pred[0], 1, nec.CONF)["box"]
    assert len(box) == len(xywh)
    with np.errstate(invalid="ignore"):
        assert not ((box[:, 0] < box[:, 2]) & (box[:, 1] < box[:, 3])).any()
    assert nec.small_tier_queues(box, F32(0.45)).max() == 0


@pytest.mark.parametrize("B,M,C,cap_seg", [(1, 1, 1, 1), (2, 45, 20, 16), (3, 22743, 80, 1024), (5, 13, 128, 1025),
                                           (64, 22743, 80, 2048), (7, 3, 33, 300)])
def test_restated_layout_gives_the_workspace_size(B, M, C, cap_seg):
    from yolov4_b200 import _cabi
    L = _cabi.lib()
    assert nec.layout(B, M, C, cap_seg)["total"] == L.yl_post_workspace_bytes(B, M, C, cap_seg)


def test_nms_rejects_bad_arguments_before_cuda_work():
    """Every argument error returns before the first CUDA call (this runs without a device): pointers are never touched, so
    stand-in addresses do, and a threshold of any value (NaN included) is not an error."""
    from yolov4_b200 import _cabi
    L = _cabi.lib()
    fake = 1 << 20
    B, M, C, cap_seg = 4, 100, 20, 16
    nb = L.yl_post_workspace_bytes_ex(B, M, C, cap_seg, 1)

    def call(thr=0.45, max_det=0, agnostic=0, diou=0, cap_out=32, i0=0, cnt=0, c=C, wsb=nb, ws=fake, rows=fake, meta=fake):
        return L.yl_nms_ex2(ws, wsb, B, M, c, cap_seg, thr, max_det, agnostic, diou, rows, cap_out, meta, None, i0, cnt, None)

    for thr in (0.45, float("nan"), float("inf"), -0.0, -1.0):
        assert call(thr=thr) == 0 and call(thr=thr, max_det=32, agnostic=1, diou=1, i0=B) == 0
        for kw in (dict(cap_out=0), dict(cap_out=-5), dict(max_det=-1), dict(max_det=33), dict(cap_out=8, max_det=9),
                   dict(agnostic=2), dict(diou=-1), dict(i0=-1), dict(i0=B, cnt=1), dict(cnt=B + 1), dict(ws=None),
                   dict(rows=None), dict(meta=None)):
            assert call(thr=thr, **kw) == 1, (thr, kw)
        assert call(thr=thr, c=129) == 2
        assert call(thr=thr, cnt=B, wsb=L.yl_post_workspace_bytes(B, M, C, cap_seg) - 1) == 3
        assert call(thr=thr, cnt=B, agnostic=1, wsb=nb - 1) == 3
