"""CPU-only checks of DIoU-NMS: the NumPy statement of the semantics (diou_spec) on hand-built scenes and against
torchvision's float64 DIoU, and argument validation of the C ABI and of the Python wrappers before any CUDA call."""
import numpy as np
import pytest
import torch

import agnostic_spec
import diou_spec as spec
from oracle import oracle as orc


def _pred(entries, C):
    """entries: (cx, cy, w, h, obj, {class: cls_conf}) -> one image [M, 5+C]."""
    p = np.zeros((len(entries), 5 + C), np.float32)
    for m, (cx, cy, w, h, obj, confs) in enumerate(entries):
        p[m, :5] = (cx, cy, w, h, obj)
        for c, v in confs.items():
            p[m, 5 + c] = v
    return p


def _run(entries, C, conf, thr, agnostic=False, diou=True):
    pred = _pred(entries, C)[None]
    rows = (spec.postprocess(pred, C, conf, thr, agnostic) if diou else agnostic_spec.postprocess(pred, C, conf, thr, agnostic))[0]
    return [] if rows is None else [(tuple(float(v) for v in r[:4]), int(r[6])) for r in rows]


def _decision(a, b, thr):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)[None]
    return bool(spec.diou_ge(a, agnostic_spec.areas(a[None])[0], b, agnostic_spec.areas(b), thr)[0])


def test_offset_pair_iou_drops_diou_keeps():
    # boxes [0,0,10,10] and [3,0,13,10]: IoU 70/130 = 0.538, penalty 9/269 = 0.033, DIoU 0.505
    e = [(5, 5, 10, 10, 1.0, {0: 0.9}), (8, 5, 10, 10, 1.0, {0: 0.8})]
    assert len(_run(e, 1, 0.1, 0.52, diou=False)) == 1
    assert len(_run(e, 1, 0.1, 0.52)) == 2
    # below both values both rules suppress, above both neither does
    assert len(_run(e, 1, 0.1, 0.5)) == 1 and len(_run(e, 1, 0.1, 0.55)) == 2


def test_concentric_boxes_equal_iou_nms():
    # boxes sharing a centre at dyadic coordinates: dx = dy = 0 exactly, pen = 0, so DIoU-NMS is IoU-NMS
    rng = np.random.RandomState(3)
    e = []
    for k in range(60):
        cx, cy = (32.0, 32.0) if k % 2 else (96.0, 64.0)
        e.append((cx, cy, 2.0 * rng.randint(1, 30), 2.0 * rng.randint(1, 30), 1.0, {k % 3: float(rng.rand()) + 0.1}))
    pred = _pred(e, 3)
    a = pred[:, :4]
    box = np.stack([a[:, 0] - a[:, 2] / 2, a[:, 1] - a[:, 3] / 2, a[:, 0] + a[:, 2] / 2, a[:, 1] + a[:, 3] / 2], 1)
    _, pen = spec.iou_and_penalty(box[0], agnostic_spec.areas(box[:1])[0], box[::2], agnostic_spec.areas(box[::2]))
    assert not pen.any()
    for thr in (0.3, 0.5, 0.7):
        for agn in (False, True):
            got = spec.postprocess(pred[None], 3, 0.05, thr, agn)[0]
            want = agnostic_spec.postprocess(pred[None], 3, 0.05, thr, agn)[0]
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
        assert np.array_equal(spec.postprocess(pred[None], 3, 0.05, thr)[0].view(np.uint32),
                              orc.postprocess(pred[None], 3, 0.05, thr)[0].view(np.uint32))


def test_exact_tie_is_suppressed():
    # a = [0,0,4,4], b = [0,0,4,2]: iou = 8/16 = 0.5, centres (2,2) and (2,1), enclosing box 4 x 4, pen = 1/32: every value is
    # exact, fl(iou - pen) = 0.46875
    a, b = [0, 0, 4, 4], [0, 0, 4, 2]
    assert _decision(b, a, 0.46875) and _decision(a, b, 0.46875)
    assert not _decision(b, a, float(np.nextafter(np.float32(0.46875), np.float32(1))))
    e = [(2, 2, 4, 4, 1.0, {0: 0.9}), (2, 1, 4, 2, 1.0, {0: 0.8})]
    assert len(_run(e, 1, 0.1, 0.46875)) == 1
    assert len(_run(e, 1, 0.1, float(np.nextafter(np.float32(0.46875), np.float32(1))))) == 2


def test_nan_penalty_keeps_the_pair():
    # disjoint finite boxes whose centre distance and enclosing diagonal overflow: iou = -0, pen = inf / inf = NaN.  IoU
    # suppresses at thr <= 0 (-0 >= 0); DIoU does not
    a, b = [-2e38, 0, -1e38, 1], [1e38, 0, 2e38, 1]
    iou, pen = spec.iou_and_penalty(np.float32(a), np.float32(1e38), np.float32([b]), np.float32([1e38]))
    assert iou[0] == 0 and np.isnan(pen[0])
    for thr in (0.0, -0.5):
        assert not _decision(a, b, thr)
        assert agnostic_spec.iou_ge(np.float32(a), np.float32(1e38), np.float32([b]), np.float32([1e38]), thr)[0]
    # one point twice: c^2 = 0, pen = 0 / 0
    assert not _decision([5, 5, 5, 5], [5, 5, 5, 5], -1.0)


def test_degenerate_boxes_never_suppress_at_positive_threshold():
    nan, inf = np.float32(np.nan), np.float32(np.inf)
    e = [(nan, 50, 20, 20, 1.0, {0: 0.9, 1: 0.8}),          # NaN coordinate
         (100, 100, 0, 0, 1.0, {0: 0.9, 1: 0.8}),           # zero area
         (150, 150, -4, 6, 1.0, {0: 0.9, 1: 0.8}),          # negative extent
         (200, 200, inf, 10, 1.0, {0: 0.9, 1: 0.8}),        # infinite extent
         (300, 300, 3e38, 3e38, 1.0, {0: 0.9, 1: 0.8})]     # finite extents, overflowing area
    for thr in (0.5, 1e-4):
        assert len(_run(e, 2, 0.1, thr, agnostic=True)) == 10  # no copy suppresses another, itself included
        assert len(_run(e + e, 2, 0.1, thr)) == 20
    for box in ([0, 0, 0, 0], [5, 5, 5, 9], [0, 0, -1, 3], [nan, 0, 1, 1], [0, 0, inf, 1]):
        assert not _decision(box, box, 0.5)


def test_thresholds_le_zero_let_disjoint_boxes_suppress():
    # [0,0,10,10] and [100,100,110,110]: iou 0, pen 20000/24200, DIoU -0.826
    e = [(5, 5, 10, 10, 1.0, {0: 0.9}), (105, 105, 10, 10, 1.0, {0: 0.8})]
    assert len(_run(e, 1, 0.1, 0.0, diou=False)) == 1
    assert len(_run(e, 1, 0.1, 0.0)) == 2
    assert len(_run(e, 1, 0.1, -0.5)) == 2
    assert len(_run(e, 1, 0.1, -0.9)) == 1
    # thr > 1: nothing is suppressed
    assert len(_run(e + [(5, 5, 10, 10, 1.0, {0: 0.7})], 1, 0.1, 1.5)) == 3


def test_diou_with_agnostic_across_classes():
    # the offset pair in two classes: agnostic IoU keeps one, agnostic DIoU keeps both, with their classes
    e = [(5, 5, 10, 10, 1.0, {0: 0.9}), (8, 5, 10, 10, 1.0, {2: 0.8})]
    assert [c for _, c in _run(e, 3, 0.1, 0.52, agnostic=True, diou=False)] == [0]
    assert sorted(c for _, c in _run(e, 3, 0.1, 0.52, agnostic=True)) == [0, 2]
    # one box in several classes: self DIoU = self IoU = 1, so it still keeps only its best class
    e = [(50, 50, 20, 20, 1.0, {1: 0.9, 3: 0.6, 5: 0.95})]
    assert [c for _, c in _run(e, 6, 0.1, 0.5, agnostic=True)] == [5]


def test_decision_against_torchvision_float64():
    """The spec's decision against torchvision's float64 DIoU on seeded random pairs, wherever that value is farther than 1e-5
    from the threshold (closer pairs are decided by fp32 rounding, which the spec states and float64 does not)."""
    tv = pytest.importorskip("torchvision")
    rng = np.random.RandomState(11)

    def boxes(n):
        xy = (rng.rand(n, 2) * 30).astype(np.float32)
        wh = (rng.rand(n, 2) * 30 + 1).astype(np.float32)
        return np.concatenate([xy, xy + wh], 1).astype(np.float32)

    a, b = boxes(300), boxes(300)
    ref = tv.ops.distance_box_iou(torch.from_numpy(a).double(), torch.from_numpy(b).double(), eps=0.0).numpy()
    aa, ab = agnostic_spec.areas(a), agnostic_spec.areas(b)
    checked = 0
    for thr in (-0.3, 0.1, 0.3, 0.5, 0.7):
        got = np.stack([spec.diou_ge(a[i], aa[i], b, ab, thr) for i in range(len(a))])
        far = np.abs(ref - thr) > 1e-5
        assert np.array_equal(got[far], ref[far] >= thr)
        assert (ref[far] >= thr).any() and (ref[far] < thr).any()
        checked += int(far.sum())
    assert checked > 0.99 * 5 * ref.size


def test_spec_greedy_is_a_valid_nms():
    """Oracle-free: kept boxes of a class never reach DIoU >= thr, and every dropped candidate has an earlier kept one that does."""
    rng = np.random.RandomState(2)
    pred = np.zeros((300, 8), np.float32)
    pred[:, 0:2] = rng.rand(300, 2) * 100
    pred[:, 2:4] = rng.rand(300, 2) * 40 + 2
    pred[:, 4] = rng.rand(300)
    pred[:, 5:] = rng.rand(300, 3)
    cand = agnostic_spec.candidates(pred, 3, 0.05)
    order = agnostic_spec.image_order(cand)
    pos = np.empty(len(order), np.int64)
    pos[order] = np.arange(len(order))
    k = spec.kept(cand, 0.45)
    kept = np.zeros(len(order), bool)
    kept[k] = True
    ar = agnostic_spec.areas(cand["box"])
    for i in range(len(order)):
        same = (cand["cls"] == cand["cls"][i]) & kept & (pos < pos[i])
        hit = spec.diou_ge(cand["box"][i], ar[i], cand["box"][same], ar[same], 0.45).any()
        assert hit != kept[i]


# ---- argument validation --------------------------------------------------------------------------------------------
def _lib():
    from yolov4_b200 import _cabi
    return _cabi, _cabi.lib()


@pytest.mark.parametrize("diou", [-1, 2, 255])
@pytest.mark.parametrize("agnostic", [0, 1])
def test_nms_ex2_rejects_bad_diou(diou, agnostic):
    _, L = _lib()
    ws_bytes = L.yl_post_workspace_bytes_ex(2, 1000, 80, 64, agnostic)
    # every other argument is well formed (pointers are never dereferenced on the host), so only diou can be refused
    assert L.yl_nms_ex2(4096, ws_bytes, 2, 1000, 80, 64, 0.5, 0, agnostic, diou, 4096, 16, 4096, None, 0, 2, None) == 1


def test_nms_ex2_checks_the_other_arguments_as_nms_ex():
    _, L = _lib()
    ws_bytes = L.yl_post_workspace_bytes_ex(2, 1000, 80, 64, 0)
    for diou in (0, 1):
        assert L.yl_nms_ex2(4096, ws_bytes, 2, 1000, 80, 64, 0.5, 0, 2, diou, 4096, 16, 4096, None, 0, 2, None) == 1
        assert L.yl_nms_ex2(4096, ws_bytes, 2, 1000, 80, 64, 0.5, 17, 0, diou, 4096, 16, 4096, None, 0, 2, None) == 1
        assert L.yl_nms_ex2(4096, ws_bytes - 1, 2, 1000, 80, 64, 0.5, 0, 0, diou, 4096, 16, 4096, None, 0, 2, None) == 3
        # no images: nothing to launch, so this succeeds without a device
        assert L.yl_nms_ex2(4096, ws_bytes, 2, 1000, 80, 64, 0.5, 0, 0, diou, 4096, 16, 4096, None, 0, 0, None) == 0


def test_detect_host_ex2_rejects_null_context_and_bad_diou():
    _cabi, L = _lib()
    rows = np.zeros((1, 16, 7), np.float32)
    counts = np.zeros((1,), np.int32)
    ptrs = _cabi.ptrs([4096, 4096, 4096])
    for diou in (0, 1, 2, -1):
        assert L.yl_detect_host_ex2(None, ptrs, 0.5, 0.5, 0, 0, diou, rows.ctypes.data, counts.ctypes.data) == 1


@pytest.mark.parametrize("bad", [1, 0, None, "yes", np.bool_(True), 1.0])
def test_wrappers_reject_non_bool_diou_before_any_cuda_work(bad):
    import yolov4_b200 as yb
    # CPU tensors: a wrapper that got past the diou check would raise TypeError for the tensors, with another message
    with pytest.raises(TypeError, match="diou"):
        yb.detect_raw([torch.zeros(1, 255, 4, 4)], 80, 0.5, 0.5, diou=bad)
    with pytest.raises(TypeError, match="diou"):
        yb.postprocess(torch.zeros(1, 10, 85), 80, 0.5, 0.5, diou=bad)
    with pytest.raises(TypeError, match="diou"):
        yb.HeadPostprocessor(1, [8, 4, 2], 80, 0.5, 0.5, device="cuda", diou=bad)
