"""CPU-only checks of class-agnostic NMS: the NumPy statement of the semantics (agnostic_spec) on hand-built scenes, its
candidate filter and greedy pass against the C oracle, and argument validation of the C ABI and of the Python wrappers before
any CUDA call."""
import numpy as np
import pytest
import torch

import agnostic_spec as spec
from oracle import oracle as orc


def _pred(entries, C):
    """entries: (cx, cy, w, h, obj, {class: cls_conf}) -> one image [M, 5+C]."""
    p = np.zeros((len(entries), 5 + C), np.float32)
    for m, (cx, cy, w, h, obj, confs) in enumerate(entries):
        p[m, :5] = (cx, cy, w, h, obj)
        for c, v in confs.items():
            p[m, 5 + c] = v
    return p


def _run(entries, C, conf, thr):
    rows = spec.postprocess(_pred(entries, C)[None], C, conf, thr)[0]
    return [] if rows is None else [(tuple(float(v) for v in r[:4]), int(r[6]), float(r[5])) for r in rows]


def test_same_box_in_several_classes_keeps_its_best_class():
    # box 0 passes in classes 1 (0.9), 3 (0.6) and 5 (0.95); box 1, far away, in classes 1 and 3
    e = [(50, 50, 20, 20, 1.0, {1: 0.9, 3: 0.6, 5: 0.95}), (200, 200, 10, 10, 0.5, {1: 0.5, 3: 0.8})]
    got = _run(e, 6, 0.1, 0.5)
    assert [(c, v) for _, c, v in got] == [(3, np.float32(0.8)), (5, np.float32(0.95))]
    # per-class NMS keeps all five pairs
    assert len(spec.postprocess(_pred(e, 6)[None], 6, 0.1, 0.5, agnostic=False)[0]) == 5


def test_overlap_across_classes_suppresses():
    # two different boxes with IoU 0.81 in different classes: the higher score wins, the other is dropped
    e = [(50, 50, 20, 20, 1.0, {0: 0.7}), (51, 51, 20, 20, 1.0, {2: 0.9})]
    assert [c for _, c, _ in _run(e, 3, 0.1, 0.5)] == [2]
    assert sorted(c for _, c, _ in _run(e, 3, 0.1, 0.9)) == [0, 2]


def test_score_ties_across_classes_lower_class_first():
    # one box, equal scores in classes 4 and 2: the lower class is first in the image-wide order and keeps the box
    e = [(50, 50, 20, 20, 0.5, {4: 0.5, 2: 0.5})]
    assert [c for _, c, _ in _run(e, 5, 0.1, 0.5)] == [2]
    # two overlapping boxes, equal scores, classes 3 and 1: class 1 wins even though its box row is lower
    e = [(50, 50, 20, 20, 0.5, {3: 0.5}), (52, 50, 20, 20, 0.5, {1: 0.5})]
    assert [c for _, c, _ in _run(e, 4, 0.1, 0.5)] == [1]


def test_score_ties_inside_a_class_higher_row_first():
    e = [(50, 50, 20, 20, 0.5, {1: 0.5}), (52, 50, 20, 20, 0.5, {1: 0.5})]
    got = _run(e, 2, 0.1, 0.5)
    assert len(got) == 1 and got[0][0][0] == 42.0              # row 1 (cx 52) precedes row 0


def test_degenerate_boxes_keep_every_copy():
    nan, inf = np.float32(np.nan), np.float32(np.inf)
    e = [(nan, 50, 20, 20, 1.0, {0: 0.9, 1: 0.8}),          # NaN coordinate
         (100, 100, 0, 0, 1.0, {0: 0.9, 1: 0.8}),           # zero area
         (150, 150, -4, 6, 1.0, {0: 0.9, 1: 0.8}),          # negative extent
         (200, 200, inf, 10, 1.0, {0: 0.9, 1: 0.8}),        # infinite extent
         (300, 300, 3e38, 3e38, 1.0, {0: 0.9, 1: 0.8})]     # finite extents, overflowing area
    got = _run(e, 2, 0.1, 0.5)
    assert len(got) == 10                                     # self-IoU below thr (NaN or 0): no copy suppresses another
    # a regular box next to them still loses its second label
    got = _run(e + [(400, 400, 10, 10, 1.0, {0: 0.9, 1: 0.8})], 2, 0.1, 0.5)
    assert len(got) == 11


def test_thresholds_le_zero_one_and_above_one():
    e = [(50, 50, 20, 20, 1.0, {0: 0.9, 1: 0.8}), (500, 500, 20, 20, 1.0, {1: 0.7}),
         (150, 150, -4, 6, 1.0, {0: 0.6, 1: 0.5}), (np.nan, 50, 20, 20, 1.0, {0: 0.4})]
    # thr <= 0: disjoint boxes have IoU 0 >= thr, and a negative-extent box has IoU -0 against itself; only NaN escapes
    for thr in (0.0, -0.5):
        assert sorted((c, v) for _, c, v in _run(e, 2, 0.1, thr)) == [(0, np.float32(0.4)), (0, np.float32(0.9))]
    # thr = 1: only identical boxes suppress each other
    assert len(_run(e, 2, 0.1, 1.0)) == 5
    # thr > 1: nothing is suppressed, every candidate is kept
    assert len(_run(e, 2, 0.1, 1.5)) == 6


def _pathological(seed, B=2, M=400, C=6):
    rng = np.random.RandomState(seed)
    pred = np.zeros((B, M, 5 + C), np.float32)
    pred[..., 0:2] = rng.rand(B, M, 2) * 100
    pred[..., 2:4] = rng.rand(B, M, 2) * 40
    pred[..., 4] = rng.rand(B, M)
    pred[..., 5:] = rng.rand(B, M, C) ** 3
    pred[0, 0:20, 2:4] = 0.0
    pred[0, 5:10, 0:2] = pred[0, 0:5, 0:2]
    pred[0, 30, 0] = np.nan
    pred[0, 31, 2] = np.inf
    pred[0, 32, 5 + C - 1] = np.nan
    pred[1, 40, 4] = np.nan
    pred[1, 41, 4] = -0.5
    pred[1, 50:60, :] = pred[1, 60:70, :]
    pred[1, 70:75, 4] = -2.0
    pred[1, 70:75, 5:] = -0.75
    return pred


def _bits_equal(a, b):
    return (a is None and b is None) or (a is not None and b is not None and a.shape == b.shape and
                                         np.array_equal(a.view(np.uint32), b.view(np.uint32)))


@pytest.mark.parametrize("conf,thr", [(0.05, 0.45), (0.3, 0.0001), (0.0, 0.5), (0.05, 0.0), (0.05, -1.0), (0.05, 1.0), (0.05, 1.5)])
def test_spec_per_class_mode_equals_the_oracle(conf, thr):
    """The spec's candidate filter and greedy pass, run per class, reproduce the C oracle's postprocess bit for bit."""
    pred = _pathological(7)
    want = orc.postprocess(pred, 6, conf, thr)
    got = spec.postprocess(pred, 6, conf, thr, agnostic=False)
    assert all(_bits_equal(g, w) for g, w in zip(got, want))


@pytest.mark.parametrize("thr", [0.45, 0.0, 1.0])
def test_one_class_agnostic_equals_per_class(thr):
    pred = _pathological(8, C=1)
    want = orc.postprocess(pred, 1, 0.05, thr)
    got = spec.postprocess(pred, 1, 0.05, thr)
    assert all(_bits_equal(g, w) for g, w in zip(got, want))


def test_agnostic_rows_are_a_subset_in_the_usual_order():
    pred = _pathological(9)
    for b, rows in enumerate(spec.postprocess(pred, 6, 0.05, 0.45)):
        cand = spec.candidates(pred[b], 6, 0.05)
        allr = spec.rows_of(cand, np.arange(len(cand["s"])))
        pos = [np.nonzero((allr.view(np.uint32) == r.view(np.uint32)).all(1))[0][0] for r in rows]
        assert pos == sorted(pos)                             # the order of the full candidate list, restricted
        assert len(rows) <= len(np.unique(cand["row"])) + 5    # at most one label per regular box (5 degenerate ones)


# ---- argument validation --------------------------------------------------------------------------------------------
def _lib():
    from yolov4_b200 import _cabi
    return _cabi, _cabi.lib()


def test_workspace_query():
    _, L = _lib()
    base = L.yl_post_workspace_bytes(2, 1000, 80, 64)
    assert L.yl_post_workspace_bytes_ex(2, 1000, 80, 64, 0) == base
    assert L.yl_post_workspace_bytes_ex(2, 1000, 80, 64, 1) >= base + 8 * 2 * 80 * 64
    for bad in (-1, 2, 7):
        assert L.yl_post_workspace_bytes_ex(2, 1000, 80, 64, bad) == 0


@pytest.mark.parametrize("agnostic", [-1, 2, 255])
def test_nms_ex_rejects_bad_agnostic(agnostic):
    _, L = _lib()
    ws_bytes = L.yl_post_workspace_bytes_ex(2, 1000, 80, 64, 1)
    # every other argument is well formed (pointers are never dereferenced on the host), so only agnostic can be refused
    assert L.yl_nms_ex(4096, ws_bytes, 2, 1000, 80, 64, 0.5, 0, agnostic, 4096, 16, 4096, None, 0, 2, None) == 1


def test_nms_ex_rejects_agnostic_limits_and_small_workspace():
    _, L = _lib()
    big_m = 1 << 25                                           # box rows must fit 25 bits
    ws = L.yl_post_workspace_bytes_ex(1, big_m, 2, 64, 1)
    assert L.yl_nms_ex(4096, ws, 1, big_m, 2, 64, 0.5, 0, 1, 4096, 16, 4096, None, 0, 1, None) == 1
    small = L.yl_post_workspace_bytes(2, 1000, 80, 64)       # enough for per-class NMS, not for the agnostic scratch
    assert L.yl_nms_ex(4096, small, 2, 1000, 80, 64, 0.5, 0, 1, 4096, 16, 4096, None, 0, 2, None) == 3


def test_detect_host_ex_rejects_null_context():
    _cabi, L = _lib()
    rows = np.zeros((1, 16, 7), np.float32)
    counts = np.zeros((1,), np.int32)
    ptrs = _cabi.ptrs([4096, 4096, 4096])
    assert L.yl_detect_host_ex(None, ptrs, 0.5, 0.5, 0, 1, rows.ctypes.data, counts.ctypes.data) == 1
    assert L.yl_detect_host_ex(None, ptrs, 0.5, 0.5, 0, 2, rows.ctypes.data, counts.ctypes.data) == 1


@pytest.mark.parametrize("bad", [1, 0, None, "yes", np.bool_(True), 1.0])
def test_wrappers_reject_non_bool_agnostic_before_any_cuda_work(bad):
    import yolov4_b200 as yb
    # CPU tensors: a wrapper that got past the agnostic check would raise TypeError for the tensors, with another message
    with pytest.raises(TypeError, match="agnostic"):
        yb.detect_raw([torch.zeros(1, 255, 4, 4)], 80, 0.5, 0.5, agnostic=bad)
    with pytest.raises(TypeError, match="agnostic"):
        yb.postprocess(torch.zeros(1, 10, 85), 80, 0.5, 0.5, agnostic=bad)
    with pytest.raises(TypeError, match="agnostic"):
        yb.HeadPostprocessor(1, [8, 4, 2], 80, 0.5, 0.5, device="cuda", agnostic=bad)
