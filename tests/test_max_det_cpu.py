"""CPU-only checks of the per-image detection cap (max_det): argument validation of the C ABI and of the Python wrappers
happens before any CUDA call, and the spec function cap_spec.cap_detections behaves as stated on hand-built lists."""
import numpy as np
import pytest
import torch

from cap_spec import cap_detections


def _lib():
    from yolov4_b200 import _cabi
    return _cabi, _cabi.lib()


@pytest.mark.parametrize("max_det,cap_out", [(-1, 16), (-100, 16), (17, 16), (4097, 4096)])
def test_nms_topk_rejects_out_of_range_max_det(max_det, cap_out):
    _cabi, L = _lib()
    ws_bytes = L.yl_post_workspace_bytes(2, 1000, 80, 64)
    # every other argument is well formed (pointers are never dereferenced on the host), so only max_det can be refused
    assert L.yl_nms_topk(4096, ws_bytes, 2, 1000, 80, 64, 0.5, max_det, 4096, cap_out, 4096, 4096, 0, 2, None) == 1


def test_nms_topk_rejects_null_pointers():
    _cabi, L = _lib()
    ws_bytes = L.yl_post_workspace_bytes(2, 1000, 80, 64)
    assert L.yl_nms_topk(None, ws_bytes, 2, 1000, 80, 64, 0.5, 8, 4096, 16, 4096, None, 0, 2, None) == 1
    assert L.yl_nms_topk(4096, ws_bytes, 2, 1000, 80, 64, 0.5, 8, None, 16, 4096, None, 0, 2, None) == 1
    assert L.yl_nms_topk(4096, ws_bytes, 2, 1000, 80, 64, 0.5, 8, 4096, 16, None, None, 0, 2, None) == 1


def test_detect_host_topk_rejects_null_context():
    _cabi, L = _lib()
    rows = np.zeros((1, 16, 7), np.float32)
    counts = np.zeros((1,), np.int32)
    ptrs = _cabi.ptrs([4096, 4096, 4096])
    assert L.yl_detect_host_topk(None, ptrs, 0.5, 0.5, 8, rows.ctypes.data, counts.ctypes.data) == 1


@pytest.mark.parametrize("bad", [0, -1, 2.5, True, "3"])
def test_wrappers_reject_bad_max_det_before_any_cuda_work(bad):
    import yolov4_b200 as yb
    # CPU tensors: a wrapper that got past the max_det check would raise TypeError instead
    with pytest.raises(ValueError):
        yb.detect_raw([torch.zeros(1, 255, 4, 4)], 80, 0.5, 0.5, max_det=bad)
    with pytest.raises(ValueError):
        yb.postprocess(torch.zeros(1, 10, 85), 80, 0.5, 0.5, max_det=bad)
    with pytest.raises(ValueError):
        yb.HeadPostprocessor(1, [8, 4, 2], 80, 0.5, 0.5, device="cuda", max_det=bad)


def _row(cls, obj, conf, tag):
    # the box columns carry a tag so the test can tell rows apart
    return [tag, 0.0, 1.0, 1.0, obj, conf, float(cls)]


def test_cap_detections_ties_across_and_inside_classes():
    # uncapped order: class ascending, score descending inside a class; scores 0.5, 0.25, 0.25 | 0.25, 0.25 | 0.125
    r = np.array([_row(0, 1.0, 0.5, 0), _row(0, 0.5, 0.5, 1), _row(0, 1.0, 0.25, 2),
                  _row(3, 0.25, 1.0, 3), _row(3, 0.5, 0.5, 4), _row(5, 0.5, 0.25, 5)], np.float32)
    def tags(out):
        return [int(t) for t in out[0][:, 0]]
    assert tags(cap_detections([r], 1)) == [0]
    assert tags(cap_detections([r], 2)) == [0, 1]              # the tie run starts: class 0's first tie
    assert tags(cap_detections([r], 3)) == [0, 1, 2]           # both class-0 ties before class 3's
    assert tags(cap_detections([r], 4)) == [0, 1, 2, 3]        # inside class 3 the first tie wins
    assert tags(cap_detections([r], 5)) == [0, 1, 2, 3, 4]     # the lower score of class 5 is cut
    for k in (6, 7, 1000):
        assert np.array_equal(cap_detections([r], k)[0], r)


def test_cap_detections_signed_zero_ties_and_order():
    # -0 and +0 scores tie; the kept rows stay in the uncapped order, not re-sorted by score
    r = np.array([_row(0, 0.0, 1.0, 0), _row(1, 1.0, 0.75, 1), _row(2, -0.0, 1.0, 2), _row(2, 0.0, 0.5, 3)], np.float32)
    assert np.signbit(r[2, 4]) and (r[2, 4] * r[2, 5]) == 0.0
    out = cap_detections([r], 2)[0]
    assert [int(t) for t in out[:, 0]] == [0, 1]                   # score 0.75, then the first of the zero-score ties
    out = cap_detections([r], 3)[0]
    assert [int(t) for t in out[:, 0]] == [0, 1, 2]                # -0 ties with +0: row order decides


def test_cap_detections_none_images_k1_and_tensors():
    a = np.array([_row(0, 0.9, 0.9, 0), _row(1, 1.0, 0.95, 1)], np.float32)
    out = cap_detections([None, a, torch.from_numpy(a), None], 1)
    assert out[0] is None and out[3] is None
    assert [int(t) for t in out[1][:, 0]] == [1] and np.array_equal(out[1], out[2])
    assert out[1].dtype == np.float32 and out[1].shape == (1, 7)


def test_cap_detections_matches_the_numpy_spec_on_random_rows():
    rng = np.random.default_rng(0)
    for trial in range(20):
        n = int(rng.integers(1, 200))
        # few distinct values, so ties are common across and inside classes
        r = np.zeros((n, 7), np.float32)
        r[:, 0] = np.arange(n)
        r[:, 4] = rng.choice([0.25, 0.5, 1.0], n)
        r[:, 5] = rng.choice([0.25, 0.5, 1.0], n)
        r[:, 6] = np.sort(rng.integers(0, 5, n))
        for k in (1, 7, n // 2 + 1, n, n + 1):
            got = cap_detections([r], k)[0]
            s = r[:, 4] * r[:, 5]
            keep = np.sort(np.argsort(-s, kind="stable")[:k])
            assert np.array_equal(got, r[keep])
            assert got.shape[0] == min(n, k)
            # the kept scores are the k largest
            assert np.sort(s[keep])[::-1].tolist() == np.sort(s)[::-1][:min(n, k)].tolist()
