"""CPU-only checks of the 16-bit fused-loss entry points: the typed C calls refuse an unknown dtype before any CUDA call, and the
Python wrappers reject mixed dtypes, float64 and CPU heads before any CUDA work."""
import pytest
import torch


def _args():
    from yolov4_b200 import _cabi
    import yolov4_b200 as yb
    anch = _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh])
    return _cabi, anch, _cabi.ints(yb.ANCHOR_MASK[0])


# non-null dummy pointers (never dereferenced on the host): every other argument is well formed, so only the dtype can be refused
P = 4096


@pytest.mark.parametrize("dtype", [3, -1])
@pytest.mark.parametrize("name", ["yl_loss_forward_typed", "yl_loss_forward_chained_typed"])
def test_loss_forward_typed_rejects_unknown_dtype(name, dtype):
    _cabi, anch, mask = _args()
    fn = getattr(_cabi.lib(), name)
    assert fn(P, dtype, P, 2, 76, 60, 80, 0, anch, mask, 0.7, P, P, P, P, P, P, None) == 1


@pytest.mark.parametrize("dtype", [3, -1])
def test_loss_backward_typed_rejects_unknown_dtype(dtype):
    _cabi, _, _ = _args()
    assert _cabi.lib().yl_loss_backward_typed(P, P, P, P, 2, 76, 60, 80, P, dtype, None) == 1


def test_loss_typed_entries_still_validate_their_other_arguments():
    _cabi, anch, mask = _args()
    L = _cabi.lib()
    for code in (0, 1, 2):
        assert L.yl_loss_forward_typed(None, code, P, 2, 76, 60, 80, 0, anch, mask, 0.7, P, P, P, P, P, P, None) == 1
        assert L.yl_loss_forward_typed(P, code, P, 2, 76, 300, 80, 0, anch, mask, 0.7, P, P, P, P, P, P, None) == 1   # K > 256
        assert L.yl_loss_backward_typed(P, P, P, P, 0, 76, 60, 80, P, code, None) == 1
        assert L.yl_loss_backward_typed(P, P, P, P, 2, 76, 60, 80, None, code, None) == 1


def _cfg():
    import yolov4_b200 as yb
    return {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": 80}


def _bad_head_sets():
    h = lambda F, dt: torch.zeros(1, 255, F, F, dtype=dt)             # noqa: E731
    return {
        "cpu fp32": [h(8, torch.float32), h(4, torch.float32), h(2, torch.float32)],
        "cpu fp16": [h(8, torch.float16), h(4, torch.float16), h(2, torch.float16)],
        "cpu bf16": [h(8, torch.bfloat16), h(4, torch.bfloat16), h(2, torch.bfloat16)],
        "float64": [h(8, torch.float64), h(4, torch.float64), h(2, torch.float64)],
        "mixed": [h(8, torch.float16), h(4, torch.bfloat16), h(2, torch.float16)],
        "mixed with fp32": [h(8, torch.float32), h(4, torch.float16), h(2, torch.float32)],
    }


@pytest.mark.parametrize("case", list(_bad_head_sets()))
def test_fused_loss_wrappers_reject_before_cuda_work(case):
    from yolov4_b200.yololoss import fused_yolo_loss, fused_yolo_loss_components
    heads = _bad_head_sets()[case]
    labels = torch.zeros(1, 60, 5, dtype=torch.float64)
    with pytest.raises(TypeError):
        fused_yolo_loss(heads, labels, _cfg())
    with pytest.raises(TypeError):
        fused_yolo_loss([h.requires_grad_(True) for h in heads], labels, _cfg())
    with pytest.raises(TypeError):
        fused_yolo_loss_components(heads, labels, _cfg())
