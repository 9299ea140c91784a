"""CPU-only checks of the 16-bit head-tensor entry points: dtype validation happens before any CUDA call, and the Python
wrappers reject what the fused path does not take."""
import ctypes

import pytest
import torch


def _args():
    from yolov4_b200 import _cabi
    import yolov4_b200 as yb
    anch = _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh])
    mask = _cabi.ints([v for m in yb.ANCHOR_MASK for v in m])
    return _cabi, anch, mask


@pytest.mark.parametrize("dtype", [3, -1, 100])
def test_filter_raw_typed_rejects_unknown_dtype(dtype):
    _cabi, anch, mask = _args()
    L = _cabi.lib()
    Fs = [76, 38, 19]
    M = sum(3 * f * f for f in Fs)
    ws_bytes = L.yl_post_workspace_bytes(1, M, 80, 1024)
    # every other argument is well formed (the pointers are never dereferenced on the host), so only the dtype can be refused
    rp = _cabi.ptrs([4096, 4096, 4096])
    assert L.yl_filter_raw_typed(rp, dtype, _cabi.ints(Fs), 3, 1, 80, anch, mask, 0.5, 4096, ws_bytes, M, 1024, 0, 1, 3,
                                 None) == 1


@pytest.mark.parametrize("dtype", [3, -1])
def test_context_create_typed_rejects_unknown_dtype_before_touching_a_device(dtype):
    _cabi, anch, mask = _args()
    L = _cabi.lib()
    ctx = ctypes.c_void_p()
    assert L.yl_context_create_typed(ctypes.byref(ctx), 0, 2, _cabi.ints([52, 26, 13]), 3, 80, dtype, anch, mask, 1024, 4096) == 1
    assert ctx.value is None


def test_wrappers_reject_16bit_cpu_tensors_and_keep_the_contract_literal_surfaces_fp32():
    import yolov4_b200 as yb
    for dt in (torch.float16, torch.bfloat16):
        with pytest.raises(TypeError):
            yb.detect_raw([torch.zeros(1, 255, 4, 4, dtype=dt)], 80)
        with pytest.raises(TypeError):
            yb.postprocess(torch.zeros(1, 10, 85, dtype=dt), 80)
        cfg = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": 80}
        with pytest.raises(TypeError):
            yb.YOLOLayer(cfg, 0).eval()(torch.zeros(1, 255, 4, 4, dtype=dt))
