"""fp16 / bf16 head tensors in the fused detection path: a 16-bit head is widened exactly to fp32, so detect_raw on it must
equal detect_raw on h.float() and the oracle on the widened arrays bit for bit (rows and counts)."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as orc                                     # noqa: E402  (checker only)
import yolov4_b200 as yb                                              # noqa: E402
from yolov4_b200 import _cabi                                         # noqa: E402
from yolov4_b200.synth import synth_head_outputs                      # noqa: E402

DTYPES = [torch.float16, torch.bfloat16]
CFG80 = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": 80}


def bit_equal(a, b):
    """Bitwise equality of fp32 arrays, except that any NaN equals any NaN."""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a.view(np.uint32)[~na], b.view(np.uint32)[~nb]))


def assert_lists_bit_equal(got, ref, what=""):
    assert len(got) == len(ref), what
    for b, (g, r) in enumerate(zip(got, ref)):
        assert (g is None) == (r is None), f"{what} image {b}: None mismatch"
        if r is None:
            continue
        g = g.detach().cpu().numpy() if isinstance(g, torch.Tensor) else g
        r = r.detach().cpu().numpy() if isinstance(r, torch.Tensor) else r
        assert g.dtype == np.float32 and g.shape == r.shape, f"{what} image {b}: {g.dtype} {g.shape} vs {r.shape}"
        assert bit_equal(g, r), f"{what} image {b}: rows differ"


def check_parity(h16, C, conf, nmst, what=""):
    """detect_raw(h16) == detect_raw(widened) == oracle(widened); returns the oracle's result."""
    wide = [h.float() for h in h16]
    got = yb.detect_raw(h16, C, conf, nmst)
    assert_lists_bit_equal(got, yb.detect_raw(wide, C, conf, nmst), what=f"{what} vs widened fp32")
    want = orc.detect([w.cpu().numpy() for w in wide], C, conf, nmst, nthreads=8)
    assert_lists_bit_equal(got, want, what=f"{what} vs oracle")
    return want


def to16(raws, dt):
    return [r.to(dt) for r in raws]


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("img,B,seed,clustered,conf,nmst", [(608, 4, 0, False, 1e-4, 0.4), (608, 2, 1, True, 1e-4, 0.4),
                                                          (608, 2, 2, True, 0.2, 0.5), (416, 3, 3, True, 0.01, 0.45)])
def test_parity_with_widened_fp32_and_oracle(dt, img, B, seed, clustered, conf, nmst):
    raws = to16(synth_head_outputs(B, img, 80, seed=seed, device="cuda", clustered=clustered,
                                   fg_prob=0.02 if clustered else 0.005), dt)
    want = check_parity(raws, 80, conf, nmst, what=f"{img} B{B} conf {conf}")
    if clustered and conf < 0.1:
        dense = torch.cat([yb.YOLOLayer(CFG80, l, device="cuda").eval()(r.float()) for l, r in enumerate(raws)], 1)
        n_cand = int(((dense[:, :, 5:] * dense[:, :, 4:5]) >= float(np.float32(conf))).sum())
        assert sum(0 if w is None else len(w) for w in want) < n_cand, "NMS must suppress something in the clustered case"


@pytest.mark.parametrize("dt", DTYPES)
def test_odd_shapes_and_four_flag_words(dt):
    for img, C, B in ((96, 4, 5), (64, 20, 1), (96, 33, 2), (64, 128, 2)):
        raws = to16(synth_head_outputs(B, img, C, seed=img + C, device="cuda", fg_prob=0.05, clustered=True), dt)
        check_parity(raws, C, 0.01, 0.45, what=f"img {img} C {C}")


_SPECIALS = {
    # NaN (quiet, signalling, negative), +-inf, largest finite, smallest / largest subnormal, -0
    torch.float16: [0x7E00, 0x7C01, 0xFE00, 0x7C00, 0xFC00, 0x7BFF, 0xFBFF, 0x0001, 0x8001, 0x03FF, 0x8000],
    # several NaN payloads, +-inf, largest finite (3.39e38) and a value near 3e38, subnormals, -0
    torch.bfloat16: [0x7FC0, 0x7FC1, 0xFFC0, 0x7F81, 0x7F80, 0xFF80, 0x7F7F, 0xFF7F, 0x7F62, 0x0001, 0x8001, 0x007F, 0x8000],
}


@pytest.mark.parametrize("dt", DTYPES)
def test_special_values(dt):
    C = 80
    raws = to16(synth_head_outputs(2, 96, C, seed=7, device="cuda", fg_prob=0.1, clustered=True), dt)
    three = torch.tensor(3.0, dtype=dt).view(torch.int16).item()
    for r in raws:
        F = r.shape[2]
        bits = r.view(torch.int16).view(2, 3, 5 + C, F * F)
        for k, v in enumerate(_SPECIALS[dt]):
            sv = v - 0x10000 if v >= 0x8000 else v                # the bit pattern as int16
            b = k % 2
            for ch, a in ((4, 0), (5 + 7, 1), (0, 2), (2, 1), (5 + 79, 2)):     # objectness, class 7, tx, tw, class 79
                cell = (3 * k + ch) % (F * F)
                if ch != 4:                                   # keep the box alive so the class / box value matters
                    bits[b, a, 4, cell] = three
                bits[b, a, ch, cell] = sv
    for conf, nmst in ((0.001, 0.45), (0.3, 0.5), (0.0, 0.5)):
        check_parity(raws, C, conf, nmst, what=f"special values conf {conf}")


@pytest.mark.parametrize("dt", DTYPES)
def test_unaligned_bases_equal_the_aligned_run(dt):
    raws = to16(synth_head_outputs(2, 416, 80, seed=9, device="cuda", fg_prob=0.02, clustered=True), dt)
    want = yb.detect_raw(raws, 80, 0.01, 0.45)
    assert_lists_bit_equal(want, orc.detect([r.float().cpu().numpy() for r in raws], 80, 0.01, 0.45, nthreads=8))
    for off in (1, 2, 3, 4):
        views = []
        for r in raws:
            buf = torch.empty(r.numel() + 8, dtype=dt, device="cuda")
            v = buf[off:off + r.numel()].view(r.shape)
            v.copy_(r)
            assert v.is_contiguous() and v.data_ptr() % 16 == (2 * off) % 16
            views.append(v)
        assert_lists_bit_equal(yb.detect_raw(views, 80, 0.01, 0.45), want, what=f"offset {off}")


@pytest.mark.parametrize("dt", DTYPES)
def test_channels_last_input_equals_contiguous(dt):
    raws = to16(synth_head_outputs(2, 416, 80, seed=10, device="cuda", fg_prob=0.02, clustered=True), dt)
    cl = [r.contiguous(memory_format=torch.channels_last) for r in raws]
    assert not cl[0].is_contiguous()
    assert_lists_bit_equal(yb.detect_raw(cl, 80, 0.01, 0.45), yb.detect_raw(raws, 80, 0.01, 0.45))


@pytest.mark.parametrize("dt", DTYPES)
def test_all_zero_logits_oversized_segments(dt):
    """Random-init degenerate case: every score is exactly 0.25, segments exceed cap_seg and the capacity grows."""
    raws = [torch.zeros(2, 255, f, f, device="cuda", dtype=dt) for f in (20, 10, 5)]
    raws[0][1, 4] = -20.0
    want = check_parity(raws, 80, 0.2, 0.5)
    assert len(want[0]) > 20000


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("n_groups", [1, 4])
def test_head_postprocessor_graph_replay(dt, n_groups):
    raws = to16(synth_head_outputs(8, 608, 80, seed=11, device="cuda"), dt)
    want = yb.detect_raw(raws, 80, 1e-4, 0.4)
    hp = yb.HeadPostprocessor(8, [76, 38, 19], 80, 1e-4, 0.4, n_groups=n_groups).capture(raws)
    for _ in range(3):
        hp.replay()
    torch.cuda.synchronize()
    assert_lists_bit_equal(hp.results(), want)
    fresh = to16(synth_head_outputs(8, 608, 80, seed=12, device="cuda"), dt)
    for dst, src in zip(hp._captured_inputs, fresh):
        dst.copy_(src)
    hp.replay()
    torch.cuda.synchronize()
    assert_lists_bit_equal(hp.results(), yb.detect_raw(fresh, 80, 1e-4, 0.4))


@pytest.mark.parametrize("dt", DTYPES)
def test_full_size_properties_b64(dt):
    raws = to16(synth_head_outputs(64, 608, 80, seed=0, device="cuda"), dt)
    out = yb.detect_raw(raws, 80, 1e-4, 0.4)
    assert len(out) == 64
    total = 0
    for o in out:
        assert o is not None and o.shape[1] == 7 and o.dtype == torch.float32
        cls = o[:, 6]
        assert torch.all(cls[1:] >= cls[:-1]), "classes ascending"
        score = o[:, 4] * o[:, 5]
        same = cls[1:] == cls[:-1]
        assert torch.all(score[1:][same] <= score[:-1][same]), "score descending inside a class"
        assert torch.all(score >= float(np.float32(1e-4)))
        total += o.shape[0]
    assert 64 * 8000 < total < 64 * 16000
    sub = yb.detect_raw([r[10:14] for r in raws], 80, 1e-4, 0.4)
    for a, b in zip(sub, out[10:14]):
        assert torch.equal(a, b), "image results do not depend on batch composition"
    want = orc.detect([r[:4].float().cpu().numpy() for r in raws], 80, 1e-4, 0.4, nthreads=8)
    assert_lists_bit_equal(out[:4], want)


@pytest.mark.parametrize("dt", DTYPES)
def test_detect_host_c_abi_16bit_buffers(dt):
    L = _cabi.lib()
    B, C = 6, 80
    raws = [r.to(dt) for r in synth_head_outputs(B, 416, C, seed=21, fg_prob=0.02, clustered=True)]
    if dt == torch.float16:
        host = [r.numpy() for r in raws]                                  # numpy float16
        code = 1
    else:
        host = [r.view(torch.int16).numpy().view(np.uint16) for r in raws]  # bfloat16 as its bit patterns
        code = 2
    wide = [r.float().numpy() for r in raws]
    Fs = [r.shape[2] for r in raws]
    ctx = ctypes.c_void_p()
    cap_out = 32768
    anch = _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh])
    mask = _cabi.ints([v for m in yb.ANCHOR_MASK for v in m])
    _cabi.check(L.yl_context_create_typed(ctypes.byref(ctx), 0, B, _cabi.ints(Fs), 3, C, code, anch, mask, 1024, cap_out))
    try:
        rows = np.zeros((B, cap_out, 7), np.float32)
        counts = np.zeros((B,), np.int32)
        ptrs = _cabi.ptrs([h.ctypes.data for h in host])
        for conf, nmst in ((0.001, 0.4), (0.2, 0.5)):
            _cabi.check(L.yl_detect_host(ctx, ptrs, float(np.float32(conf)), float(np.float32(nmst)), rows.ctypes.data,
                                         counts.ctypes.data))
            want = orc.detect(wide, C, conf, nmst, nthreads=8)
            got = [rows[b, :counts[b]] if counts[b] else None for b in range(B)]
            assert_lists_bit_equal(got, want, what=f"host path conf {conf}")
    finally:
        _cabi.check(L.yl_context_destroy(ctx))


def test_wrapper_dtype_errors():
    a = torch.zeros(1, 255, 8, 8, device="cuda", dtype=torch.float16)
    b = torch.zeros(1, 255, 4, 4, device="cuda", dtype=torch.bfloat16)
    with pytest.raises(TypeError):
        yb.detect_raw([a, b], 80)
    with pytest.raises(TypeError):
        yb.detect_raw([a.float(), b.float().half()], 80)
    with pytest.raises(TypeError):
        yb.detect_raw([a.double(), b.double()], 80)
    with pytest.raises(TypeError):
        yb.HeadPostprocessor(1, [8, 4], 80, 0.5, 0.5).run([a, b])
