"""fp16 / bf16 head tensors in the fused training loss.  A 16-bit head is widened exactly to fp32 on load, so the four components
must equal those of the fp32 path on h.float() up to the order of the fp64 sums, and the gradient, written in the head's dtype,
must be bit for bit the fp32 path's gradient on the widened heads rounded to the dtype (g32.to(dt); any NaN equals any NaN)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as orc                                     # noqa: E402  (checker only)
import yolov4_b200 as yb                                              # noqa: E402
from yolov4_b200 import _cabi                                         # noqa: E402
from yolov4_b200.synth import synth_head_outputs, synth_labels        # noqa: E402
from yolov4_b200.yololoss import fused_yolo_loss, fused_yolo_loss_components  # noqa: E402

DTYPES = [torch.float16, torch.bfloat16]
CODES = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}


def cfg_for(C):
    return {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": C}


def bit_equal16(a, b):
    """Bitwise equality of two 16-bit tensors of one dtype, except that any NaN equals any NaN."""
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    na, nb = torch.isnan(a), torch.isnan(b)
    return bool(torch.equal(na, nb) and torch.equal(a.view(torch.int16)[~na], b.view(torch.int16)[~nb]))


def loss_and_grads(heads, labels, cfg, up):
    """fused_yolo_loss on leaf copies of `heads`, back-propagated with the upstream gradient `up`."""
    hs = [h.detach().clone().requires_grad_(True) for h in heads]
    loss = fused_yolo_loss(hs, labels, cfg, 0.7)
    loss.backward(torch.tensor(up, dtype=torch.float32, device="cuda"))
    return loss.detach(), [h.grad for h in hs]


def check_against_widened(heads16, labels, cfg, ups=(1.0,)):
    """Components within rtol 1e-12 of the fp32 path on the widened heads; for every upstream gradient, the 16-bit gradient is
    g32.to(dt) bit for bit.  Returns (components, {up: (16-bit loss, 16-bit grads)})."""
    dt = heads16[0].dtype
    wide = [h.float() for h in heads16]
    c16 = fused_yolo_loss_components(heads16, labels, cfg, 0.7)
    c32 = fused_yolo_loss_components(wide, labels, cfg, 0.7)
    np.testing.assert_allclose(c16.cpu().numpy(), c32.cpu().numpy(), rtol=1e-12, atol=0, equal_nan=True)
    out = {}
    for up in ups:
        l16, g16 = loss_and_grads(heads16, labels, cfg, up)
        l32, g32 = loss_and_grads(wide, labels, cfg, up)
        assert l16.dtype == torch.float32 and l16.dim() == 0
        np.testing.assert_allclose(l16.item(), l32.item(), rtol=1e-6, equal_nan=True)
        for l, (g, w) in enumerate(zip(g16, g32)):
            assert g.dtype == dt and w.dtype == torch.float32 and g.shape == w.shape, (l, g.dtype, g.shape)
            assert bit_equal16(g, w.to(dt)), "layer %d, upstream %r: gradient differs from g32.to(%s)" % (l, up, dt)
        out[up] = (l16, g16)
    return c16, out


def oracle_loss(wide_np, labels_np, C, layers=(0, 1, 2)):
    return sum(orc.yolo_loss_layer(w, labels_np, l, C, 0.7)[0].sum() for w, l in zip(wide_np, layers))


@pytest.mark.parametrize("dt", DTYPES)
def test_608_b4_matches_widened_fp32_and_oracle(dt):
    heads = [r.to(dt) for r in synth_head_outputs(4, 608, 80, seed=77, device="cuda")]
    labels = synth_labels(4, 608, n_valid=50, seed=78, device="cuda")
    _, res = check_against_widened(heads, labels, cfg_for(80))
    loss = res[1.0][0].item()
    want = oracle_loss([h.float().cpu().numpy() for h in heads], labels.cpu().numpy(), 80)
    assert abs(loss - want) <= 1e-5 * abs(want), (loss, want)


@pytest.mark.parametrize("dt", DTYPES)
def test_golden_inputs_cast_to_16_bit(dt, golden_dir):
    import os
    g = np.load(os.path.join(golden_dir, "loss.npz"))
    C = int(g["C"])
    heads = [torch.from_numpy(g[f"raw{l}"]).cuda().to(dt) for l in range(3)]
    labels = torch.from_numpy(g["labels"]).cuda()
    _, res = check_against_widened(heads, labels, cfg_for(C))
    loss = res[1.0][0].item()
    want = oracle_loss([h.float().cpu().numpy() for h in heads], g["labels"], C)
    assert abs(loss - want) <= 1e-5 * abs(want), (loss, want)


_SPECIALS = {
    # NaN (quiet, signalling, negative), +-inf, largest finite, smallest / largest subnormal, -0 (as in test_gpu_half_inputs.py)
    torch.float16: [0x7E00, 0x7C01, 0xFE00, 0x7C00, 0xFC00, 0x7BFF, 0xFBFF, 0x0001, 0x8001, 0x03FF, 0x8000],
    torch.bfloat16: [0x7FC0, 0x7FC1, 0xFFC0, 0x7F81, 0x7F80, 0xFF80, 0x7F7F, 0xFF7F, 0x7F62, 0x0001, 0x8001, 0x007F, 0x8000],
}


def _is_nan_bits(v, dt):
    e = (v >> 10) & 0x1F if dt == torch.float16 else (v >> 7) & 0xFF
    m = v & (0x3FF if dt == torch.float16 else 0x7F)
    return e == (0x1F if dt == torch.float16 else 0xFF) and m != 0


def _degenerate_labels(C, bad_class):
    """The label rows of the pathological build_target test (zero / negative extent, inf, 1e30, NaN) among ordinary boxes of
    classes 0..7; with bad_class, one ordinary box carries a class id outside [0, C)."""
    img, B, K, n = 160, 2, 16, 12
    rng = np.random.RandomState(5)
    labels = np.zeros((B, K, 5), np.float32)
    for b in range(B):
        labels[b, :n, 0:2] = rng.uniform(4, img - 4, (n, 2))
        labels[b, :n, 2:4] = np.exp(rng.uniform(np.log(4.0), np.log(img * 0.8), (n, 2)))
        labels[b, :n, 4] = rng.randint(0, 8, n)
    labels[0, 2, 2:4] = labels[0, 1, 2:4]
    labels[1, 1, 2] = np.inf
    labels[1, 4, 3] = 1e30
    labels[1, 5, 2] = 0.0
    labels[0, 6, 2] = -20.0
    labels[0, 7, 2:4] = (-20.0, -30.0)
    labels[1, 8, 3] = np.nan
    if bad_class:
        labels[0, 9, 2:4] = (40.0, 50.0)
        labels[0, 9, 4] = C + 5
    return torch.from_numpy(labels).cuda()


def _plant_specials(heads, dt, C, with_nan):
    """Special bit patterns in the tx / ty / tw / th / objectness planes (every other cell) and in the class channels 0..7 and
    C-1 of every cell, so the matched cells carry them too."""
    vals = [v for v in _SPECIALS[dt] if with_nan or not _is_nan_bits(v, dt)]
    vals = [v - 0x10000 if v >= 0x8000 else v for v in vals]                 # the bit patterns as int16
    n = len(vals)
    for l, h in enumerate(heads):
        F2 = h.shape[2] * h.shape[3]
        bits = h.view(torch.int16).view(h.shape[0], 3, 5 + C, F2)
        cells = torch.arange(F2, device="cuda")
        table = torch.tensor(vals, dtype=torch.int16, device="cuda")
        for b in range(h.shape[0]):
            for a in range(3):
                for ch in range(5):
                    sel = cells[(cells + ch + a + b) % 2 == 0]
                    bits[b, a, ch, sel] = table[(sel // 2 + ch + 3 * a + l) % n]
                for c in list(range(8)) + [C - 1]:
                    bits[b, a, 5 + c] = table[(cells + c + a + b + l) % n]


def _forward_status(heads, lab, C):
    """The typed C forward on the three heads with a status buffer: (loss4, status)."""
    L = _cabi.lib()
    code = CODES[heads[0].dtype]
    B, K = int(lab.shape[0]), int(lab.shape[1])
    loss4 = torch.zeros(4, dtype=torch.float64, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    anch = _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh])
    keep = []
    for l, r in enumerate(heads):
        F = int(r.shape[2])
        bufs = (torch.empty((B, 3, F, F), dtype=torch.float32, device="cuda"), torch.empty((B, K), dtype=torch.int32, device="cuda"),
                torch.empty((B, K), dtype=torch.int32, device="cuda"), torch.empty((B, K, 4 + C), dtype=torch.float32, device="cuda"))
        keep.append(bufs)
        fn = L.yl_loss_forward_typed if l == 0 else L.yl_loss_forward_chained_typed
        _cabi.check(fn(r.data_ptr(), code, lab.data_ptr(), B, F, K, C, l, anch, _cabi.ints(yb.ANCHOR_MASK[l]), float(np.float32(0.7)),
                       loss4.data_ptr(), bufs[0].data_ptr(), bufs[1].data_ptr(), bufs[2].data_ptr(), bufs[3].data_ptr(),
                       status.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return loss4, int(status.item())


@pytest.mark.parametrize("with_nan", [True, False])
@pytest.mark.parametrize("dt", DTYPES)
def test_special_values_and_degenerate_labels(dt, with_nan):
    C = 80
    heads = [r.to(dt) for r in synth_head_outputs(2, 160, C, seed=7, device="cuda", fg_prob=0.1, clustered=True)]
    _plant_specials(heads, dt, C, with_nan)
    for bad_class in (False, True):
        labels = _degenerate_labels(C, bad_class)
        check_against_widened(heads, labels, cfg_for(C), ups=(1.0, 65536.0))
        statuses = [_forward_status(hs, labels, C)[1] for hs in (heads, [h.float() for h in heads])]
        assert statuses[0] == statuses[1], statuses
        if bad_class:
            assert statuses[0] == 1, "a matched GT with a class id outside [0, C) must set status"


@pytest.mark.parametrize("dt", DTYPES)
def test_loss_scale_and_overflow(dt):
    heads = [r.to(dt) for r in synth_head_outputs(2, 608, 80, seed=31, device="cuda")]
    labels = synth_labels(2, 608, n_valid=50, seed=32, device="cuda")
    big = 2.0 ** 24 if dt == torch.float16 else float(np.finfo(np.float32).max)
    _, res = check_against_widened(heads, labels, cfg_for(80), ups=(1.0, 65536.0, big))
    # check_against_widened compared every gradient bit for bit with g32.to(dt), so the inf positions and signs are those of g32
    assert any(bool(torch.isinf(g).any()) for g in res[big][1]), "the large scale must overflow some gradients"
    assert not any(bool(torch.isinf(g).any()) for g in res[1.0][1])


@pytest.mark.parametrize("dt", DTYPES)
def test_under_autocast_with_grad_scaler(dt):
    torch.manual_seed(0)
    B, img, C, cin = 2, 416, 80, 16
    Fs = [img // 8, img // 16, img // 32]
    xs = [torch.randn(B, cin, F, F, device="cuda") for F in Fs]
    convs = [torch.nn.Conv2d(cin, 3 * (5 + C), 1).cuda() for _ in Fs]
    opt = torch.optim.SGD([p for c in convs for p in c.parameters()], lr=1e-3)
    labels = synth_labels(B, img, n_valid=30, seed=5, device="cuda")
    scaler = torch.amp.GradScaler("cuda")
    with torch.autocast("cuda", dtype=dt):
        heads = [conv(x) for conv, x in zip(convs, xs)]
        for h in heads:
            h.retain_grad()
        loss = fused_yolo_loss(heads, labels, cfg_for(C), 0.7)
        comps = fused_yolo_loss_components(heads, labels, cfg_for(C), 0.7)
    assert all(h.dtype == dt for h in heads) and loss.dtype == torch.float32
    np.testing.assert_allclose(comps.cpu().numpy(), fused_yolo_loss_components([h.detach().float() for h in heads], labels,
                                                                                cfg_for(C), 0.7).cpu().numpy(), rtol=1e-12)
    scaler.scale(loss).backward()
    up = float(scaler.get_scale())
    _, g32 = loss_and_grads([h.detach().float() for h in heads], labels, cfg_for(C), up)
    for h, w in zip(heads, g32):
        assert h.grad.dtype == dt
        assert bit_equal16(h.grad, w.to(dt))
    assert all(c.weight.grad is not None and c.weight.grad.dtype == torch.float32 for c in convs)
    scaler.step(opt)
    scaler.update()
    assert all(torch.isfinite(c.weight).all() for c in convs)


@pytest.mark.parametrize("dt", DTYPES)
def test_graph_replay_matches_eager(dt):
    """The fp32 graph-replay test with 16-bit heads: the scales' kernels overlap (programmatic dependent launch) and the caching
    allocator would reuse a freed per-scale buffer inside the graph."""
    B = 16
    heads = [r.to(dt) for r in synth_head_outputs(B, 608, 80, seed=41, device="cuda")]
    labels = synth_labels(B, 608, n_valid=50, seed=42, device="cuda")
    eager = fused_yolo_loss_components(heads, labels, cfg_for(80), 0.7).clone()
    wide = fused_yolo_loss_components([h.float() for h in heads], labels, cfg_for(80), 0.7)
    np.testing.assert_allclose(eager.cpu().numpy(), wide.cpu().numpy(), rtol=1e-12, atol=0)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fused_yolo_loss_components(heads, labels, cfg_for(80), 0.7)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fused_yolo_loss_components(heads, labels, cfg_for(80), 0.7)
    for _ in range(5):
        g.replay()
        torch.cuda.synchronize()
        assert torch.allclose(out, eager, rtol=1e-12, atol=0), (out.tolist(), eager.tolist())


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("img,C,B", [(416, 80, 3), (96, 4, 5), (64, 128, 2)])
def test_odd_shapes(dt, img, C, B):
    heads = [r.to(dt) for r in synth_head_outputs(B, img, C, seed=img + C, device="cuda", fg_prob=0.05, clustered=True)]
    labels = synth_labels(B, img, n_valid=min(50, img // 4), n_classes=C, seed=img, device="cuda")
    labels[..., 2:4].clamp_(max=img * 0.6)
    if img == 416:
        assert heads[2].shape[2] == 13 and heads[2][0, 1].data_ptr() % 4 == 2        # 13x13 planes at 2-byte alignment
    check_against_widened(heads, labels, cfg_for(C), ups=(1.0, 1024.0))


def test_mixed_dtypes_raise_before_cuda_work():
    a = torch.zeros(1, 255, 8, 8, device="cuda", dtype=torch.float16)
    b = torch.zeros(1, 255, 4, 4, device="cuda", dtype=torch.bfloat16)
    c = torch.zeros(1, 255, 2, 2, device="cuda", dtype=torch.float16)
    labels = torch.zeros(1, 60, 5, device="cuda")
    for heads in ([a, b, c], [a.float(), b.half(), c], [a.double(), b.double(), c.double()]):
        with pytest.raises(TypeError):
            fused_yolo_loss(heads, labels, cfg_for(80))
        with pytest.raises(TypeError):
            fused_yolo_loss_components(heads, labels, cfg_for(80))
