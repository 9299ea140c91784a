"""Every dispatch branch of yl_decode.cu against the CPU oracle, bit for bit.

k_decode_dense: tiles with a tail batch or none, one tile or a partial tail tile, tiles over 48 KB of shared memory, destinations
at every residue of 16 bytes in a slice of a larger buffer.  k_decode_train and both backward exports: the vector kernels (<4>: F*F
% 4 == 0 and 16-byte aligned bases) and the scalar ones (<1>).  Plus the YOLOLayer module on non-contiguous heads and the launch
limits of the eval decode."""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
import yolov4_b200 as yb
from yolov4_b200 import _cabi
from spec_math_bounds import SIG_MAX_ULP

pytestmark = pytest.mark.gpu

CANARY = np.uint32(0x7FC0DEAD)                    # a quiet NaN with a payload no kernel writes


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _cfg(C):
    return {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": C}


def _bits_equal(a, b):
    """Bitwise equality of fp32 arrays, except that any NaN equals any NaN."""
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    assert a.shape == b.shape, (a.shape, b.shape)
    bad = (a.view(np.uint32) != b.view(np.uint32)) & ~(np.isnan(a) & np.isnan(b))
    if bad.any():
        i = np.argwhere(bad)[0]
        raise AssertionError(f"{int(bad.sum())} words differ, first at {tuple(i)}: {a[tuple(i)]!r} vs {b[tuple(i)]!r}")


SPECIALS = np.array([np.nan, np.inf, -np.inf, 0.0, -0.0, 100.0, -100.0, 86.0, -86.0, 86.00001, -86.00001, 88.7, -88.7, 88.8,
                     -88.8, 89.5, -105.0, 1e-40, -1e-40, 3e38, -3e38], np.float32)


def _logits(shape, seed):
    """Head values in the fast sigmoid range (|x| <= 86) with about 3 % from SPECIALS: the slow range, NaN, +-inf, +-0,
    subnormals, the overflow edges of exp."""
    rs = np.random.RandomState(seed)
    x = (rs.randn(*shape) * 4).astype(np.float32)
    m = rs.rand(*shape) < 0.03
    x[m] = SPECIALS[rs.randint(0, SPECIALS.size, int(m.sum()))]
    return x


# ------------------------------------------------------------------------------------------------ k_decode_dense
@pytest.mark.parametrize("F", [1, 2, 3, 8, 13, 19, 20, 65])
@pytest.mark.parametrize("C", [1, 3, 27, 28, 80, 187, 188, 300])
def test_decode_dense_every_tile_shape_into_a_slice_of_a_canary_buffer(C, F):
    """5+C = 32 (C=27) has no tail batch; C=187 is a tile of exactly 48 KB and C >= 188 takes the opt-in shared-memory branch.
    F=1..8 is one tile per (image, anchor), 13, 19, 20 and 65 end in a partial tile.  Row offsets 0..3 put the destination at
    every 16-byte residue that 5+C allows, so the float4 copy loop and the scalar one both run; rows_per_image leaves rows
    after the slice, and no word outside the slice may change."""
    B, nch, M = 2, 5 + C, 3 * F * F
    layer = (C + F) % 3
    raw = _logits((B, 3 * nch, F, F), seed=1000 * C + F)
    want = orc.decode_eval(raw, layer, C)
    raw_d = torch.from_numpy(raw).cuda()
    anch = _cabi.floats(orc.masked_anchors_grid(layer).ravel())
    for off in range(4):
        rows = M + off + 5
        buf = torch.full((B, rows, nch), int(CANARY.view(np.int32)), dtype=torch.int32, device="cuda").view(torch.float32)
        _cabi.check(_cabi.lib().yl_decode_dense(raw_d.data_ptr(), B, F, C, anch, float(orc.STRIDES[layer]), buf.data_ptr(),
                                                rows, off, _stream()))
        got = buf.cpu().numpy()
        _bits_equal(got[:, off:off + M], want)
        outside = np.ones(rows, bool)
        outside[off:off + M] = False
        assert (got[:, outside].view(np.uint32) == CANARY).all(), f"row_offset {off}: a word outside the slice changed"


# ------------------------------------------------------------------------------------------------ k_decode_train
def _shifted_like(shape):
    """An uninitialised fp32 CUDA tensor whose base is 4 bytes past a 16-byte boundary."""
    n = int(np.prod(shape))
    return torch.empty(n + 1, device="cuda")[1:].view(shape)


TRAIN_CASES = [(1, None), (19, None), (38, None), (38, "raw"), (38, "output"), (38, "pred")]   # (F, base offset by 4 bytes)


@pytest.mark.parametrize("F,shift", TRAIN_CASES)
@pytest.mark.parametrize("C", [1, 4, 80])
def test_decode_train_vector_and_scalar_kernels_match_the_oracle(C, F, shift):
    """F=38 with aligned bases runs k_decode_train<4>; an odd F or one base offset by 4 bytes runs <1>.  Oracle parity of `pred`
    pins x/y = sigmoid + grid and w/h = exp * anchor."""
    B, nch = 2, 5 + C
    layer = (C + F) % 3
    raw = _logits((B, 3 * nch, F, F), seed=7 * C + F)
    want_out, want_pred = orc.decode_train(raw, layer, C)
    bufs = {"raw": (B, 3 * nch, F, F), "output": (B, 3, nch, F, F), "pred": (B, 3, 4, F, F)}
    t = {k: (_shifted_like(s) if k == shift else torch.empty(s, device="cuda")) for k, s in bufs.items()}
    t["raw"].copy_(torch.from_numpy(raw))
    anch = _cabi.floats(orc.masked_anchors_grid(layer).ravel())
    _cabi.check(_cabi.lib().yl_decode_train(t["raw"].data_ptr(), B, F, C, anch, t["output"].data_ptr(), t["pred"].data_ptr(),
                                            _stream()))
    _bits_equal(t["output"].cpu().numpy(), want_out.transpose(0, 1, 4, 2, 3))
    _bits_equal(t["pred"].cpu().numpy(), want_pred.transpose(0, 1, 4, 2, 3))


# ------------------------------------------------------------------------------------------------ backward
def _upstream(shape, seed):
    """Upstream gradients with +-0, +-inf, NaN, subnormals and large values among normal ones."""
    rs = np.random.RandomState(seed)
    g = rs.randn(*shape).astype(np.float32)
    sp = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1e-40, -1e-40, 1e-45, 3e38, -3e38], np.float32)
    m = rs.rand(*shape) < 0.05
    g[m] = sp[rs.randint(0, sp.size, int(m.sum()))]
    return g


def _sigmoid_backward(g, o):
    """(g * (1 - o)) * o on the sigmoid channels (xy, obj, cls), g on w/h: every operation an fp32 rounding, as ATen's
    sigmoid_backward.  g, o planar [B, 3, nch, F, F]."""
    with np.errstate(all="ignore"):
        r = (g * (np.float32(1.0) - o)) * o
    r[:, :, 2:4] = g[:, :, 2:4]
    return r


BWD_CASES = [(19, None), (38, None), (38, "src"), (38, "grad"), (38, "out")]


@pytest.mark.parametrize("F,shift", BWD_CASES)
@pytest.mark.parametrize("from_raw", [True, False], ids=["backward_raw", "backward"])
def test_decode_train_backward_exports_bit_exact(from_raw, F, shift):
    """yl_decode_train_backward_raw recomputes o = sigmoid(raw) with the forward's bits; yl_decode_train_backward takes o as
    given.  F=38 with aligned bases runs <4>, an odd F or an offset base <1>."""
    B, C = 2, 4
    nch = 5 + C
    raw = _logits((B, 3 * nch, F, F), seed=F)
    o = np.ascontiguousarray(orc.decode_train(raw, 0, C)[0].transpose(0, 1, 4, 2, 3))          # planar [B, 3, nch, F, F]
    g = _upstream(o.shape, seed=F + 1)
    want = _sigmoid_backward(g, o)
    shapes = {"src": raw.shape, "grad": g.shape, "out": raw.shape}
    t = {k: (_shifted_like(s) if k == shift else torch.empty(s, device="cuda")) for k, s in shapes.items()}
    t["src"].copy_(torch.from_numpy(raw if from_raw else o.reshape(raw.shape)))
    t["grad"].copy_(torch.from_numpy(g))
    fn = _cabi.lib().yl_decode_train_backward_raw if from_raw else _cabi.lib().yl_decode_train_backward
    _cabi.check(fn(t["src"].data_ptr(), t["grad"].data_ptr(), B, F, C, t["out"].data_ptr(), _stream()))
    got = t["out"].cpu().numpy().reshape(o.shape)
    _bits_equal(got, want)
    # against float64 g s (1 - s): o is within SIG_MAX_ULP * 2^-24 of s, and 1 - o and the two products round once each
    s = 1.0 / (1.0 + np.exp(-raw.astype(np.float64).reshape(o.shape)))
    exact = g.astype(np.float64) * s * (1.0 - s)
    sig_ch = np.ones(nch, bool)
    sig_ch[2:4] = False
    fin = np.isfinite(exact) & np.isfinite(g) & sig_ch[None, None, :, None, None]
    tol = np.abs(g[fin]).astype(np.float64) * (SIG_MAX_ULP + 1.0) * 2.0 ** -24 + 2.0 ** -148
    assert (np.abs(got[fin] - exact[fin]) <= tol).all()


@pytest.mark.parametrize("F", [12, 13])
def test_yololayer_train_gradient_through_the_in_place_masked_output(F):
    """The reference's YOLOLoss.forward multiplies dict['output'] (a permuted view) by its masks in place before the loss;
    the gradient reaching the head is then (g * mask * (1 - o)) * o with o the forward's sigmoid.  F=12 runs the <4> kernels,
    F=13 the <1> ones."""
    B, C = 2, 4
    nch = 5 + C
    raw_np = _logits((B, 3 * nch, F, F), seed=40 + F)
    raw = torch.from_numpy(raw_np).cuda().requires_grad_(True)
    d = yb.YOLOLayer(_cfg(C), 0, device="cuda").train()(raw)
    out = d["output"]
    rs = np.random.RandomState(F)
    mask = torch.from_numpy((rs.rand(B, 3, F, F) < 0.5).astype(np.float32)).cuda()
    w = torch.from_numpy(rs.randn(B, 3, F, F, nch).astype(np.float32)).cuda()
    out[..., 4] *= mask                                                                 # yololoss.py:402
    (out * w).sum().backward()
    g = w.clone()
    g[..., 4] *= mask
    g = np.ascontiguousarray(g.cpu().numpy().transpose(0, 1, 4, 2, 3))
    o = np.ascontiguousarray(orc.decode_train(raw_np, 0, C)[0].transpose(0, 1, 4, 2, 3))
    _bits_equal(raw.grad.cpu().numpy().reshape(g.shape), _sigmoid_backward(g, o))


# ------------------------------------------------------------------------------------------------ non-contiguous heads
@pytest.mark.parametrize("form", ["channels_last", "slice"])
def test_yololayer_non_contiguous_heads_give_the_contiguous_bits(form):
    """Eval and train outputs and the gradient reaching the head are those of the contiguous tensor."""
    B, C, F = 2, 4, 12
    nch = 5 + C
    base = torch.from_numpy(_logits((B, 3 * nch, F, F), seed=5)).cuda()
    if form == "channels_last":
        store = base.to(memory_format=torch.channels_last)

        def view(t):
            return t
    else:
        store = torch.zeros(B + 1, 3 * nch + 7, F + 3, F + 5, device="cuda")

        def view(t):
            return t[1:, 3:3 + 3 * nch, 1:1 + F, 2:2 + F]
        view(store).copy_(base)
    assert torch.equal(view(store).view(torch.int32), base.view(torch.int32)) and not view(store).is_contiguous()
    layer = yb.YOLOLayer(_cfg(C), 1, device="cuda")
    assert torch.equal(layer.eval()(base).view(torch.int32), layer.eval()(view(store)).view(torch.int32))
    w = torch.randn(B, 3, F, F, nch, device="cuda")
    runs = []
    for leaf, head in ((base.clone().requires_grad_(True), lambda t: t), (store.clone().requires_grad_(True), view)):
        d = layer.train()(head(leaf))
        (d["output"] * w).sum().backward()
        runs.append((d, leaf))
    (d0, l0), (d1, l1) = runs
    for k in ("output", "pred"):
        assert torch.equal(d0[k].detach().view(torch.int32), d1[k].detach().view(torch.int32)), k
    assert torch.equal(l0.grad.view(torch.int32), view(l1.grad).view(torch.int32))
    rest = l1.grad.clone()
    view(rest).zero_()
    assert not rest.any()


# ------------------------------------------------------------------------------------------------ launch limits
def test_eval_decode_of_more_images_than_one_launch_can_index():
    """B*3 = 65538 (image, anchor) pairs exceed gridDim.y <= 65535: the decode goes out in slices."""
    B, C, F = 21846, 1, 1
    raw = _logits((B, 3 * (5 + C), F, F), seed=3)
    got = yb.YOLOLayer(_cfg(C), 2, device="cuda").eval()(torch.from_numpy(raw).cuda())
    _bits_equal(got.cpu().numpy(), orc.decode_eval(raw, 2, C))


def test_eval_decode_tile_at_the_shared_memory_limit_decodes_and_one_class_more_is_refused():
    """A tile is 64 boxes * (5+C) floats: the largest C whose tile fits the opt-in limit (227 KB on a B200: C = 903) decodes,
    the next raises before any launch, and the refusal does not disturb the next call."""
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    c_max = optin // (64 * 4) - 5
    with pytest.raises(_cabi.YoloHeadError):
        yb.YOLOLayer(_cfg(c_max + 1), 0, device="cuda").eval()(torch.zeros(1, 3 * (6 + c_max), 2, 2, device="cuda"))
    raw = _logits((1, 3 * (5 + c_max), 2, 2), seed=11)
    got = yb.YOLOLayer(_cfg(c_max), 0, device="cuda").eval()(torch.from_numpy(raw).cuda())
    _bits_equal(got.cpu().numpy(), orc.decode_eval(raw, 0, c_max))
