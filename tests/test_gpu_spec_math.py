"""Every fp32 bit pattern through the spec exp and sigmoid of the decode kernels (DESIGN.md section 4).

The kernels evaluate the spec functions in several forms that must give the same bits: the scalar sequence and its |x| <= 86 fast
path (exponent-field scaling, MUFU.RCP plus one Newton step), packed fp32x2 pairs (spec_exp2), and batches of 4 or 8 sigmoids with
one range test (spec_sigmoid_batch), which send every member down the scalar path when one member is out of range or NaN.  The
inputs are all 2^32 patterns, generated on the device in chunks.  With C = 1 and every masked anchor 1.0, the train decode's `pred`
w/h planes are spec_exp(t) and its sigmoid planes spec_sigmoid(t); with C = 27 the eval decode's obj / class columns are
spec_sigmoid(t)."""
import concurrent.futures
import os

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from yolov4_b200 import _cabi
from spec_math_bounds import EXP_MAX_ULP, SIG_MAX_ULP, SIG_ZERO_EDGE

pytestmark = pytest.mark.gpu

CHUNK = 1 << 24
N_CHUNKS = (1 << 32) // CHUNK
F = 1024
F2 = F * F
ONES = [1.0] * 6                     # masked anchors in grid units: pred w/h = exp(t) * 1.0


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _patterns(c):
    """Chunk c of the 2^32 fp32 bit patterns, in pattern order."""
    v = torch.arange(c * CHUNK, (c + 1) * CHUNK, dtype=torch.int64, device="cuda")
    return (v - ((v >> 31) << 32)).to(torch.int32).view(torch.float32)


def _padded(x, per):
    v = torch.zeros(-(-x.numel() // per) * per, device="cuda")
    v[:x.numel()] = x
    return v


def _shifted(t):
    """A copy of t whose base is 4 bytes past a 16-byte boundary."""
    s = torch.empty(t.numel() + 1, device="cuda")[1:].view(t.shape)
    s.copy_(t)
    return s


def _decode_train(s, shift=False):
    """(sigmoid, exp) of every element of the 1-D tensor s from one yl_decode_train call with C = 1.  The planes of each anchor are
    [A, B, A, B, A, B], so every element lands on a sigmoid channel (tx / ty) and an exp channel (tw / th).  shift=False runs
    k_decode_train<4> (F*F % 4 == 0, aligned bases); shift=True offsets every base by 4 bytes, which selects k_decode_train<1>."""
    n = s.numel()
    raw = _padded(s, 6 * F2).view(-1, 2, F2).repeat(1, 3, 1)           # [3B, 6, F2]
    out, pred = torch.empty_like(raw), torch.empty(raw.shape[0], 4, F2, device="cuda")
    if shift:
        raw, out, pred = _shifted(raw), _shifted(out), _shifted(pred)
    _cabi.check(_cabi.lib().yl_decode_train(raw.data_ptr(), raw.shape[0] // 3, F, 1, _cabi.floats(ONES), out.data_ptr(),
                                            pred.data_ptr(), _stream()))
    return out[:, :2].reshape(-1)[:n], pred[:, 2:4].reshape(-1)[:n]


def _train_fast(x):
    """Each value four times in a row: every 4-wide sigmoid batch and every exp pair is uniform, so an in-range value takes the
    packed fast path."""
    sig, ex = _decode_train(x.repeat_interleave(4))
    return sig[::4], ex[::4]


def _train_poisoned(x):
    """[x0, P, x1, P, ...]: every 4-wide batch and every exp pair (t0, t1), (t2, t3) has an out-of-range companion P, 100.0 in
    odd-numbered batches and NaN in even ones, so every value takes the path of a batch that failed its range test."""
    j = torch.arange(x.numel(), device="cuda")
    poison = torch.where((j >> 1) % 2 == 0, torch.tensor(float("nan"), device="cuda"), torch.tensor(100.0, device="cuda"))
    sig, ex = _decode_train(torch.stack([x, poison], 1).view(-1))
    return sig[::2], ex[::2]


def _dense_sigmoid(x, poison):
    """sigmoid of every element of x from yl_decode_dense with C = 27: with 5 + C = 32 channels, a thread's channels kr, kr+4, ...,
    kr+28 (kr < 4) form one 8-wide batch with one range test.  poison=False: all 32 channels of a box hold the same value, so every
    batch is uniform.  poison=True: channels 0-3 (slot 0 of every batch) hold 100.0 or NaN, channels 4-31 hold 28 values."""
    n = x.numel()
    if poison:
        v = _padded(x, 3 * 28 * F2).view(-1, 28, F2)
        p = torch.arange(F2, device="cuda")
        comp = torch.where(p % 2 == 0, torch.tensor(100.0, device="cuda"), torch.tensor(float("nan"), device="cuda"))
        raw = torch.cat([comp.expand(v.shape[0], 4, F2), v], 1)
    else:
        raw = _padded(x, 3 * F2).view(-1, 1, F2).expand(-1, 32, F2).contiguous()
    G = raw.shape[0]
    out = torch.empty(G, F2, 32, device="cuda")
    _cabi.check(_cabi.lib().yl_decode_dense(raw.data_ptr(), G // 3, F, 27, _cabi.floats(ONES), 8.0, out.data_ptr(), 3 * F2, 0,
                                            _stream()))
    if poison:
        return out[:, :, 4:].transpose(1, 2).reshape(-1)[:n]
    cols = out[:, :, 4:].view(torch.int32)
    assert torch.equal(cols, cols[:, :, :1].expand_as(cols)), "the 28 sigmoid columns of one uniform box differ"
    return out[:, :, 4].reshape(-1)[:n]


def _assert_same(a, b, x, what):
    """Bit-identical, except that any NaN equals any NaN."""
    bad = (a.view(torch.int32) != b.view(torch.int32)) & ~(a.isnan() & b.isnan())
    if bool(bad.any()):
        i = int(bad.nonzero()[0])
        xb = int(x.view(torch.int32)[i]) & 0xFFFFFFFF
        raise AssertionError(f"{what}: {int(bad.sum())} inputs differ, first x = {x[i].item()!r} (0x{xb:08x}): "
                             f"{a[i].item()!r} vs {b[i].item()!r}")


def test_every_float_gives_the_same_bits_in_every_kernel_form():
    """Fast path == the path of a batch with an out-of-range member, on every input; k_decode_train<4> == <1> == k_decode_dense."""
    for c in range(N_CHUNKS):
        x = _patterns(c)
        sig, ex = _train_fast(x)
        sig_p, ex_p = _train_poisoned(x)
        _assert_same(sig_p, sig, x, "sigmoid, 4-wide batch with a poisoned member vs uniform batch")
        _assert_same(ex_p, ex, x, "exp, pair with a poisoned member vs uniform pair")
        sig1, ex1 = _decode_train(x, shift=True)
        _assert_same(sig1, sig, x, "sigmoid, k_decode_train<1> vs <4>")
        _assert_same(ex1, ex, x, "exp, k_decode_train<1> vs <4>")
        _assert_same(_dense_sigmoid(x, False), sig, x, "sigmoid, k_decode_dense uniform 8-wide batch vs k_decode_train")
        _assert_same(_dense_sigmoid(x, True), sig, x, "sigmoid, k_decode_dense poisoned 8-wide batch vs k_decode_train")


def _oracle_check(x, sig, ex):
    Fo = 64
    raw = np.zeros(-(-x.size // (6 * Fo * Fo)) * 6 * Fo * Fo, np.float32)
    raw[:x.size] = x
    raw = np.tile(raw.reshape(-1, 2, Fo * Fo), (1, 3, 1)).reshape(-1, 18, Fo, Fo)
    out, pred = orc.decode_train(raw, 0, 1, anchors=[[8, 8]] * 9)              # layer 0, stride 8: masked anchors 1.0
    want_sig = np.ascontiguousarray(out.transpose(0, 1, 4, 2, 3)).reshape(-1, 6, Fo * Fo)[:, :2].reshape(-1)[:x.size]
    want_ex = np.ascontiguousarray(pred.transpose(0, 1, 4, 2, 3)).reshape(-1, 4, Fo * Fo)[:, 2:4].reshape(-1)[:x.size]
    for got, want, what in ((sig, want_sig, "sigmoid"), (ex, want_ex, "exp")):
        bad = (got.view(np.uint32) != want.view(np.uint32)) & ~(np.isnan(got) & np.isnan(want))
        if bad.any():
            i = int(np.argmax(bad))
            raise AssertionError(f"{what} vs oracle: {int(bad.sum())} inputs differ, first x = {x[i]!r} "
                                 f"(0x{int(x.view(np.uint32)[i]):08x}): {got[i]!r} vs {want[i]!r}")


def test_kernels_match_the_oracle_on_every_float():
    """The oracle's plain C restatement (the general exp sequence with its two scaling multiplies, IEEE division) against the
    GPU fast paths; the test above carries the result to every form.  The oracle spends about 100 ns per value, mostly on
    subnormal arithmetic, so the 2^32 values are spread over a thread pool (ctypes releases the GIL)."""
    workers = os.cpu_count() or 4
    part = CHUNK // 8
    pending = []
    with concurrent.futures.ThreadPoolExecutor(workers) as pool:
        for c in range(N_CHUNKS):
            x = _patterns(c)
            sig, ex = _train_fast(x)
            x, sig, ex = x.cpu().numpy(), sig.cpu().numpy(), ex.cpu().numpy()
            for k in range(0, CHUNK, part):
                pending.append(pool.submit(_oracle_check, x[k:k + part], sig[k:k + part], ex[k:k + part]))
            while len(pending) > 2 * workers:
                pending.pop(0).result()
        for f in pending:
            f.result()


def _ulp_err(r, R):
    """max |r - R| in units of the fp32 ulp at the float64 value R (2^-149 where R is subnormal)."""
    if R.numel() == 0:
        return 0.0
    _, e = torch.frexp(R)                                                      # R = m 2^e, 0.5 <= |m| < 1
    ulp = ((e.to(torch.int64) - 24).clamp(min=-149) + 1023).bitwise_left_shift(52).view(torch.float64)
    return float(((r.double() - R).abs() / ulp).max())


def test_every_float_is_within_the_stated_error_of_float64():
    inf, nan = float("inf"), float("nan")
    sig, ex = _train_fast(torch.tensor([inf, -inf, nan], device="cuda"))
    assert sig.tolist()[:2] == [1.0, 0.0] and ex.tolist()[:2] == [inf, 0.0] and sig[2].isnan() and ex[2].isnan()
    assert int(sig.view(torch.int32)[1]) == 0 and int(ex.view(torch.int32)[1]) == 0          # +0, not -0
    worst_exp = worst_sig = 0.0
    for c in range(N_CHUNKS):
        x = _patterns(c)
        sig, ex = _train_fast(x)
        x64 = x.double()
        nan_in = x.isnan()
        assert torch.equal(ex.isnan(), nan_in) and torch.equal(sig.isnan(), nan_in)
        # exp: +inf exactly where the float64 value rounds past FLT_MAX, +0 below the clamp, else within EXP_MAX_ULP
        E = torch.exp(x64)
        over = E.float().isinf()
        assert torch.equal(ex.isinf(), over) and bool((ex[over] > 0).all())
        assert bool((ex[x < -104.0].view(torch.int32) == 0).all())
        fin = ~nan_in & ~over
        worst_exp = max(worst_exp, _ulp_err(ex[fin], E[fin]))
        # sigmoid: +0 exactly on x <= SIG_ZERO_EDGE, where exp(-x) overflows
        S = 1.0 / (1.0 + torch.exp(-x64))
        zero = x <= float(SIG_ZERO_EDGE)
        assert torch.equal(sig.view(torch.int32) == 0, zero)
        normal = S >= 2.0 ** -126
        worst_sig = max(worst_sig, _ulp_err(sig[normal], S[normal]))
        sub = ~nan_in & ~normal & ~zero
        assert bool(((sig[sub].double() - S[sub]).abs() < 2.0 ** -126).all())
    print(f"\nmax error over every fp32 input: exp {worst_exp:.6f} ulp, sigmoid {worst_sig:.6f} ulp (normal results)")
    assert worst_exp <= EXP_MAX_ULP
    assert worst_sig <= SIG_MAX_ULP
