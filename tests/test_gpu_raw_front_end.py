"""The fused front end (yl_filter_raw_typed: k_flag_tma<NW> or k_flag_raw<T,NW>, then k_emit_flagged<T,NW>) on every flag and emit
dispatch branch: odd and mixed grid lists, one to three heads, fp32 heads at every base residue, TMA tail tiles, every class-count
form, both threshold modes, the emit kernel's dense-tile fallback, special values, stage splits and image groups, batches past
one launch's gridDim.y, and class logits planted exactly at the threshold of the spec's test.

Every case runs through the C ABI (yl_post_reset, yl_filter_raw_typed, yl_nms) into a workspace filled with 0xFF and checks:
  1. every image's candidate total (meta[2B+b]) and largest (image, class) segment (meta[B+b]) equal those of the literal filter
     (agnostic_spec.candidates) over the oracle's decode, since NMS can hide a missing candidate;
  2. the rows equal orc.postprocess(orc.decode_eval_cat(raws, C), ...) bit for bit (NaN equals NaN);
  3. every form of the same values (base residues, stage splits, image groups) writes the same bytes;
  4. the flag and emit kernels that ran (torch.profiler) are those raw_edge_cases.flag_kernel names for the case.
The profiler stops reporting kernels in a process that has captured a CUDA graph, so check 4 runs in the two fresh processes
of the last tests (the default flag kernel and YL_FLAG=ldg), which run this file's case table again.
"""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import yolov4_b200 as yb                                              # noqa: E402
from yolov4_b200 import _cabi                                         # noqa: E402

import raw_edge_cases as rec                                          # noqa: E402
from oracle import oracle as orc                                      # noqa: E402  (checker only)
from test_gpu_dense_front_end import _pow2, expected_counts           # noqa: E402
from test_gpu_parity import assert_lists_bit_equal                    # noqa: E402

NMS = 0.45
TORCH_DT = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}
CODE = {"f32": 0, "f16": 1, "bf16": 2}
KNAME = {"f32": "float", "f16": "__half", "bf16": "__nv_bfloat16"}
ANCH = _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh])
MASK = _cabi.ints([v for m in yb.ANCHOR_MASK for v in m])
LOW, HIGH = 1e-3, 0.2              # k_flag_tma's threshold range (fp32) and k_flag_raw's objectness-first range
FRESH = os.environ.get("YL_RAW_FRONT_END_FRESH") == "1"             # set by the fresh-process tests: check the kernels too


def _f32(x):
    return float(np.float32(x))


def on_device(raws, dt, residues=None):
    """Each head (float32 arrays holding values of dt) copied to a CUDA buffer of dt at base residue residues[l] bytes mod 16."""
    out = []
    for l, r in enumerate(raws):
        t = torch.from_numpy(np.ascontiguousarray(r)).to(TORCH_DT[dt])
        es = t.element_size()
        off = (residues[l] if residues else 0) // es
        buf = torch.empty(t.numel() + 16 // es, dtype=t.dtype, device="cuda")
        v = buf[off:off + t.numel()].view(t.shape)
        v.copy_(t)
        assert v.data_ptr() % 16 == off * es
        out.append(v)
    return out


def run_cabi(heads, C, conf, cap_seg, cap_out, calls=None):
    """yl_filter_raw_typed calls (img_first, img_count, stages) into one workspace filled with 0xFF (yl_post_reset first unless
    the first call folds the reset, stages bit 2), then one yl_nms over all images.  Returns (rows, meta) as NumPy arrays."""
    B, Fs = heads[0].shape[0], [h.shape[2] for h in heads]
    M = sum(3 * f * f for f in Fs)
    dt = {v: k for k, v in TORCH_DT.items()}[heads[0].dtype]
    calls = calls or [(0, B, 3)]
    L = _cabi.lib()
    nb = L.yl_post_workspace_bytes(B, M, C, cap_seg)
    ws = torch.full((nb,), 255, dtype=torch.uint8, device="cuda")
    rows = torch.full((B, cap_out, 7), 7.0, device="cuda")
    meta = torch.full((3 * B,), -1, dtype=torch.int32, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    rp, fs = _cabi.ptrs([h.data_ptr() for h in heads]), _cabi.ints(Fs)
    if not calls[0][2] & 4:
        _cabi.check(L.yl_post_reset(ws.data_ptr(), nb, B, M, C, cap_seg, st))
    for i0, n, stages in calls:
        _cabi.check(L.yl_filter_raw_typed(rp, CODE[dt], fs, len(Fs), B, C, ANCH, MASK, _f32(conf), ws.data_ptr(), nb, M, cap_seg,
                                          i0, n, stages, st))
    _cabi.check(L.yl_nms(ws.data_ptr(), nb, B, M, C, cap_seg, _f32(NMS), rows.data_ptr(), cap_out, meta.data_ptr(), 0, B, st))
    torch.cuda.synchronize()
    return rows.cpu().numpy(), meta.cpu().numpy()


def launched(fn):
    """fn() under torch.profiler: (its result, {front-end kernel name: launches})."""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {}
    for e in prof.key_averages():
        m = re.search(r"(k_flag_tma|k_flag_raw|k_emit_flagged)<([^>]*)>", e.key)
        if m:
            k = "%s<%s>" % (m.group(1), re.sub(r"\s", "", m.group(2)))
            names[k] = names.get(k, 0) + e.count
    return out, names


def expected_kernels(Fs, C, conf, dt, residues):
    flag, (edt, nw), vec = rec.flag_kernel(Fs, C, conf, dt, residues)
    f = "k_flag_tma<%d>" % flag[1] if flag[0] == "tma" else "k_flag_raw<%s,%d>" % (KNAME[flag[1]], flag[2])
    return {f, "k_emit_flagged<%s,%d>" % (KNAME[edt], nw)}, vec


def check_raw(raws, C, conf, dt="f32", residues=((0, 0, 0),), calls=(None,), kernel=None, what=""):
    """Runs raws (values of dt) at every residue combination and with every call list, asserts counts, rows, equal bytes and
    the kernels of every residue combination (kernel: 'tma' or 'raw' to pin the flag kernel of the first one).  Returns the
    oracle's rows and the expected candidate totals."""
    Fs = [r.shape[2] for r in raws]
    dense = orc.decode_eval_cat([np.ascontiguousarray(r, np.float32) for r in raws], C)
    tot, seg = expected_counts(dense, C, conf)
    want = orc.postprocess(dense, C, conf, NMS, nthreads=8)
    B = dense.shape[0]
    cap_seg, cap_out = _pow2(max(16, seg.max())), _pow2(max(16, tot.max()))
    first, fails = None, {}
    for res in residues:
        heads = on_device(raws, dt, res)
        want_k, vec = expected_kernels(Fs, C, conf, dt, [h.data_ptr() % 16 for h in heads])
        for cl in calls:
            label = "residues %s calls %s" % (res[:len(Fs)], cl)
            if cl is None and FRESH:
                (rows, meta), names = launched(lambda: run_cabi(heads, C, conf, cap_seg, cap_out))
            else:
                rows, meta = run_cabi(heads, C, conf, cap_seg, cap_out, cl)
            got = [rows[b, :meta[b]] if meta[b] > 0 else None for b in range(B)]
            try:
                if cl is None and FRESH:
                    assert set(names) == want_k, "kernels %s, expected %s (vector widths %s)" % (sorted(names), sorted(want_k), vec)
                    if kernel is not None and res == residues[0]:
                        assert any(n.startswith("k_flag_" + kernel) for n in want_k) or os.environ.get("YL_FLAG") == "ldg", \
                            "the case is meant for k_flag_%s, the dispatch gives %s" % (kernel, sorted(want_k))
                assert np.array_equal(meta[2 * B:], tot), "candidates per image %s, literal filter %s" % (meta[2 * B:], tot)
                assert np.array_equal(meta[B:2 * B], seg), "largest segment per image %s, literal filter %s" % (meta[B:2 * B], seg)
                assert_lists_bit_equal(got, want, what="rows vs oracle")
                if first is None:
                    first = got
                assert all(g is None and f is None or np.array_equal(g.view(np.uint32), f.view(np.uint32))
                           for g, f in zip(got, first)), "rows differ from the first run's bytes"
            except AssertionError as e:
                fails[label] = str(e).split("\n")[0]
    assert not fails, "%s %s C %d conf %r: %d runs fail: %s" % (what, dt, C, float(conf), len(fails), fails)
    return want, tot


SPLITS = (None, [(0, 2, 1), (0, 2, 2)], [(0, 2, 7)], [(0, 1, 3), (1, 1, 3)])


# ------------------------------------------------------------------------------------------------ odd and mixed grids
ODD_GRIDS = ([75, 38, 19], [13, 7, 4], [7, 4, 2], [6, 3, 2], [75, 37, 18], [76, 37, 18])


@pytest.mark.parametrize("conf", [LOW, HIGH])
@pytest.mark.parametrize("Fs", ODD_GRIDS, ids=[str(f) for f in ODD_GRIDS])
def test_odd_and_mixed_grids(Fs, conf):
    """A lower scale with an odd grid puts the next even scale's table rows at an offset that is not a multiple of 4: that scale
    takes the scalar path ([76, 37, 18]: k_flag_tma streams 76x76 and its scalar warps take the even 18x18)."""
    raws = rec.plant_specials(rec.heads(2, Fs, 80, seed=sum(Fs)), 80, seed=1)
    check_raw(raws, 80, conf, calls=SPLITS, what=str(Fs))


# ------------------------------------------------------------------------------------------------ head counts and TMA tiles
SHAPES = ([1], [2], [4], [8], [12], [16], [20], [2, 1], [9, 5], [16, 8], [20, 12, 8], [16, 4, 2], [12, 8, 2])


@pytest.mark.parametrize("conf", [LOW, HIGH])
@pytest.mark.parametrize("Fs", SHAPES, ids=[str(f) for f in SHAPES])
def test_head_counts_and_tma_tiles(Fs, conf):
    """One to three heads; F*F below 128 (F = 2, 4, 8: one short TMA tile), with a tail tile (F = 12, 20: np < 128) and an exact
    multiple (F = 16).  C = 24 is the smallest TMA ring (three 8-class chunks)."""
    check_raw(rec.heads(2, Fs, 24, seed=len(Fs) * 100 + Fs[0]), 24, conf, calls=(None, SPLITS[1]), what=str(Fs))


# ------------------------------------------------------------------------------------------------ fp32 base residues
RESIDUES = ((0, 0, 0), (4, 8, 12), (12, 4, 8), (0, 4, 0), (0, 0, 8), (8, 0, 0))


@pytest.mark.parametrize("conf", [LOW, HIGH])
@pytest.mark.parametrize("Fs", ([16, 8, 4], [20, 10, 6]), ids=str)
def test_every_fp32_base_residue(Fs, conf):
    """Each head at its own base residue: all unaligned means no TMA scale (k_flag_raw with one box per lane on even grids);
    one unaligned scale means k_flag_tma streams the others and its scalar warps take the unaligned one."""
    check_raw(rec.heads(2, Fs, 24, seed=Fs[0]), 24, conf, residues=RESIDUES, what=str(Fs))
    assert rec.flag_kernel(Fs, 24, LOW, "f32", [4, 8, 12], flag_env="tma")[0][0] == "raw"
    assert rec.flag_kernel(Fs, 24, LOW, "f32", [0, 4, 0], flag_env="tma")[2] == [4, 1, 4]


# ------------------------------------------------------------------------------------------------ class counts
CLASS_COUNTS = (1, 8, 16, 17, 24, 31, 32, 33, 63, 64, 65, 96, 97, 127, 128)


@pytest.mark.parametrize("conf", [LOW, HIGH])
@pytest.mark.parametrize("C", CLASS_COUNTS)
def test_every_class_count_form(C, conf):
    """NW = 1..4, no TMA ring below three chunks (C <= 16), partial chunks (C % 8 != 0), flag-word edges (C = 32k, 32k + 1)."""
    check_raw(rec.plant_specials(rec.heads(2, [16, 8, 4], C, seed=C), C, seed=C), C, conf, what="C %d" % C)


# ------------------------------------------------------------------------------------------------ threshold modes
@pytest.mark.parametrize("conf", [float(np.nextafter(np.float32(0.02), np.float32(0))), 0.02, 0.0, -0.5, float("nan"), 1.0, 1.5],
                         ids=["below_0.02", "0.02", "0", "-0.5", "nan", "1", "1.5"])
def test_threshold_modes(conf):
    """The last dense-mode threshold (k_flag_tma) and the first objectness-first one (k_flag_raw), conf <= 0 (every non-NaN pair
    passes), NaN (nothing does) and conf >= 1 (only sigmoid == 1 on both sides passes at 1)."""
    Fs, C = [16, 8, 4], 24
    raws = rec.plant_specials(rec.heads(2, Fs, C, seed=3), C, seed=4)
    v = raws[1].reshape(2, 3, 5 + C, 64)
    v[0, 1, 4, 5:20] = 30.0
    v[0, 1, 5 + 3, 5:20] = 20.0
    v[1, 2, 4, 40:44] = 17.0
    v[1, 2, 5:, 40:44] = 16.5
    _, tot = check_raw(raws, C, conf, calls=(None, SPLITS[2]), what="threshold mode")
    if conf == 1.0:
        assert tot.sum() > 0
    if conf != conf or conf > 1:
        assert tot.sum() == 0


# ------------------------------------------------------------------------------------------------ emit fallback
@pytest.mark.parametrize("C,n,extra", [(128, 2, 0), (128, 2, 1), (8, 32, 0), (8, 32, 1), (2, 128, 0), (3, 128, 0), (9, 32, 0)])
@pytest.mark.parametrize("conf", [LOW, HIGH])
def test_emit_dense_tile_fallback(C, n, extra, conf):
    """n live boxes with every class flagged (plus `extra` boxes with one) in one warp tile of a vector scale (128 boxes: 16x16)
    and of a scalar one (32 boxes: 13x13): a queue of exactly 256 flagged pairs, one more (box-by-box fallback), more than 32
    flagged boxes in one batch (C = 2), whole boxes of 128 classes."""
    Fs, B = [16, 13], 2
    raws = [np.zeros((B, 3, 5 + C, f * f), np.float32) for f in Fs]
    for v in raws:
        v[:, :, 4] = -30.0
        v[:, :, 5:] = -20.0
    for v, b, a, p0 in ((raws[0], 0, 1, 128), (raws[1], 1, 2, 32)):
        nb = min(n + extra, 128 if v is raws[0] else 32)
        for i in range(nb):
            v[b, a, 4, p0 + i] = 5.0
            v[b, a, 0:4, p0 + i] = (0.3 * (i % 5), -0.2 * (i % 3), 0.1 * (i % 7), 0.0)
            if i < n:
                v[b, a, 5:, p0 + i] = 3.0 + 0.01 * np.arange(C)
            else:
                v[b, a, 5 + (i * 7) % C, p0 + i] = 3.0
    raws = [v.reshape(B, 3 * (5 + C), f, f) for v, f in zip(raws, Fs)]
    _, tot = check_raw(raws, C, conf, what="emit fallback")
    assert tot[0] == n * C + (min(n + extra, 128) - n)


def test_conf_zero_flags_every_class_of_every_box():
    check_raw(rec.heads(2, [8, 4, 2], 128, seed=5), 128, 0.0, calls=(None, SPLITS[1]), what="conf 0")


# ------------------------------------------------------------------------------------------------ special values
@pytest.mark.parametrize("conf", [LOW, HIGH, 0.0])
@pytest.mark.parametrize("Fs,C", [([16, 8, 4], 20), ([13, 7, 4], 80), ([16, 8, 4], 80)], ids=str)
def test_special_values(Fs, C, conf):
    """NaN, +-inf, +-0 and +-1e30 as objectness, class and box logits of live and dead boxes, several per scale."""
    raws = rec.heads(2, Fs, C, seed=C + Fs[0])
    for s in range(4):
        raws = rec.plant_specials(raws, C, seed=10 + s)
    check_raw(raws, C, conf, calls=(None, SPLITS[1], SPLITS[2]), what="special values")


# ------------------------------------------------------------------------------------------------ stages and image groups
@pytest.mark.parametrize("conf,kernel", [(LOW, "tma"), (HIGH, "raw")])
@pytest.mark.parametrize("Fs", ([16, 8, 4], [6, 3, 2]), ids=str)
def test_stages_and_image_groups(Fs, conf, kernel):
    """Stages 1 then 2, stages 7 (the flag kernel zeroes the counters of a 0xFF workspace), 5 then 2, and three image groups
    filtered into one workspace by separate calls (k_flag_tma's tile counters are per first image)."""
    calls = (None, [(0, 3, 1), (0, 3, 2)], [(0, 3, 7)], [(0, 3, 5), (0, 3, 2)], [(0, 1, 3), (1, 1, 3), (2, 1, 3)],
             [(0, 1, 7), (1, 2, 3)], [(2, 1, 1), (0, 2, 1), (0, 3, 2)])
    check_raw(rec.heads(3, Fs, 24, seed=Fs[0] + 17), 24, conf, calls=calls, kernel=kernel, what=str(Fs))


# ------------------------------------------------------------------------------------------------ exact-threshold logits
@pytest.mark.parametrize("conf", rec.THRESHOLD_CONFS, ids=[repr(c) for c in rec.THRESHOLD_CONFS])
@pytest.mark.parametrize("dt", rec.DTYPES)
@pytest.mark.parametrize("Fs,C", [([16, 8, 4], 128), ([13, 7, 4], 20)], ids=str)
def test_exact_threshold_logits(Fs, C, dt, conf):
    """t* (the smallest logit of the element type that passes fl32(obj * sigmoid(t)) >= conf) as one class of a box and its
    predecessor as another: exactly the t* pairs are candidates, and boxes whose classes are all pred(t*) give none.  Planted
    at class indices on chunk and word edges, box positions on lane, tile and scale edges.  16-bit heads on 16x16 / 8x8 / 4x4
    take the paired half compare against the bound rounded down (flag_or2); 13x13 / 7x7 / 4x4 the scalar path."""
    raws, expected = rec.threshold_case(Fs, C, conf, dt)
    _, tot = check_raw(raws, C, conf, dt=dt, what="t* %s" % Fs)
    assert tot.tolist() == [sum(1 for e in expected if e[0] == b) for b in range(2)]


# ------------------------------------------------------------------------------------------------ launch limit
@pytest.mark.parametrize("conf", [LOW, HIGH])
@pytest.mark.parametrize("B", [21845, 21846])
def test_more_images_than_one_launch_can_index(B, conf):
    """B*3 = 65538 (image, anchor) pairs exceed gridDim.y <= 65535: k_flag_raw and k_emit_flagged go out in slices of 21845
    images, and only the first flag slice may zero the counters.  The batch repeats three images; its last one, alone in the
    second slice, is a fourth."""
    Fs, C = [4, 2, 1], 20
    base = rec.heads(4, Fs, C, seed=99)
    for r in base:
        r.reshape(4, 3, 5 + C, -1)[:, :, 4] += 3.0
    idx = np.arange(B) % 3
    idx[-1] = 3
    dense = orc.decode_eval_cat(base, C)
    tot, seg = expected_counts(dense, C, conf)
    want = orc.postprocess(dense, C, conf, NMS)
    cap_seg, cap_out = _pow2(max(16, seg.max())), _pow2(max(16, max(0 if w is None else len(w) for w in want)))
    it = torch.from_numpy(idx).cuda()
    heads = [torch.from_numpy(r).cuda()[it].contiguous() for r in base]
    n_slices = 1 if B <= 21845 else 2
    tma = rec.flag_kernel(Fs, C, conf, "f32")[0][0] == "tma"
    want_k = {"k_flag_tma<1>": 1} if tma else {"k_flag_raw<float,1>": n_slices}
    want_k["k_emit_flagged<float,1>"] = n_slices
    for calls in (None, [(0, B, 7)]):
        if FRESH:
            (rows, meta), names = launched(lambda: run_cabi(heads, C, conf, cap_seg, cap_out, calls))
            assert names == want_k, names
        else:
            rows, meta = run_cabi(heads, C, conf, cap_seg, cap_out, calls)
        assert np.array_equal(meta[2 * B:], tot[idx]) and np.array_equal(meta[B:2 * B], seg[idx])
        assert np.array_equal(meta[:B], np.array([0 if w is None else len(w) for w in want])[idx])
        for d in range(4):
            if want[d] is not None:
                sel = rows[idx == d, :len(want[d])]
                assert (sel.view(np.uint32) == want[d].view(np.uint32)[None]).all(), "image %d's rows" % d


# ------------------------------------------------------------------------------------------------ every entry point
@pytest.mark.parametrize("conf", [LOW, HIGH])
@pytest.mark.parametrize("Fs", ODD_GRIDS[:5], ids=[str(f) for f in ODD_GRIDS[:5]])
def test_odd_grids_through_every_entry(Fs, conf):
    """detect_raw, HeadPostprocessor (one and three image groups, captured and replayed once) and the host-buffer context.  Last
    in the file: it captures CUDA graphs."""
    B, C = 3, 20
    raws = rec.heads(B, Fs, C, seed=7 + sum(Fs))
    want = orc.detect(raws, C, conf, NMS)
    assert_lists_bit_equal(orc.postprocess(orc.decode_eval_cat(raws, C), C, conf, NMS), want, what="oracle forms")
    heads = [torch.from_numpy(r).cuda() for r in raws]
    assert_lists_bit_equal(yb.detect_raw(heads, C, conf, NMS), want, what="detect_raw")
    M, cap_out = sum(3 * f * f for f in Fs), 32768
    for g in (1, 3):
        hp = yb.HeadPostprocessor(B, Fs, C, conf, NMS, cap_seg=_pow2(M), cap_out=cap_out, n_groups=g).capture(heads)
        hp.replay()
        torch.cuda.synchronize()
        assert_lists_bit_equal(hp.results(), want, what="HeadPostprocessor n_groups %d" % g)
    ctx = ctypes.c_void_p()
    L = _cabi.lib()
    _cabi.check(L.yl_context_create(ctypes.byref(ctx), 0, B, _cabi.ints(Fs), 3, C, ANCH, MASK, _pow2(M), cap_out))
    try:
        rows, counts = np.zeros((B, cap_out, 7), np.float32), np.zeros((B,), np.int32)
        _cabi.check(L.yl_detect_host(ctx, _cabi.ptrs([r.ctypes.data for r in raws]), _f32(conf), _f32(NMS), rows.ctypes.data,
                                     counts.ctypes.data))
        assert_lists_bit_equal([rows[b, :counts[b]] if counts[b] else None for b in range(B)], want, what="yl_detect_host")
    finally:
        _cabi.check(L.yl_context_destroy(ctx))


# ------------------------------------------------------------------------------------------------ k_flag_raw everywhere
@pytest.mark.parametrize("flag", ["tma", "ldg"])
def test_case_table_and_its_kernels_in_a_fresh_process(flag):
    """The case table again in a fresh process, now also asserting the kernels that ran: with the default flag kernel, and with
    YL_FLAG=ldg (read when the library loads), where k_flag_raw handles every threshold."""
    if FRESH:
        pytest.skip("already in the fresh process")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, YL_FLAG=flag, YL_RAW_FRONT_END_FRESH="1")
    p = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "-p", "no:cacheprovider", os.path.abspath(__file__),
                        "-k", "not fresh_process and not every_entry" + (" and not more_images" if flag == "ldg" else "")],
                       cwd=root, env=env, capture_output=True, text=True, timeout=1500)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-2000:]
    passed = re.search(r"(\d+) passed", p.stdout)
    assert passed and int(passed.group(1)) >= 170 and "skipped" not in p.stdout, p.stdout[-1000:]
