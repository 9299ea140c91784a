"""The builders of the fused front end's edge cases (raw_edge_cases.py), checked without a GPU: the planted t* logits really sit
at the exact test's edge, the odd-grid lists really put a vector-eligible scale at a table row that is not a multiple of 4, and
yl_filter_raw_typed rejects bad arguments before any CUDA work."""
import ctypes

import numpy as np
import pytest

import agnostic_spec as spec
import raw_edge_cases as rec
from oracle import oracle as orc

ODD_GRIDS = ([75, 38, 19], [13, 7, 4], [7, 4, 2], [6, 3, 2], [75, 37, 18])
BENCH_GRIDS = ([76, 38, 19], [52, 26, 13])


@pytest.mark.parametrize("dt", rec.DTYPES)
@pytest.mark.parametrize("conf", rec.THRESHOLD_CONFS, ids=[repr(c) for c in rec.THRESHOLD_CONFS])
def test_t_star_passes_and_nothing_below_it_does(conf, dt):
    """For every regime: t* passes, its predecessor fails, and none of the 4096 values below t* passes (the spec sigmoid is
    not proven monotone to the ulp, so the bisection alone would not show that t* is the smallest)."""
    regimes = rec.threshold_regimes(conf, dt)
    assert len(regimes) >= (2 if conf > 0.5 else 4), "too few reachable regimes"   # sigmoid(to) >= 1.2e-38: obj is never subnormal
    for r, to, obj, ts, pr in regimes:
        assert obj == rec.sigmoid(to) and obj >= np.float32(conf)
        assert rec.to_elem(ts, dt) == ts and rec.to_elem(pr, dt) == pr and pr < ts
        assert rec.passes(obj, ts, conf) and not rec.passes(obj, pr, conf), (r, to, ts)
        below = rec.values_below(ts, 4096, dt)
        assert below[-1] == pr
        assert not any(rec.passes(obj, t, conf) for t in below), (r, to, ts)


def test_ratio_regimes_reach_both_sides_of_the_bound_cap():
    """class_logit_bound caps q = (conf / obj)(1 - 1e-5) at 0.9: the regimes put conf / obj on both sides of that cap, and at 1."""
    ratios = [float(np.float32(0.2)) / float(obj) for _, _, obj, _, _ in rec.threshold_regimes(0.2, "f32")]
    q = [r * (1 - 1e-5) for r in ratios]
    assert any(0.9 < v < 0.90001 for v in q) and any(0.89999 < v < 0.9 for v in q)
    assert any(abs(r - 1) < 1e-6 for r in ratios)
    assert any(float(np.float32(1e-30)) / float(obj) < 1e-7 for _, _, obj, _, _ in rec.threshold_regimes(1e-30, "f32"))


@pytest.mark.parametrize("dt", rec.DTYPES)
@pytest.mark.parametrize("Fs,C", [([16, 8, 4], 128), ([13, 7, 4], 20), ([9], 33)])
def test_threshold_case_has_exactly_the_planted_candidates(Fs, C, dt):
    """The literal filter over the oracle's decode of a threshold case finds exactly the planted t* pairs."""
    for conf in (1e-3, 0.2, rec.THRESHOLD_CONFS[-1]):
        raws, expected = rec.threshold_case(Fs, C, conf, dt)
        for r in raws:
            assert np.array_equal(rec.to_elem(r, dt), r, equal_nan=True)
        dense = orc.decode_eval_cat(raws, C)
        got = []
        for b in range(dense.shape[0]):
            cand = spec.candidates(dense[b], C, conf)
            got += [(b, int(r), int(c)) for r, c in zip(cand["row"], cand["cls"])]
        assert sorted(got) == expected and len(expected) >= 8


def test_odd_grid_lists_put_a_vector_scale_at_an_unaligned_table_row():
    for Fs in ODD_GRIDS:
        offs = rec.row_offsets(Fs)
        assert any((f * f) % 4 == 0 and off % 4 != 0 for f, off in zip(Fs, offs)), Fs
        _, _, vec = rec.flag_kernel(Fs, 80, 1e-3, "f32", flag_env="tma")
        assert all(v == 1 for f, off, v in zip(Fs, offs, vec) if off % 4 != 0)
    for Fs in BENCH_GRIDS:
        assert all(off % 4 == 0 for off in rec.row_offsets(Fs)), Fs
        assert rec.flag_kernel(Fs, 80, 1e-4, "f32", flag_env="tma")[2] == [4, 4, 1]


def test_filter_rejects_bad_arguments_before_cuda_work():
    """Every argument error returns before the first CUDA call (this runs without a device); the pointers are never touched,
    so stand-in addresses do."""
    from yolov4_b200 import _cabi
    L = _cabi.lib()
    fake = ctypes.c_void_p(1 << 20)
    anch = _cabi.floats([v for wh in orc.ANCHORS_PX for v in wh])
    mask = _cabi.ints([v for m in orc.ANCHOR_MASK for v in m])
    Fs, C, B = [4, 2, 1], 20, 21846
    M = sum(3 * f * f for f in Fs)
    raw = _cabi.ptrs([1 << 20] * 3)
    nb = L.yl_post_workspace_bytes(B, M, C, 16)

    def call(dtype=0, fs=Fs, n=3, b=B, c=C, m=M, ws=fake, wsb=nb, cap=16, i0=0, cnt=B, stages=3, r=raw):
        return L.yl_filter_raw_typed(r, dtype, _cabi.ints(fs), n, b, c, anch, mask, 1e-3, ws, wsb, m, cap, i0, cnt, stages, None)

    assert call(cnt=0) == 0 and call(i0=B, cnt=0) == 0       # no image: nothing to launch, nothing touched
    for kw in (dict(i0=1), dict(cnt=B + 1), dict(i0=-1, cnt=1), dict(cnt=-1), dict(stages=0), dict(stages=4), dict(stages=8),
               dict(dtype=3), dict(n=0), dict(n=4), dict(b=0), dict(m=M + 1), dict(fs=[4, 0, 1]), dict(cap=0), dict(ws=None),
               dict(r=None)):
        assert call(**kw) == 1, kw
    assert call(c=129) == 2
    assert call(wsb=nb - 1) == 3
