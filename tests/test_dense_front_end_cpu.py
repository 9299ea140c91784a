"""CPU checks of the dense front end's reference on its special-value truth table: agnostic_spec.candidates (the literal filter
the GPU test counts against) agrees with the C oracle, and a filter that takes the 'any class passes' shortcut for zero or
infinite objectness disagrees with it -- the defect test_gpu_dense_front_end.py looks for -- while the shortcut restricted to
finite positive objectness agrees everywhere."""
import numpy as np
import pytest

import agnostic_spec as spec
import dense_edge_cases as dec
from oracle import oracle as orc

TABLE = dec.truth_table()


def _bits_equal(a, b):
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(a.view(np.uint32)[~na], b.view(np.uint32)[~nb])


def test_truth_table_shape():
    assert TABLE.shape == (len(dec.TABLE_OBJ) * len(dec.TABLE_MAX), 5 + dec.TABLE_C)
    nc = dec.TABLE_NUM_CLASSES
    with np.errstate(invalid="ignore"):
        mx = np.max(TABLE[:, 5:5 + nc], axis=1)
    want = np.tile(np.array(dec.TABLE_MAX, np.float32), len(dec.TABLE_OBJ))
    assert _bits_equal(mx, want), "the first num_classes classes have exactly the table's max"
    assert np.isfinite(TABLE[:, 5 + nc:]).all() and (TABLE[:, 5 + nc:] < 0).any(1).all()
    box = np.stack([TABLE[:, 0] - 4, TABLE[:, 1] - 4, TABLE[:, 0] + 4, TABLE[:, 1] + 4], 1)
    ar = spec.areas(box)
    for i in range(len(box)):
        others = np.arange(len(box)) != i
        assert not spec.iou_ge(box[i], ar[i], box[others], ar[others], 1e-6).any(), "boxes must not overlap"


@pytest.mark.parametrize("conf", dec.TABLE_CONF, ids=[repr(float(c)) for c in dec.TABLE_CONF])
def test_spec_candidates_equal_the_oracle_on_the_truth_table(conf):
    nc = dec.TABLE_NUM_CLASSES
    cand = spec.candidates(TABLE, nc, conf)
    assert np.array_equal(np.argwhere(dec.literal_pairs(TABLE, nc, conf)), np.stack([cand["row"], cand["cls"]], 1).reshape(-1, 2))
    # no box overlaps another, so per-class NMS keeps every candidate and the oracle's rows are exactly the candidates
    want = spec.rows_of(cand, np.arange(len(cand["row"])))
    got = orc.postprocess(TABLE[None], nc, conf, 0.45)[0]
    assert (got is None) == (want is None)
    if want is not None:
        assert _bits_equal(got, want)


def _obj_of(rows):
    return TABLE[rows, 4]


def test_the_old_shortcut_disagrees_exactly_at_zero_and_infinite_objectness():
    nc = dec.TABLE_NUM_CLASSES
    wrong_rows = set()
    for conf in dec.TABLE_CONF:
        lit = dec.literal_pairs(TABLE, nc, conf)
        old = dec.shortcut_pairs(TABLE, nc, conf, dec.shortcut_before_fix)
        assert not (lit & ~old).any(), "the shortcut only adds candidates"
        extra = np.nonzero((old & ~lit).any(1))[0]
        obj = _obj_of(extra)
        assert ((obj == 0) | (obj == np.inf)).all(), f"conf {conf}: extra rows with obj {obj}"
        wrong_rows.update((float(conf), int(r)) for r in extra)
    n_max = len(dec.TABLE_MAX)

    def row(obj, mx):
        return [i for i, o in enumerate(dec.TABLE_OBJ) if _bits_equal(o, obj)][0] * n_max + \
            [i for i, m in enumerate(dec.TABLE_MAX) if _bits_equal(m, mx)][0]

    # obj = +-0, classes [+inf, 0.25], conf 0: 0 * inf is NaN, so the reference drops the row; 0 * 0.25 >= 0 passes
    assert (0.0, row(dec.F32(0), dec.INF)) in wrong_rows and (0.0, row(dec.F32(-0.0), dec.INF)) in wrong_rows
    # obj = +inf, classes [0, -0.5], conf -inf: inf * 0 is NaN; inf * -0.5 = -inf >= -inf passes
    assert (float("-inf"), row(dec.INF, dec.F32(0))) in wrong_rows


@pytest.mark.parametrize("conf", dec.TABLE_CONF, ids=[repr(float(c)) for c in dec.TABLE_CONF])
def test_the_fixed_shortcut_agrees_with_the_literal_filter(conf):
    nc = dec.TABLE_NUM_CLASSES
    assert np.array_equal(dec.shortcut_pairs(TABLE, nc, conf, dec.shortcut_fixed), dec.literal_pairs(TABLE, nc, conf))


def test_the_fixed_shortcut_agrees_on_random_rows_with_special_values():
    rng = np.random.RandomState(3)
    pool = np.array(dec.TABLE_OBJ + dec.TABLE_MAX + [np.float32(0.25), np.float32(-2)], np.float32)
    for nc in (1, 3, 6):
        pred = np.zeros((4000, 11), np.float32)
        pred[:, 4:] = np.where(rng.rand(4000, 7) < 0.5, rng.choice(pool, (4000, 7)), rng.rand(4000, 7).astype(np.float32))
        for conf in dec.TABLE_CONF:
            assert np.array_equal(dec.shortcut_pairs(pred, nc, conf, dec.shortcut_fixed), dec.literal_pairs(pred, nc, conf))
