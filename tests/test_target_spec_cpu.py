"""CPU-only: the C oracle's build_target against the literal NumPy statement of the reference's scatter (target_spec) on the
hostile label sets of loss_edge_cases -- negative and fractional class ids, collisions, K = 256, zero and non-positive rows
among the first n, cell edges, out-of-grid centres, degenerate extents, ignore thresholds, class counts and anchor masks.
Masks and targets must agree bit for bit (any NaN equals any NaN), and IndexError must be raised in exactly the same cases."""
import numpy as np
import pytest

import loss_edge_cases as cases
import target_spec as spec
from oracle import oracle as orc


def bit_equal(a, b):
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(a.view(np.uint32)[~na], b.view(np.uint32)[~nb])


def _run(fn, *args, **kw):
    try:
        return fn(*args, **kw)
    except IndexError:
        return IndexError


@pytest.mark.parametrize("name", sorted(cases.VALID) + sorted(cases.ERROR))
def test_spec_equals_oracle(name):
    c = cases.get(name)
    C, mask, lab = c["C"], c["mask"], c["labels"]
    raised = []
    for l in range(3):
        _, pred = orc.decode_train(c["raws"][l], l, C, mask=mask)
        for thr in c["thrs"]:
            want = _run(orc.build_target, pred, lab, l, C, thr, mask=mask)
            got = _run(spec.build_target, pred, lab, l, C, thr, mask=mask)
            assert (got is IndexError) == (want is IndexError), (name, l, thr)
            raised.append(want is IndexError)
            if want is IndexError:
                continue
            for what, g, w in zip(("target", "obj_mask", "tgt_mask", "tgt_scale"), got, want):
                assert bit_equal(g, w), "%s layer %d thr %r: %s differs" % (name, l, thr, what)
    assert any(raised) == c["error"], "%s: the reference %s raise" % (name, "does not" if c["error"] else "does")


def test_class_id_wrap_lands_where_python_indexing_puts_it():
    """One GT, every class id in [-(10+C), C): the one-hot channel is 5 + cls, wrapped once by the row length."""
    C, img = 4, 96
    raws = cases.heads(1, img, C, seed=3)
    _, pred = orc.decode_train(raws[0], 0, C)
    base = np.zeros((1, 2, 5), np.float32)
    base[0, 0] = (40.3, 50.7, 20.0, 30.0, 0.0)
    t0, _, _, _ = orc.build_target(pred, base, 0, C)
    cell = tuple(np.argwhere(t0[0, ..., 4] == 1)[0])
    for cid in range(-(10 + C), C):
        lab = base.copy()
        lab[0, 0, 4] = cid
        t, _, _, _ = spec.build_target(pred, lab, 0, C)
        want = t0[(0,) + cell].copy()
        want[5:] = 0
        want[(5 + cid) % (5 + C)] = 1
        assert bit_equal(t[(0,) + cell], want), cid
    for cid in (C, C + 5, -(11 + C)):
        lab = base.copy()
        lab[0, 0, 4] = cid
        with pytest.raises(IndexError):
            spec.build_target(pred, lab, 0, C)
