"""CPU-only checks of the drop-in boundary: the C-ABI library builds, loads and exports every symbol that
include/yolo_head.h declares; host-side argument validation needs no GPU."""
import ctypes
import os
import re
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "yolo_head.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(yl_[a-z_0-9]+)\s*\(", text)))


def test_library_builds_loads_and_exports_header_symbols():
    from yolov4_b200 import _cabi, build
    path = build.build_lib()
    assert os.path.exists(path)
    L = ctypes.CDLL(path)
    declared = _declared_symbols()
    assert len(declared) >= 14
    for name in declared:
        assert hasattr(L, name), "libyolohead.so does not export %s" % name
    assert sorted(_cabi.EXPORTS) == declared
    assert _cabi.lib().yl_abi_version() == 1


def test_pure_host_entry_points_without_gpu():
    from yolov4_b200 import _cabi
    L = _cabi.lib()
    # workspace sizing is host arithmetic
    n = L.yl_post_workspace_bytes(64, 22743, 80, 1024)
    assert n > 64 * 80 * 1024 * 16
    assert L.yl_post_workspace_bytes(64, 22743, 80, 4096) > n
    assert L.yl_post_workspace_bytes(0, 1, 1, 1) == 0
    assert L.yl_error_string(0) == b"ok"
    assert b"cap_seg" in L.yl_error_string(4)
    # argument validation happens before any CUDA call
    assert L.yl_filter_dense(None, 1, 10, 80, 80, 0.5, None, 0, 16, 0, 1, None) == 1
    assert L.yl_build_target(None, None, None, 1, 4, 60, 80, 0, None, None, 0.7, None, None, None, None, None, None) == 1


def test_host_wrappers_reject_cpu_and_wrong_dtype():
    import yolov4_b200 as yb
    cfg = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": 80}
    layer = yb.YOLOLayer(cfg, 1)
    assert layer.stride == 16 and layer.n_anchors == 3 and layer.masked_anchors.dtype == torch.float64
    assert len(list(layer.state_dict().keys())) == 0            # checkpoints load unchanged (val.py:82-83)
    with pytest.raises(TypeError):
        layer.eval()(torch.zeros(1, 255, 4, 4))
    with pytest.raises(ValueError):
        layer.eval()(torch.zeros(1, 254, 4, 4))
    with pytest.raises(TypeError):
        yb.postprocess(torch.zeros(1, 10, 85, dtype=torch.float64), 80)
    with pytest.raises(ValueError):
        yb.postprocess(torch.zeros(10, 85), 80)
    with pytest.raises(TypeError):
        yb.detect_raw([torch.zeros(1, 255, 4, 4)], 80)


def test_synth_generator_is_seeded_and_shaped():
    from yolov4_b200.synth import synth_head_outputs, synth_labels
    a = synth_head_outputs(2, 96, 80, seed=3)
    b = synth_head_outputs(2, 96, 80, seed=3)
    assert [tuple(t.shape) for t in a] == [(2, 255, 12, 12), (2, 255, 6, 6), (2, 255, 3, 3)]
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    lab = synth_labels(3, 608, n_valid=50)
    assert lab.shape == (3, 60, 5) and (lab[:, 50:] == 0).all() and (lab[:, :50, 2:4] > 0).all()


def test_bench_reference_arm_prints_exactly_one_json_line():
    """The driver parses stdout of bench.py: one JSON line, nothing else (library banners go to stderr)."""
    import json
    import subprocess
    import sys
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-seconds", "0.5"], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout[:2000]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["higher_is_better"] is True
    # the unmodified reference when it is installed under baseline/_ref (tools/install_reference.sh), else the oracle's C port
    have_ref = os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "yolo"))
    assert d["cpu_baseline"]["kind"] == ("reference" if have_ref else "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline_port"]["kind"] == "port" and d["cpu_baseline_port"]["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]


def _stand_in_reference(monkeypatch):
    """The reference's module layout as far as patch_reference() touches it (yolo/model/yololayer.py, yolo/util/utils.py,
    yolo/model/yololoss.py, and yolo/model/yolov4.py, which imports YOLOLayer by name), with placeholder bodies: what is
    checked here is the rebinding, not the reference's arithmetic.  yolo.engine is left out, as where apex is not installed."""
    import types

    class YOLOLayer(torch.nn.Module):
        pass

    class YOLOLoss(torch.nn.Module):
        def build_target(self, *args):
            raise NotImplementedError

        def forward(self, *args):
            raise NotImplementedError

    def postprocess(*args):
        raise NotImplementedError

    mods = {n: types.ModuleType(n) for n in ("yolo", "yolo.model", "yolo.util", "yolo.model.yololayer", "yolo.util.utils",
                                             "yolo.model.yololoss", "yolo.model.yolov4")}
    mods["yolo.model.yololayer"].YOLOLayer = YOLOLayer
    mods["yolo.model.yolov4"].YOLOLayer = YOLOLayer
    mods["yolo.util.utils"].postprocess = postprocess
    mods["yolo.model.yololoss"].YOLOLoss = YOLOLoss
    for name, m in mods.items():
        monkeypatch.setitem(sys.modules, name, m)
        if "." in name:
            parent, _, child = name.rpartition(".")
            setattr(mods[parent], child, m)


def test_patch_reference_rebinds_the_boundary_symbols(monkeypatch):
    """patch_reference() against the installed reference (baseline/_ref), else against stand-ins of its module layout: every symbol
    of the drop-in boundary (SURVEY 8b) is rebound to the B200 implementation -- no CUDA needed to check the binding itself.
    (Round 1 shipped a patch_reference() that raised on its second line: `from . import postprocess` returns the re-exported
    FUNCTION.)"""
    import importlib
    ref = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(os.path.join(ref, "yolo")):
        monkeypatch.syspath_prepend(ref)
    else:
        _stand_in_reference(monkeypatch)
    import yolov4_b200 as yb
    ml = importlib.import_module("yolo.model.yololayer")
    mu = importlib.import_module("yolo.util.utils")
    mlo = importlib.import_module("yolo.model.yololoss")
    m4 = importlib.import_module("yolo.model.yolov4")
    saved = (ml.YOLOLayer, mu.postprocess, mlo.YOLOLoss.build_target, mlo.YOLOLoss.forward, m4.YOLOLayer)
    try:
        done = yb.patch_reference(loss_forward=False)
        assert ml.YOLOLayer is yb.YOLOLayer and m4.YOLOLayer is yb.YOLOLayer
        assert mu.postprocess is importlib.import_module("yolov4_b200.postprocess").postprocess
        assert mlo.YOLOLoss.build_target is yb.YOLOLoss.build_target
        assert mlo.YOLOLoss.forward is saved[3] and "yolo.model.yololoss.YOLOLoss.forward" not in done
        done = yb.patch_reference()
        assert mlo.YOLOLoss.forward is yb.YOLOLoss.forward and "yolo.model.yololoss.YOLOLoss.forward" in done
        # the patched class still builds without CUDA and carries no state (checkpoints load unchanged, val.py:82-83)
        layer = ml.YOLOLayer({"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": 80}, 1)
        assert len(layer.state_dict()) == 0 and layer.stride == 16
    finally:
        ml.YOLOLayer, mu.postprocess, mlo.YOLOLoss.build_target, mlo.YOLOLoss.forward, m4.YOLOLayer = saved


def test_source_hash_staleness_detection(tmp_path):
    """The loader never uses a library built from other sources: build.is_stale() compares a hash of csrc/ + include/ with the one
    recorded next to the library (file times do not survive a snapshot copy)."""
    from yolov4_b200 import build as b
    assert not b.is_stale(), "the tests run against a library built from the current sources"
    h = b.source_hash()
    assert len(h) == 16 and h == open(b.LIB + ".srchash").read().strip()
    from yolov4_b200 import _cabi
    assert _cabi.lib().yl_source_hash().decode() == h
