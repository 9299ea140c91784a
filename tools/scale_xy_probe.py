"""Measures YOLOv4's grid-sensitivity decode (scale_x_y) against the plain decode on every kernel it touches; prints one JSON line.

Detection: B=64 @608, 80 classes, fp32 heads from synth_head_outputs (seed 0), at conf 1e-4 / nms 0.4 and at conf 0.2 / nms 0.5,
scale_x_y None against yolov4.cfg's (1.2, 1.1, 1.05).  The inputs (495 MB) exceed the 126 MB L2.  For each:
  emit_us           median device time of k_emit_flagged per launch, torch.profiler (CUDA activities), in a pass of its own
  step_alone_us     one graph-replayed HeadPostprocessor step, CUDA events over --iters replays
  step_3_in_flight  three graph-replayed steps in flight on three streams, as bench.py runs them
  rows              detections of the batch
Dense decode: k_decode_dense of each of the three scales (yl_decode_dense_ex), median per launch under torch.profiler.
Fused loss: forward and forward + backward of fused_yolo_loss(iou_loss='ciou'), B=64 @608, 50 GTs per image, fp32 and fp16
heads, with and without the scales, CUDA events.
The first --check-images images of each scaled detection result are checked bit for bit against the literal algorithm on the
spec-decoded tensor (tests/scale_xy_spec.py + the oracle's postprocess); the script exits non-zero on a difference.

  python tools/scale_xy_probe.py [--out FILE]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from agnostic_probe import bits_equal, gpu_info, step3_time, time_events  # noqa: E402

IMG, C, B = 608, 80, 64
GRIDS = [IMG // 8, IMG // 16, IMG // 32]
WORKLOADS = [(1e-4, 0.4), (0.2, 0.5)]
YOLOV4 = (1.2, 1.1, 1.05)


def profiled(fn, runs, names):
    """Median device time per launch (us) of every kernel whose name contains one of `names`, over `runs` calls of fn."""
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(runs):
            fn()
        torch.cuda.synchronize()
    durs = {k: [] for k in names}
    for ev in prof.events():
        for k in names:
            if k in ev.name and str(ev.device_type).endswith("CUDA"):
                durs[k].append(ev.time_range.elapsed_us())
    return {k: float(np.median(v)) for k, v in durs.items() if v}


def detection(yb, raws, conf, nms, args):
    out = {"conf": conf, "nms": nms}
    res = {}
    for name, sxy in (("plain", None), ("scaled", YOLOV4)):
        hps = [yb.HeadPostprocessor(B, GRIDS, C, conf, nms, scale_x_y=sxy).capture(raws) for _ in range(3)]
        t1 = time_events(lambda: hps[0].replay(), args.iters)
        t3 = step3_time(hps, args.iters)
        hps[0].replay()
        torch.cuda.synchronize()
        res[name] = hps[0].results()
        emit = profiled(lambda: hps[0].run(raws), args.prof_runs, ["k_emit_flagged"])
        out[name] = {"emit_us": emit.get("k_emit_flagged"), "step_alone_us": 1e6 * t1, "step_3_in_flight_us": 1e6 * t3,
                     "rows": int(sum(0 if r is None else len(r) for r in res[name]))}
        del hps
        torch.cuda.empty_cache()
    return out, res["scaled"]


def check(orc, spec, raws, conf, nms, got, n):
    dense = spec.decode_eval_cat([r[:n].cpu().numpy() for r in raws], C, YOLOV4)
    want = orc.postprocess(dense, C, conf, nms, nthreads=8)
    return [{"image": b, "rows": 0 if want[b] is None else int(len(want[b])),
             "equal_to_spec": bool((got[b] is None and want[b] is None) or
                                   (got[b] is not None and want[b] is not None and bits_equal(got[b].cpu().numpy(), want[b])))}
            for b in range(n)]


def dense_decode(yb, raws, args):
    from yolov4_b200 import _cabi
    L = _cabi.lib()
    M = sum(3 * f * f for f in GRIDS)
    out = torch.empty((B, M, 5 + C), dtype=torch.float32, device="cuda")
    res = {}
    for name, sxy in (("plain", (1.0, 1.0, 1.0)), ("scaled", YOLOV4)):
        per = {}
        off = 0
        for l, r in enumerate(raws):
            s = 8 << l
            anch = _cabi.floats([v / s for i in yb.ANCHOR_MASK[l] for v in yb.ANCHORS_PX[i]])

            def call(l=l, r=r, off=off, anch=anch, s=s):
                _cabi.check(L.yl_decode_dense_ex(r.data_ptr(), B, GRIDS[l], C, anch, float(s), sxy[l], out.data_ptr(), M, off,
                                                 torch.cuda.current_stream().cuda_stream))
            per["F%d" % GRIDS[l]] = profiled(call, args.prof_runs, ["k_decode_dense"]).get("k_decode_dense")
            off += 3 * GRIDS[l] ** 2
        res[name] = per
    return res


def loss(yb, args):
    from yolov4_b200.synth import synth_labels
    from yolov4_b200.yololoss import fused_yolo_loss
    import loss_edge_cases as cases
    from oracle import oracle as orc
    cfg = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": C}
    lab_np = synth_labels(B, IMG, n_valid=50, seed=1).numpy()
    raws = cases.heads(B, IMG, C, 1)
    cases.plant_near_gts(raws, lab_np, C, orc.ANCHOR_MASK, every=2)
    lab = torch.from_numpy(np.ascontiguousarray(lab_np, np.float32)).cuda()
    out = {}
    for dt in (torch.float32, torch.float16):
        heads = [torch.from_numpy(r).cuda().to(dt).requires_grad_(True) for r in raws]
        for name, sxy in (("plain", None), ("scaled", YOLOV4)):
            kw = dict(iou_loss="ciou", scale_x_y=sxy)

            def fwd():
                with torch.no_grad():
                    fused_yolo_loss(heads, lab, cfg, **kw)

            def fwd_bwd():
                fused_yolo_loss(heads, lab, cfg, **kw).backward()
            out["%s_%s" % (str(dt).split(".")[1], name)] = {"forward_us": 1e6 * time_events(fwd, args.iters),
                                                            "forward_backward_us": 1e6 * time_events(fwd_bwd, args.iters)}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--prof-runs", type=int, default=30)
    ap.add_argument("--check-images", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("scale_xy_probe.py measures on a GPU; there is none here")
    import yolov4_b200 as yb
    from oracle import oracle as orc
    import scale_xy_spec as spec
    from yolov4_b200.synth import synth_head_outputs
    raws = synth_head_outputs(B, IMG, C, seed=0, device="cuda")
    res = {"probe": "scale_xy_probe", "workload": "B=%d @%d, %d classes, fp32 synth_head_outputs seed 0; scale_x_y %r" % (
        B, IMG, C, YOLOV4), "gpu": gpu_info(), "detection": []}
    checked = []
    for conf, nms in WORKLOADS:
        d, got = detection(yb, raws, conf, nms, args)
        d["checked_images"] = check(orc, spec, raws, conf, nms, got, args.check_images)
        checked += d["checked_images"]
        res["detection"].append(d)
    res["k_decode_dense_us"] = dense_decode(yb, raws, args)
    del raws
    torch.cuda.empty_cache()
    res["fused_loss_ciou_50gt"] = loss(yb, args)
    ok = all(c["equal_to_spec"] for c in checked)
    res["parity_ok"] = ok
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if not ok:
        raise SystemExit("parity check failed: a scaled detection result differs from the literal algorithm")


if __name__ == "__main__":
    main()
