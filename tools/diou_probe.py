"""Measures DIoU-NMS on the fused detection path against IoU-NMS, per class and agnostic; prints one JSON line.

Workloads: B=64 @608, 80 classes, fp32 heads from synth_head_outputs (seed 0), at conf 1e-4 / nms 0.4 and at conf 0.2 / nms 0.5.
The inputs (495 MB) exceed the 126 MB L2, so the streaming filter passes read from HBM.

For each workload and each of the four modes (per_class_iou, per_class_diou, agnostic_iou, agnostic_diou):
  kernels_us        median device time per launch of every back-end kernel, from torch.profiler (CUDA activities) over
                    --prof-runs HeadPostprocessor.run() calls, in a profiling pass of its own; backend_us is their sum
  step_alone_us     one graph-replayed step (HeadPostprocessor.capture / replay), CUDA events over --iters replays
  step_3_in_flight  three graph-replayed steps in flight on three streams, as bench.py runs them
  rows              detections of the batch
The first --check-images images of each DIoU result are checked bit for bit against tests/diou_spec.py (the literal algorithm,
on the CPU); the script exits non-zero on a difference.

  python tools/diou_probe.py [--out FILE]
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

from agnostic_probe import bits_equal, gpu_info, kernel_times, step3_time, time_events  # noqa: E402

IMG, C, B = 608, 80, 64
GRIDS = [IMG // 8, IMG // 16, IMG // 32]
WORKLOADS = [(1e-4, 0.4), (0.2, 0.5)]
MODES = {"per_class_iou": (False, False), "per_class_diou": (False, True), "agnostic_iou": (True, False), "agnostic_diou": (True, True)}
BACKEND = {True: ["k_segment_nms_agnostic", "k_gather_rows"], False: ["k_segment_nms_bins", "k_segment_nms_big", "k_gather_rows"]}


def measure(yb, spec, orc, conf, nms, args):
    from yolov4_b200.synth import synth_head_outputs
    raws = synth_head_outputs(B, IMG, C, seed=0, device="cuda")
    out = {"B": B, "conf": conf, "nms": nms}
    results = {}
    for mode, (agn, diou) in MODES.items():
        hps = [yb.HeadPostprocessor(B, GRIDS, C, conf, nms, agnostic=agn, diou=diou).capture(raws) for _ in range(3)]
        t_step = time_events(lambda: hps[0].replay(), args.iters)
        t_step3 = step3_time(hps, args.iters)
        hps[0].replay()
        torch.cuda.synchronize()
        results[mode] = hps[0].results()
        kern = kernel_times(hps[0], raws, args.prof_runs)
        out[mode] = {"kernels_us": kern, "backend_us": sum(kern.get(k, 0.0) for k in BACKEND[agn]),
                     "step_alone_us": 1e6 * t_step, "step_3_in_flight_us": 1e6 * t_step3,
                     "step_3_in_flight_images_per_s": B / t_step3,
                     "rows": int(sum(0 if r is None else len(r) for r in results[mode]))}
        del hps
        torch.cuda.empty_cache()
    n = args.check_images
    dense = orc.decode_eval_cat([r[:n].cpu().numpy() for r in raws], C)
    checked = []
    for b in range(n):
        for agn in (False, True):
            mode = "agnostic_diou" if agn else "per_class_diou"
            want = spec.postprocess(dense[b:b + 1], C, conf, nms, agn)[0]
            checked.append({"image": b, "mode": mode, "rows": 0 if want is None else int(len(want)),
                            "iou_rows": 0 if results[mode.replace("diou", "iou")][b] is None else
                            int(len(results[mode.replace("diou", "iou")][b])),
                            "equal_to_spec": bool(bits_equal(results[mode][b], want))})
    out["checked_images"] = checked
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--prof-runs", type=int, default=30)
    ap.add_argument("--check-images", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("diou_probe.py measures on a GPU; there is none here")
    import yolov4_b200 as yb
    from oracle import oracle as orc
    import diou_spec as spec
    res = {"probe": "diou_probe", "workload": "B=%d @%d, %d classes, fp32 synth_head_outputs seed 0" % (B, IMG, C),
           "gpu": gpu_info(), "settings": [measure(yb, spec, orc, conf, nms, args) for conf, nms in WORKLOADS]}
    ok = all(c["equal_to_spec"] for s in res["settings"] for c in s["checked_images"])
    res["parity_ok"] = ok
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if not ok:
        raise SystemExit("parity check failed: a DIoU result differs from the literal algorithm")


if __name__ == "__main__":
    main()
