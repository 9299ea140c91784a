"""Measures class-agnostic NMS on the fused detection path against the per-class back end it replaces; prints one JSON line.

Workloads: B=64 @608, 80 classes, fp32 heads from synth_head_outputs (seed 0), at conf 1e-4 / nms 0.4 and at conf 0.2 / nms 0.5.
The inputs (495 MB) exceed the 126 MB L2, so the streaming filter passes read from HBM.

For each workload, agnostic and per-class:
  kernels_us        median device time per launch of every back-end kernel, from torch.profiler (CUDA activities) over
                    --prof-runs HeadPostprocessor.run() calls, in a profiling pass of its own; backend_us is their sum
                    (agnostic: k_segment_nms_agnostic + k_gather_rows; per-class: k_segment_nms_bins + k_segment_nms_big +
                    k_gather_rows)
  step_alone_us     one graph-replayed step (HeadPostprocessor.capture / replay), CUDA events over --iters replays
  step_3_in_flight  three graph-replayed steps in flight on three streams, as bench.py runs them
  rows              detections of the batch
The first --check-images images of each agnostic result are checked bit for bit against tests/agnostic_spec.py (the literal
algorithm, on the CPU), which also gives their candidate, distinct-box and kept counts; the script exits non-zero on a difference.

  python tools/agnostic_probe.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

IMG, C, B = 608, 80, 64
GRIDS = [IMG // 8, IMG // 16, IMG // 32]
WORKLOADS = [(1e-4, 0.4), (0.2, 0.5)]
KERNELS = ["k_segment_nms_agnostic", "k_segment_nms_bins", "k_segment_nms_big", "k_gather_rows", "k_flag_raw", "k_flag_tma",
           "k_emit_flagged"]
BACKEND = {True: ["k_segment_nms_agnostic", "k_gather_rows"], False: ["k_segment_nms_bins", "k_segment_nms_big", "k_gather_rows"]}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        name, power = [x.strip() for x in out[torch.cuda.current_device()].split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:  # the reading is informative; the measurement does not depend on it
        return {"name": torch.cuda.get_device_name(), "power_limit": "unknown (%s)" % type(e).__name__}


def time_events(fn, iters, warm=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / iters


def step3_time(hps, iters):
    streams = [torch.cuda.Stream() for _ in range(3)]
    state = {"i": 0}

    def step3():
        p = state["i"] % 3
        with torch.cuda.stream(streams[p]):
            hps[p].replay()
        state["i"] += 1

    main = torch.cuda.current_stream()
    for s in streams:
        s.wait_stream(main)
    for _ in range(6):
        step3()
    for s in streams:
        main.wait_stream(s)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in streams:
        s.wait_stream(main)
    for _ in range(iters):
        step3()
    for s in streams:
        main.wait_stream(s)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / iters


def kernel_times(hp, raws, runs):
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        hp.run(raws)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(runs):
            hp.run(raws)
        torch.cuda.synchronize()
    durs = {k: [] for k in KERNELS}
    for ev in prof.events():
        for k in KERNELS:
            if k in ev.name and str(ev.device_type).endswith("CUDA"):
                durs[k].append(ev.time_range.elapsed_us())
    return {k: float(np.median(v)) for k, v in durs.items() if v}


def bits_equal(a, b):
    if (a is None) != (b is None):
        return False
    if a is None:
        return True
    a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def measure(yb, spec, orc, conf, nms, args):
    from yolov4_b200.synth import synth_head_outputs
    raws = synth_head_outputs(B, IMG, C, seed=0, device="cuda")
    out = {"B": B, "conf": conf, "nms": nms}
    results = {}
    for agn in (True, False):
        hps = [yb.HeadPostprocessor(B, GRIDS, C, conf, nms, agnostic=agn).capture(raws) for _ in range(3)]
        t_step = time_events(lambda: hps[0].replay(), args.iters)
        t_step3 = step3_time(hps, args.iters)
        hps[0].replay()
        torch.cuda.synchronize()
        results[agn] = hps[0].results()
        kern = kernel_times(hps[0], raws, args.prof_runs)
        out["agnostic" if agn else "per_class"] = {
            "kernels_us": kern, "backend_us": sum(kern.get(k, 0.0) for k in BACKEND[agn]),
            "step_alone_us": 1e6 * t_step, "step_3_in_flight_us": 1e6 * t_step3,
            "step_3_in_flight_images_per_s": B / t_step3,
            "rows": int(sum(0 if r is None else len(r) for r in results[agn]))}
        del hps
        torch.cuda.empty_cache()
    n = args.check_images
    dense = orc.decode_eval_cat([r[:n].cpu().numpy() for r in raws], C)
    checked = []
    for b in range(n):
        cand = spec.candidates(dense[b], C, conf)
        want = spec.rows_of(cand, spec.agnostic_kept(cand, nms))
        checked.append({"image": b, "candidates": int(len(cand["s"])), "distinct_boxes": int(len(np.unique(cand["row"]))),
                        "agnostic_kept": 0 if want is None else int(len(want)),
                        "per_class_kept": 0 if results[False][b] is None else int(len(results[False][b])),
                        "equal_to_spec": bool(bits_equal(results[True][b], want))})
    out["checked_images"] = checked
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--prof-runs", type=int, default=30)
    ap.add_argument("--check-images", type=int, default=4)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("agnostic_probe.py measures on a GPU; there is none here")
    import yolov4_b200 as yb
    from oracle import oracle as orc
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import agnostic_spec as spec
    res = {"probe": "agnostic_probe", "workload": "B=%d @%d, %d classes, fp32 synth_head_outputs seed 0" % (B, IMG, C),
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
        raise SystemExit("parity check failed: an agnostic result differs from the literal algorithm")


if __name__ == "__main__":
    main()
