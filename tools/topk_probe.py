"""Measures the per-image detection cap (max_det) on the fused detection path and prints one JSON line.

Workloads: B=64 @608 at conf 1e-4 / nms 0.4 (about 11.5k kept rows per image) and B=256 @608 at conf 0.2 / nms 0.5, 80 classes,
fp32 heads from synth_head_outputs (seed 0), each with max_det None (uncapped), 100 and 300.  Every capped result is checked
bit for bit in the same run against tests/cap_spec.py:cap_detections applied to the uncapped result; the script exits non-zero on a
difference.

For each (workload, max_det):
  kernels_us        median device time per launch of k_select_topk, k_gather_rows and the two NMS kernels, from torch.profiler
                    (CUDA activities) over --prof-runs HeadPostprocessor.run() calls, in a profiling pass of its own
  step_alone_us     one graph-replayed step (HeadPostprocessor.capture / replay), CUDA events over --iters replays
  step_3_in_flight  three graph-replayed steps in flight on three streams, as bench.py runs them
  gather_bytes      bytes of rows the gather writes per step (sum of the per-image row counts x 28)
  host_leg          yl_detect_host_topk from pinned host buffers, images/s
  exchange          single-rank DetectionExchange (self window) push + wait + release per step with cap_out = hp.cap_out,
                    CUDA events; with one GPU the multi-rank exchange is not measured
The inputs (495 MB at B=64, 1.98 GB at B=256) exceed the 126 MB L2, so the streaming passes read from HBM.

  python tools/topk_probe.py [--out FILE]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

IMG, C = 608, 80
GRIDS = [IMG // 8, IMG // 16, IMG // 32]
WORKLOADS = [(64, 1e-4, 0.4), (256, 0.2, 0.5)]
CAPS = [None, 100, 300]
KERNELS = ["k_segment_nms_bins", "k_segment_nms_big", "k_select_topk", "k_gather_rows"]


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


def rows_equal(a, b):
    if len(a) != len(b):
        return False
    for x, y in zip(a, b):
        if (x is None) != (y is None):
            return False
        if x is None:
            continue
        x = x.cpu().numpy() if isinstance(x, torch.Tensor) else x
        y = y.cpu().numpy() if isinstance(y, torch.Tensor) else y
        if x.shape != y.shape or not np.array_equal(x.view(np.uint32), y.view(np.uint32)):
            return False
    return True


def kernel_times(hp, raws, runs):
    """Median device time per launch of each back-end kernel, from torch.profiler."""
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
    return {k: (float(np.median(v)) if v else None) for k, v in durs.items()}


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


def host_leg(yb, _cabi, raws, B, conf, nms, max_det, steps):
    L = _cabi.lib()
    host = [r.cpu().pin_memory() for r in raws]
    cap_out = 16384 if max_det is None else (max_det + 3) // 4 * 4
    ctx = ctypes.c_void_p()
    anch = _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh])
    mask = _cabi.ints([v for m in yb.ANCHOR_MASK for v in m])
    _cabi.check(L.yl_context_create_typed(ctypes.byref(ctx), torch.cuda.current_device(), B, _cabi.ints(GRIDS), 3, C, 0, anch,
                                          mask, 1024, cap_out))
    try:
        rows = torch.empty((B, cap_out, 7), dtype=torch.float32).pin_memory()
        cnt = torch.zeros((B,), dtype=torch.int32).pin_memory()
        ptrs = _cabi.ptrs([h.data_ptr() for h in host])
        f32 = lambda v: float(np.float32(v))  # noqa: E731
        call = lambda: _cabi.check(L.yl_detect_host_topk(ctx, ptrs, f32(conf), f32(nms), max_det or 0, rows.data_ptr(),  # noqa: E731
                                                         cnt.data_ptr()))
        for _ in range(3):
            call()
        t0 = time.perf_counter()
        for _ in range(steps):
            call()
        torch.cuda.synchronize()
        sec = (time.perf_counter() - t0) / steps
        res = [rows[b, :int(cnt[b])].clone() if int(cnt[b]) else None for b in range(B)]
    finally:
        _cabi.check(L.yl_context_destroy(ctx))
    return {"images_per_s": B / sec, "ms_per_call": 1e3 * sec}, res


def exchange_time(hp, iters):
    from yolov4_b200.sharded import DetectionExchange
    ex = DetectionExchange(hp.B, hp.cap_out, hp.device, slots=2)
    try:
        state = {"i": 0}

        def step():
            slot = state["i"] % 2
            ex.push(hp.rows, hp.meta[:hp.B], slot)
            ex.wait(slot)
            ex.release(slot)
            state["i"] += 1
        t = time_events(step, 200)
        ok = ex.status() == 0
    finally:
        ex.close()
    return {"push_wait_release_us": 1e6 * t, "cap_out": hp.cap_out, "status_ok": ok, "world": 1}


def measure(yb, _cabi, cap_detections, B, conf, nms, args):
    from yolov4_b200.synth import synth_head_outputs
    raws = synth_head_outputs(B, IMG, C, seed=0, device="cuda")
    out = {"B": B, "conf": conf, "nms": nms, "per_max_det": {}}
    uncapped = None
    for K in CAPS:
        hps = [yb.HeadPostprocessor(B, GRIDS, C, conf, nms, max_det=K).capture(raws) for _ in range(3)]
        t_step = time_events(lambda: hps[0].replay(), args.iters)
        t_step3 = step3_time(hps, args.iters)
        hps[0].replay()
        torch.cuda.synchronize()
        got = hps[0].results()
        counts = hps[0].meta[:B].cpu().numpy()
        kern = kernel_times(hps[0], raws, args.prof_runs)
        host, host_rows = host_leg(yb, _cabi, raws, B, conf, nms, K, args.host_steps)
        xchg = exchange_time(hps[0], args.iters) if B <= 64 else None
        entry = {"kernels_us": kern, "step_alone_us": 1e6 * t_step, "step_3_in_flight_us": 1e6 * t_step3,
                 "step_3_in_flight_images_per_s": B / t_step3, "gather_bytes": int(counts.sum()) * 28,
                 "rows_buffer_bytes": B * hps[0].cap_out * 28, "host_leg": host, "exchange_single_rank": xchg,
                 "detections": int(counts.sum())}
        if K is None:
            uncapped = got
            entry["host_rows_equal_graph_rows"] = bool(rows_equal(host_rows, got))
        else:
            want = cap_detections(uncapped, K)
            entry["parity_vs_spec"] = bool(rows_equal(got, want) and rows_equal(host_rows, want))
            entry["images_capped"] = int((hps[0].uncapped.cpu().numpy() > K).sum())
        out["per_max_det"][str(K)] = entry
        del hps
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--prof-runs", type=int, default=30)
    ap.add_argument("--host-steps", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("topk_probe.py measures on a GPU; there is none here")
    import yolov4_b200 as yb
    from yolov4_b200 import _cabi
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from cap_spec import cap_detections
    res = {"probe": "topk_probe", "workload": "@%d, %d classes, fp32 synth_head_outputs seed 0" % (IMG, C), "gpu": gpu_info(),
           "gpus_visible": torch.cuda.device_count(),
           "multi_rank_exchange": "not measured (this probe times the single-rank exchange only)",
           "settings": [measure(yb, _cabi, cap_detections, B, conf, nms, args) for B, conf, nms in WORKLOADS]}
    ok = all(e.get("parity_vs_spec", True) and e.get("host_rows_equal_graph_rows", True)
             for s in res["settings"] for e in s["per_max_det"].values())
    res["parity_ok"] = ok
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if not ok:
        raise SystemExit("parity check failed: a capped result differs from cap_detections of the uncapped result")


if __name__ == "__main__":
    main()
