"""Where the time of k_segment_nms_bins (the small NMS tier) goes on the bench workload; prints one JSON line.

Workload: B=64 @608, 80 classes, fp32 synth_head_outputs (seed 0), conf 1e-4 / nms 0.4, as bench.py runs it.

  phase_cycles      probe build (-DYL_NMS_PROBE): thread 0 of every CTA adds the clock64() cycles of each phase, each closed
                    by a barrier, into a device array; reported per CTA that ran the small tier to the end, with the share of
                    the sum.  The barriers the probe adds make the kernel slower than the library's: read the shares.
  counts            per such CTA: records, queued candidate pairs, rows with a suppressor, kept rows
  stop_after_us     builds with -DYL_NMS_PROBE_STOP=k return after phase k: median device time per launch of the kernel
                    (torch.profiler, CUDA activities); phase_us is the difference between consecutive stops.  A stop build
                    drops work whose results stay in registers, so such work is charged to the phase that first stores them
  overlap           three graph-replayed steps in flight on three streams (as bench.py runs them), one torch.profiler
                    trace: per back-end kernel the median duration of a launch and the median share of it during which a
                    k_flag_tma of another step is resident
  ab                with --ab LIB (repeatable): the kernel's median, one step alone and three steps in flight, for the default
                    library and each LIB, alternated --rounds times in this process

  python tools/nms_phase_probe.py --build-only        # compile the variants (no GPU needed)
  python tools/nms_phase_probe.py [--out FILE] [--ab LIB ...]
"""
import argparse
import json
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

from yolov4_b200 import build as yb_build  # noqa: E402

IMG, C, B = 608, 80, 64
GRIDS = [IMG // 8, IMG // 16, IMG // 32]
CONF, NMS = 1e-4, 0.4
KERNEL = "k_segment_nms_bins"
BACKEND = ["k_emit_flagged", "k_segment_nms_bins", "k_segment_nms_big", "k_gather_rows"]
PHASES = ["table zeroing + PDL wait", "record load", "rank sort", "bins + table inserts",
          "prefix/suffix OR scan", "candidate enumeration", "exact pair tests", "single-warp resolve", "row staging + store"]
COUNTS = {9: "ctas", 11: "queued_pairs", 12: "records", 13: "rows_with_suppressor", 14: "kept_rows"}
VDIR = os.path.join(yb_build.HERE, "variants")
VARIANTS = {"probe": ["-DYL_NMS_PROBE"]}
VARIANTS.update({"stop%d" % k: ["-DYL_NMS_PROBE_STOP=%d" % k] for k in range(len(PHASES) - 1)})


def variant_path(name):
    return os.path.join(VDIR, "libyolohead_nms_%s.so" % name)


def build_variants():
    """The default library, then every variant: yl_nms.cu with the variant's defines, linked with the default objects."""
    yb_build.build_lib()
    os.makedirs(VDIR, exist_ok=True)
    bdir = os.path.join(yb_build.HERE, "build")
    others = [os.path.join(bdir, os.path.basename(s)[:-3] + ".o") for s in yb_build.sources()
              if os.path.basename(s) != "yl_nms.cu"]
    src = os.path.join(yb_build.CSRC, "yl_nms.cu")

    def one(item):
        name, defs = item
        obj = os.path.join(VDIR, "yl_nms_%s.o" % name)
        subprocess.check_call([yb_build._nvcc()] + yb_build.NVCC_FLAGS + defs + ["-c", src, "-o", obj])
        subprocess.check_call([yb_build._nvcc(), "-shared", "-o", variant_path(name), obj] + others +
                              ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"])
        return name

    with ThreadPoolExecutor(max_workers=min(len(VARIANTS), os.cpu_count() or 1)) as ex:
        for name in ex.map(one, VARIANTS.items()):
            print("built", variant_path(name), flush=True)


def use_lib(path):
    """Point the binding at another build; HeadPostprocessors made afterwards call into it."""
    from yolov4_b200 import _cabi
    _cabi._lib = None
    if path is None:
        os.environ.pop("YL_LIB", None)
    else:
        os.environ["YL_LIB"] = path
    return _cabi.lib()


def kernel_medians(hp, raws, runs, names):
    import torch
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        hp.run(raws)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(runs):
            hp.run(raws)
        torch.cuda.synchronize()
    durs = {k: [] for k in names}
    for ev in prof.events():
        for k in names:
            if k in ev.name and str(ev.device_type).endswith("CUDA"):
                durs[k].append(ev.time_range.elapsed_us())
    return {k: float(np.median(v)) for k, v in durs.items() if v}


def overlap(hps):
    """Three graph-replayed steps in flight; per back-end kernel: median launch duration and median share of it next to a
    k_flag_tma of another step."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    streams = [torch.cuda.Stream() for _ in range(3)]
    main = torch.cuda.current_stream()

    def steps(k):
        for s in streams:
            s.wait_stream(main)
        for i in range(k):
            with torch.cuda.stream(streams[i % 3]):
                hps[i % 3].replay()
        for s in streams:
            main.wait_stream(s)
        torch.cuda.synchronize()

    steps(9)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        steps(60)
    evs = [(ev.name, ev.time_range.start, ev.time_range.end) for ev in prof.events() if str(ev.device_type).endswith("CUDA")]

    def short(name):
        for k in BACKEND + ["k_flag_tma"]:
            if k in name:
                return k
        return None

    evs = [(short(n), s, e) for n, s, e in evs if short(n)]
    flag = sorted((s, e) for n, s, e in evs if n == "k_flag_tma")
    out = {"k_flag_tma": {"launches": len(flag), "median_us": float(np.median([e - s for s, e in flag])) if flag else None}}
    for k in BACKEND:
        durs, shares = [], []
        for n, s, e in evs:
            if n != k or e <= s:
                continue
            # a step's own flag kernel ends before its back end starts, so any overlap is with another step's
            ov = sum(max(0.0, min(e, fe) - max(s, fs)) for fs, fe in flag)
            durs.append(e - s)
            shares.append(min(1.0, ov / (e - s)))
        if durs:
            out[k] = {"launches": len(durs), "median_us": float(np.median(durs)),
                      "median_share_next_to_flag": float(np.median(shares)), "mean_share_next_to_flag": float(np.mean(shares))}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--build-only", action="store_true")
    ap.add_argument("--runs", type=int, default=40, help="profiled HeadPostprocessor.run() calls per variant")
    ap.add_argument("--iters", type=int, default=300, help="replays per step timing of --ab")
    ap.add_argument("--rounds", type=int, default=3, help="alternations of --ab")
    ap.add_argument("--ab", action="append", default=[], metavar="LIB", help="another build of the library to compare with")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.build_only:
        build_variants()
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("nms_phase_probe.py measures on a GPU; there is none here")
    for name in VARIANTS:
        if not os.path.exists(variant_path(name)):
            raise SystemExit("%s is missing: run with --build-only first" % variant_path(name))
    from agnostic_probe import gpu_info, step3_time, time_events
    import yolov4_b200 as yb
    from yolov4_b200.synth import synth_head_outputs
    raws = synth_head_outputs(B, IMG, C, seed=0, device="cuda")
    res = {"probe": "nms_phase_probe", "workload": "B=%d @%d, %d classes, fp32 synth_head_outputs seed 0, conf %g / nms %g"
           % (B, IMG, C, CONF, NMS), "gpu": gpu_info()}

    def hp_for(path):
        use_lib(path)
        return yb.HeadPostprocessor(B, GRIDS, C, CONF, NMS)

    # phase cycles
    L = use_lib(variant_path("probe"))
    import ctypes
    L.yl_nms_probe_read.restype = ctypes.c_int
    L.yl_nms_probe_read.argtypes = [ctypes.c_void_p, ctypes.c_int]
    acc = (ctypes.c_ulonglong * 16)()
    hp = yb.HeadPostprocessor(B, GRIDS, C, CONF, NMS)
    for _ in range(3):
        hp.run(raws)
    torch.cuda.synchronize()
    assert L.yl_nms_probe_read(acc, 1) == 0
    for _ in range(args.runs):
        hp.run(raws)
    torch.cuda.synchronize()
    assert L.yl_nms_probe_read(acc, 1) == 0
    ctas = max(1, acc[9])
    tot = sum(acc[k] for k in range(len(PHASES)))
    res["phase_cycles"] = {PHASES[k]: {"cycles_per_cta": acc[k] / ctas, "share": acc[k] / max(1, tot)} for k in range(len(PHASES))}
    res["counts"] = {v: (acc[k] / args.runs if k == 9 else acc[k] / ctas) for k, v in COUNTS.items()}
    res["counts"]["ctas"] = acc[9] / args.runs
    res["probe_kernel_us"] = kernel_medians(hp, raws, args.runs, [KERNEL]).get(KERNEL)
    del hp

    # stop-after-phase variants and the full kernel
    stops = {}
    for k in range(len(PHASES) - 1):
        stops[PHASES[k]] = kernel_medians(hp_for(variant_path("stop%d" % k)), raws, args.runs, [KERNEL]).get(KERNEL)
    stops[PHASES[-1]] = kernel_medians(hp_for(None), raws, args.runs, [KERNEL]).get(KERNEL)
    res["stop_after_us"] = stops
    prev, res["phase_us"] = 0.0, {}
    for k in PHASES:
        res["phase_us"][k] = stops[k] - prev
        prev = stops[k]

    # overlap with the next steps' streaming pass (default library)
    use_lib(None)
    hps = [yb.HeadPostprocessor(B, GRIDS, C, CONF, NMS).capture(raws) for _ in range(3)]
    res["overlap"] = overlap(hps)
    del hps

    if args.ab:
        libs = [None] + [os.path.abspath(p) for p in args.ab]
        rows = {("default" if p is None else p): [] for p in libs}
        for _ in range(args.rounds):
            for p in libs:
                hps = [hp_for(p).capture(raws) for _ in range(3)]
                t1 = time_events(lambda: hps[0].replay(), args.iters)
                t3 = step3_time(hps, args.iters)
                km = kernel_medians(hp_for(p), raws, args.runs, BACKEND)
                rows["default" if p is None else p].append({"kernels_us": km, "step_alone_us": 1e6 * t1,
                                                           "step_3_in_flight_us": 1e6 * t3})
                del hps
                torch.cuda.empty_cache()
        res["ab"] = rows
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
