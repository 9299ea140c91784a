"""Measures the fused detection path on fp32, fp16 and bf16 head tensors and prints one JSON line.

Workload: B=64 @608, 80 classes, the seeded mixture of synth_head_outputs (seed 0), at conf 1e-4 / nms 0.4 and at conf 0.2 / nms 0.5
(the sparse, objectness-first mode of the flag kernel).  The 16-bit inputs are the fp32 ones rounded to the 16-bit type; every
16-bit result is checked bit for bit against the fp32 path on the widened inputs in the same run, and the script exits non-zero
on a difference.

For each dtype:
  flag_pass   the streaming flag kernel alone (stage 1 of yl_filter_raw_typed, counters reset inside it), CUDA events over many
              launches; GB/s on the algorithmic bytes B*M*85*esize, as a fraction of the measured copy bandwidth of the B200
              (6547.8 GB/s, DESIGN section 5.1) and of the data-sheet HBM3e bandwidth (7.7 TB/s).  fp32 runs the kernel the step
              runs: k_flag_tma at conf 1e-4, k_flag_raw in the sparse mode; the fp32 k_flag_raw is timed as well (YL_FLAG=ldg in a
              fresh process) because the 16-bit inputs always take that kernel
  emit_pass   the emit kernel alone (stages 2|4: a counter memset and k_emit_flagged on the tables of the last flag pass)
  step        the whole chain as a HeadPostprocessor graph replay: one step alone, and three steps in flight on three streams
  host_leg    yl_detect_host from pinned host buffers of the dtype (H2D copies, kernels, D2H of the rows), images/s
The inputs (495 MB fp32, 247 MB 16-bit) exceed the 126 MB L2, so the streaming passes read from HBM.

  python tools/half_probe.py [--out FILE]
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

B, IMG, C = 64, 608, 80
GRIDS = [IMG // 8, IMG // 16, IMG // 32]
M = sum(3 * f * f for f in GRIDS)
COPY_PEAK_GBS = 6547.8          # measured copy bandwidth, B200 (DESIGN section 5.1)
DATASHEET_GBS = 7700.0          # HBM3e, NVIDIA data sheet, one B200
DTYPES = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}
CODES = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}
SETTINGS = [(1e-4, 0.4), (0.2, 0.5)]


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
        x, y = x.cpu().numpy(), y.cpu().numpy()
        if x.shape != y.shape:
            return False
        nx, ny = np.isnan(x), np.isnan(y)
        if not (np.array_equal(nx, ny) and np.array_equal(x.view(np.uint32)[~nx], y.view(np.uint32)[~ny])):
            return False
    return True


def flag_only_fp32_ldg(conf, nms, iters):
    """The fp32 k_flag_raw alone, in a fresh process (the flag kernel is chosen at library load time)."""
    code = ("import sys; sys.path.insert(0, %r); import tools.half_probe as h; print(h._flag_time_here(%r, %r, %d))"
            % (ROOT, conf, nms, iters))
    env = dict(os.environ, YL_FLAG="ldg")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=900)
    if out.returncode != 0:
        raise SystemExit("fp32 k_flag_raw probe failed:\n" + out.stderr[-3000:])
    return float(out.stdout.strip().splitlines()[-1])


def _flag_time_here(conf, nms, iters):
    import yolov4_b200 as yb
    from yolov4_b200.synth import synth_head_outputs
    raws = synth_head_outputs(B, IMG, C, seed=0, device="cuda")
    hp = yb.HeadPostprocessor(B, GRIDS, C, conf, nms)
    return time_events(lambda: _stage(hp, raws, 0, 5), iters)


def _stage(hp, raws, code, stages):
    from yolov4_b200 import _cabi
    rp = _cabi.ptrs([r.data_ptr() for r in raws])
    _cabi.check(hp.L.yl_filter_raw_typed(rp, code, hp.fs, 3, hp.B, hp.C, hp.anch, hp.mask, hp.conf, hp.ws.ptr(), hp.ws.nbytes,
                                         hp.M, hp.cap_seg, 0, hp.B, stages, torch.cuda.current_stream().cuda_stream))


def host_leg(yb, _cabi, raws, conf, nms, steps):
    L = _cabi.lib()
    code = CODES[raws[0].dtype]
    host = [r.cpu().pin_memory() for r in raws]
    cap_out = 16384
    ctx = ctypes.c_void_p()
    anch = _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh])
    mask = _cabi.ints([v for m in yb.ANCHOR_MASK for v in m])
    _cabi.check(L.yl_context_create_typed(ctypes.byref(ctx), torch.cuda.current_device(), B, _cabi.ints(GRIDS), 3, C, code, anch,
                                          mask, 1024, cap_out))
    try:
        rows = torch.empty((B, cap_out, 7), dtype=torch.float32).pin_memory()
        cnt = torch.zeros((B,), dtype=torch.int32).pin_memory()
        ptrs = _cabi.ptrs([h.data_ptr() for h in host])
        f32 = lambda v: float(np.float32(v))  # noqa: E731
        for _ in range(3):
            _cabi.check(L.yl_detect_host(ctx, ptrs, f32(conf), f32(nms), rows.data_ptr(), cnt.data_ptr()))
        t0 = time.perf_counter()
        for _ in range(steps):
            _cabi.check(L.yl_detect_host(ctx, ptrs, f32(conf), f32(nms), rows.data_ptr(), cnt.data_ptr()))
        torch.cuda.synchronize()
        sec = (time.perf_counter() - t0) / steps
        res = [rows[b, :int(cnt[b])].clone() if int(cnt[b]) else None for b in range(B)]
    finally:
        _cabi.check(L.yl_context_destroy(ctx))
    h2d = sum(h.numel() * h.element_size() for h in host)
    return {"images_per_s": B / sec, "ms_per_call": 1e3 * sec, "h2d_bytes_per_call": h2d, "h2d_gbs": h2d / sec / 1e9}, res


def measure_setting(yb, _cabi, conf, nms, args):
    from yolov4_b200.synth import synth_head_outputs
    base = synth_head_outputs(B, IMG, C, seed=0, device="cuda")
    out = {"conf": conf, "nms": nms, "per_dtype": {}}
    want = {}
    hps = {}
    inputs = {}
    for name, dt in DTYPES.items():
        raws = [r.to(dt) for r in base]
        inputs[name] = raws
        hps[name] = [yb.HeadPostprocessor(B, GRIDS, C, conf, nms).capture(raws) for _ in range(3)]
    # flag and emit passes: dtypes alternated over several rounds, median per dtype
    flag_t = {n: [] for n in DTYPES}
    emit_t = {n: [] for n in DTYPES}
    for _ in range(args.rounds):
        for name, dt in DTYPES.items():
            hp, raws = hps[name][0], hps[name][0]._captured_inputs
            flag_t[name].append(time_events(lambda: _stage(hp, raws, CODES[dt], 5), args.iters))
            _stage(hp, raws, CODES[dt], 5)
            emit_t[name].append(time_events(lambda: _stage(hp, raws, CODES[dt], 6), args.iters))
    for name, dt in DTYPES.items():
        esize = torch.tensor([], dtype=dt).element_size()
        nbytes = B * M * (5 + C) * esize
        tf = float(np.median(flag_t[name]))
        te = float(np.median(emit_t[name]))
        gbs = nbytes / tf / 1e9
        hp3 = hps[name]
        # the chain alone, then three steps in flight on three streams (as bench.py runs it)
        t_step = time_events(lambda: hp3[0].replay(), args.iters)
        streams = [torch.cuda.Stream() for _ in range(3)]
        state = {"i": 0}

        def step3():
            p = state["i"] % 3
            with torch.cuda.stream(streams[p]):
                hp3[p].replay()
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
        for _ in range(args.iters):
            step3()
        for s in streams:
            main.wait_stream(s)
        e1.record()
        torch.cuda.synchronize()
        t_step3 = e0.elapsed_time(e1) / 1e3 / args.iters
        got = hp3[0].results()
        host, host_rows = host_leg(yb, _cabi, inputs[name], conf, nms, args.host_steps)
        entry = {
            "flag_pass": {"us": 1e6 * tf, "algorithmic_bytes": nbytes, "gbs": gbs,
                          "fraction_of_measured_copy_peak_6547.8_gbs": gbs / COPY_PEAK_GBS,
                          "fraction_of_datasheet_7.7_tbs": gbs / DATASHEET_GBS,
                          "kernel": "k_flag_raw" if (name != "fp32" or conf >= 0.02) else "k_flag_tma",
                          "rounds_us": [1e6 * t for t in flag_t[name]]},
            "emit_pass_us": 1e6 * te,
            "step_alone_us": 1e6 * t_step,
            "step_3_in_flight_us": 1e6 * t_step3,
            "step_3_in_flight_images_per_s": B / t_step3,
            "host_leg": host,
            "detections": sum(0 if g is None else g.shape[0] for g in got),
        }
        if name == "fp32":
            want["graph"] = got
            want["host"] = host_rows
        else:
            wide = yb.detect_raw([r.float() for r in inputs[name]], C, conf, nms)
            entry["parity_vs_widened_fp32"] = bool(rows_equal(got, wide) and rows_equal(host_rows, wide))
        out["per_dtype"][name] = entry
    fp32_ldg = flag_only_fp32_ldg(conf, nms, args.iters) if not args.no_subprocess else None
    if fp32_ldg is not None:
        out["fp32_k_flag_raw_us"] = 1e6 * fp32_ldg
        out["fp32_k_flag_raw_gbs"] = B * M * (5 + C) * 4 / fp32_ldg / 1e9
    out["fp32_host_rows_equal_graph_rows"] = bool(rows_equal(want["host"], want["graph"]))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--host-steps", type=int, default=10)
    ap.add_argument("--no-subprocess", action="store_true", help="skip the fp32 k_flag_raw timing in a fresh process")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("half_probe.py measures on a GPU; there is none here")
    import yolov4_b200 as yb
    from yolov4_b200 import _cabi
    res = {"probe": "half_probe", "workload": "B=%d @%d, %d classes, synth_head_outputs seed 0" % (B, IMG, C),
           "gpu": gpu_info(), "l2_note": "inputs of 495 MB (fp32) / 247 MB (16-bit) exceed the 126 MB L2: the streaming passes read HBM",
           "settings": [measure_setting(yb, _cabi, conf, nms, args) for conf, nms in SETTINGS]}
    ok = all(e.get("parity_vs_widened_fp32", True) for s in res["settings"] for e in s["per_dtype"].values()) and \
        all(s["fp32_host_rows_equal_graph_rows"] for s in res["settings"])
    res["parity_ok"] = ok
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if not ok:
        raise SystemExit("parity check failed: a 16-bit result differs from the fp32 path on the widened inputs")


if __name__ == "__main__":
    main()
