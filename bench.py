#!/usr/bin/env python
"""bench.py -- images/sec of the detection-head hot path (fused decode + conf filter + per-class NMS).

Workload (BASELINE.json configs[1]): synthetic head outputs, batch 64 per GPU @608x608 (grids 76/38/19), 80 classes,
val setting conf 1e-4 / nms 0.4.  A "step" is one pass of the hot path over one batch.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]
                                                                  our arm (N>1 under torchrun, one rank per GPU); DIR receives
                                                                  the detections of the last timed step as .npy files
  python bench.py --impl reference [--gpus N] --steps K ...       CPU arm on the host cores (rank 0 only): the UNMODIFIED
                                                                  reference from baseline/_ref when it is installed, else the
                                                                  oracle's C port of it
Prints ONE JSON line (rank 0).  See DESIGN.md section 7 for what each field measures.
"""
import argparse
import ctypes
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
REF_DIR = os.path.join(ROOT, "baseline", "_ref")

IMG, C, CONF, NMS = 608, 80, 1e-4, 0.4
GRIDS = [76, 38, 19]
BYTES_PER_IMAGE = sum(3 * f * f for f in GRIDS) * (5 + C) * 4          # 7 732 620 B (SURVEY.md 8(d))
TARGET_BYTES_PER_IMAGE = 15647184 + 363888 + 1200                        # build_target: dense writes + pred + labels (SURVEY 8(d))
METRIC = "images/sec decode+NMS @608 b64 conf1e-4"
UNIT = "images/s"
# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel at B=64, from the ncu --set full captures
# under profiles/ (per front-end form; the live frac_physical below divides these by the launch time measured in this run)
TRAFFIC_PER_LAUNCH = {"k_flag_raw": 475289856 + 9423360,                # profiles/r2_k_flag_raw_ncu_full_details.txt
                      "k_flag_tma": 472751104 + 4560896}                # profiles/r2_k_flag_tma_ncu_full_details.txt
WORKLOAD = "yolov4 head outputs batch %d/GPU @608x608 (grids 76/38/19), 80 classes, conf 1e-4, nms 0.4 (BASELINE configs[1])"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "50"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def cpu_port(sample_images, threads, seed=0, min_seconds=0.0, raws=None):
    """Oracle port of the reference CPU path (decode x3 + cat + postprocess) on `sample_images` images of the workload (`raws`:
    the very arrays another arm processed; else generated from `seed`).
    Returns (images/s, seconds, list of per-image rows of the last pass, passes)."""
    from oracle import oracle as orc
    from yolov4_b200.synth import synth_head_outputs
    if raws is None:
        raws = [r.numpy() for r in synth_head_outputs(sample_images, IMG, C, seed=seed)]
    else:
        raws = [np.ascontiguousarray(r[:sample_images]) for r in raws]
    orc.detect([r[:1] for r in raws], C, CONF, NMS, nthreads=1)          # warm-up (page in, build lib)
    passes, dt = 0, 0.0
    while passes == 0 or (dt < min_seconds and passes < 1000):           # bounded sample: repeat the same images
        t0 = time.perf_counter()
        out = orc.detect(raws, C, CONF, NMS, nthreads=threads)
        dt += time.perf_counter() - t0
        passes += 1
    return sample_images * passes / dt, dt, out, passes


class RealReference:
    """The UNMODIFIED reference (baseline/_ref, installed by tools/install_reference.sh): YOLOLayer x3 (eval) + torch.cat +
    postprocess, on CPU tensors, exactly the calls of yolo/model/yolov4.py:314-324 and yolo/engine/build.py:137."""

    @staticmethod
    def available():
        return os.path.isdir(os.path.join(REF_DIR, "yolo"))

    def __init__(self):
        import torch
        sys.path.insert(0, REF_DIR)
        from yolo.model.yololayer import YOLOLayer
        from yolo.util.utils import postprocess
        import yolov4_b200 as yb
        cfg = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": C}
        self.torch = torch
        self.layers = [YOLOLayer(cfg, l, device="cpu").eval() for l in range(3)]
        self.post = postprocess

    def run(self, raws):
        torch = self.torch
        with torch.no_grad(), np.errstate(all="ignore"):
            dense = torch.cat([self.layers[l](raws[l].clone()) for l in range(3)], 1)
            return self.post(dense, C, CONF, NMS)


_JSON_FD = None


def claim_stdout():
    """stdout must carry exactly one JSON line: from here on everything written to file descriptor 1 (NCCL's version banner,
    library chatter of any rank) lands on stderr, and emit() writes the line to the real stdout."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def run_reference(args, rank, world):
    """CPU arm.  Each step is a bounded sample of the workload (images are independent, utils.py:133), sized so that the whole
    --steps K --warmup W run stays within about two minutes."""
    if rank != 0:
        return
    import torch
    from yolov4_b200.synth import synth_head_outputs
    threads = os.cpu_count() or 1
    port_v, _, _, _ = cpu_port(16, threads)                              # the C port as a second figure (one pass of 16 images)
    total_steps = args.steps + args.warmup
    if RealReference.available():
        ref = RealReference()
        torch.set_num_threads(threads)
        raws_all = synth_head_outputs(8, IMG, C, seed=0)
        t0 = time.perf_counter()
        ref.run([r[:1] for r in raws_all])                               # also the warm-up of the Python path
        t1 = time.perf_counter() - t0
        n_img = int(max(1, min(8, 110.0 / (max(total_steps, 1) * t1))))
        raws = [r[:n_img] for r in raws_all]
        for _ in range(args.warmup):
            ref.run(raws)
        t_all, rows = 0.0, 0
        for _ in range(args.steps):
            t0 = time.perf_counter()
            out = ref.run(raws)
            t_all += time.perf_counter() - t0
            rows = sum(0 if o is None else len(o) for o in out)
        kind = "reference"
        sample = ("%d images/step of the same synthetic workload (seed 0), the unmodified reference from baseline/_ref: YOLOLayer x3 "
                  "(eval) + torch.cat + postprocess on CPU tensors; torch on %d threads, its NumPy NMS loop is single-threaded; "
                  "%d rows/step" % (n_img, threads, rows))
    else:
        n_img = max(threads, 16)
        for _ in range(args.warmup):
            cpu_port(min(n_img, 8), threads)
        t_all = 0.0
        for s in range(args.steps):
            _, dt, out, _ = cpu_port(n_img, threads, seed=s)
            t_all += dt
        kind = "port"
        sample = "%d images/step of the same synthetic workload, oracle C port of YOLOLayer x3 + cat + postprocess, OpenMP over " \
                 "images (baseline/_ref is not installed)" % n_img
    value = n_img * args.steps / t_all
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_all / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD % 64, "sample_images_per_step": n_img},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "cpu_baseline_port": {"value": port_v, "unit": UNIT, "cores": threads, "kind": "port",
                              "sample": "16 images, one pass, oracle C port (OpenMP over images)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def rows_equal(got, want):
    """Bitwise equality of two lists of per-image [K,7] arrays / None."""
    if len(got) != len(want):
        return False
    for g, w in zip(got, want):
        if (g is None) != (w is None):
            return False
        if w is None:
            continue
        g = g.detach().cpu().numpy() if hasattr(g, "detach") else np.asarray(g)
        w = w.detach().cpu().numpy() if hasattr(w, "detach") else np.asarray(w)
        if g.shape != w.shape or not np.array_equal(np.ascontiguousarray(g).view(np.uint32), np.ascontiguousarray(w).view(np.uint32)):
            return False
    return True


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, per_image):
    """Writes what a caller of the timed path receives for one step, the per-image lists of [K_i, 7] rows, as
    counts.npy (float64 [n_images], rows per image) and detections.npy (float32 [R, 7], the rows of every image in image order).
    Above 64 MB in all, detections.npy keeps a fixed, seeded sample of the rows and detections_index.npy (float64 [n]) gives
    their positions in the full [R, 7] array."""
    os.makedirs(out_dir, exist_ok=True)
    counts = np.array([0 if r is None else r.shape[0] for r in per_image], np.float64)
    rows = [r.detach().cpu().numpy() if hasattr(r, "detach") else np.asarray(r) for r in per_image if r is not None]
    rows = np.concatenate(rows, 0).astype(np.float32) if rows else np.zeros((0, 7), np.float32)
    np.save(os.path.join(out_dir, "counts.npy"), counts)
    cap = (DUMP_BYTES - counts.nbytes - 3 * 4096) // (rows.itemsize * 7 + 8)     # 4 KB per file for the .npy headers
    idx_path = os.path.join(out_dir, "detections_index.npy")
    if rows.shape[0] > cap:
        idx = np.sort(np.random.default_rng(0).choice(rows.shape[0], cap, replace=False))
        np.save(idx_path, idx.astype(np.float64))
        rows = rows[idx]
    elif os.path.exists(idx_path):
        os.remove(idx_path)
    np.save(os.path.join(out_dir, "detections.npy"), rows)


def time_events(torch, fn, iters, warm=3):
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


def extras(torch, yb, dev, peak):
    """Driver-visible numbers for the other BASELINE configs and row families (B200, this run, CUDA events)."""
    from yolov4_b200.synth import synth_head_outputs, synth_labels
    cfg = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": C}
    out = {}
    # config 3: detect setting, batch 256
    B3 = 256
    raws3 = synth_head_outputs(B3, IMG, C, seed=1, device=dev)
    hp3 = yb.HeadPostprocessor(B3, GRIDS, C, 0.2, 0.5, device=dev).capture(raws3)
    rows3 = sum(0 if r is None else r.shape[0] for r in hp3.results())
    t = time_events(torch, hp3.replay, 30)
    out["config3_detect_b256_conf0.2_nms0.5"] = {"us_per_step": t * 1e6, "images_per_s": B3 / t, "rows_per_step": rows3,
                                                   "hbm_frac_on_all_planes": B3 * BYTES_PER_IMAGE / t / 1e9 / peak,
                                                   "note": "sparse objectness-first mode: the class planes of dead vectors are never read"}
    del hp3, raws3
    torch.cuda.empty_cache()
    # config 4 and the contract-literal path at B=64
    B = 64
    raws = synth_head_outputs(B, IMG, C, seed=0, device=dev)
    labels = synth_labels(B, IMG, n_valid=50, seed=2, device=dev)
    crit = yb.YOLOLoss(cfg, 0.7, device=dev)
    train_layers = [yb.YOLOLayer(cfg, l, device=dev).train() for l in range(3)]
    with torch.no_grad():
        outs = [train_layers[l](raws[l]) for l in range(3)]

    def bt():
        for l in range(3):
            crit.build_target(outs[l]["output"], outs[l]["pred"], l, labels)

    def bt3():
        yb.build_targets3([o["output"] for o in outs], [o["pred"] for o in outs], [0, 1, 2], labels, yb.ANCHORS_PX, yb.ANCHOR_MASK,
                          0.7, C)
    t = time_events(torch, bt, 10)
    t3 = time_events(torch, bt3, 10)
    out["config4_build_target_b64_50gt"] = {"us_per_step": t3 * 1e6, "images_per_s": B / t3,
                                            "write_roofline_frac": B * TARGET_BYTES_PER_IMAGE / t3 / 1e9 / peak,
                                            "bytes_per_image": TARGET_BYTES_PER_IMAGE,
                                            "form": "yl_build_target3: one launch pair for the three scales (YOLOLoss.forward)",
                                            "three_per_layer_calls_us": t * 1e6,
                                            "note": "includes the allocation of the four dense output tensors per scale (torch.empty)"}

    def dec_train():
        with torch.no_grad():
            for l in range(3):
                train_layers[l](raws[l])
    t = time_events(torch, dec_train, 10)
    out["yololayer_train_decode_b64"] = {"us_per_step": t * 1e6, "hbm_frac": (2 * B * BYTES_PER_IMAGE + B * 363888) / t / 1e9 / peak}
    del outs
    eval_layers = [yb.YOLOLayer(cfg, l, device=dev).eval() for l in range(3)]
    dense = yb.decode_dense_cat(raws, cfg)
    t_dec = time_events(torch, lambda: yb.decode_dense_cat(raws, cfg), 10)
    t_lit = time_events(torch, lambda: torch.cat([eval_layers[l](raws[l]) for l in range(3)], 1), 10)
    t_post = time_events(torch, lambda: yb.postprocess(dense, C, CONF, NMS), 10)
    out["contract_literal_b64"] = {
        "decode_dense_us": t_dec * 1e6, "decode_hbm_frac": 2 * B * BYTES_PER_IMAGE / t_dec / 1e9 / peak,
        "yololayer_x3_plus_cat_us": t_lit * 1e6,
        "postprocess_dense_us": t_post * 1e6,
        "note": "YOLOLayer.forward x3 into the cat buffer, then postprocess(prediction, ...) incl. its one D2H of counts and the "
                "Python list; the fused path above never materialises the 495 MB decoded tensor"}
    del dense
    # N2: fused loss forward + backward
    raws_g = [r.clone().requires_grad_(True) for r in raws]

    def fwd():
        return yb.fused_yolo_loss(raws_g, labels, cfg, 0.7)
    t_f = time_events(torch, fwd, 10)

    def fb():
        for r in raws_g:
            r.grad = None
        fwd().backward()
    t_fb = time_events(torch, fb, 10)
    out["n2_fused_loss_b64_50gt"] = {"forward_us": t_f * 1e6, "forward_backward_us": t_fb * 1e6}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="images per GPU per step")
    ap.add_argument("--groups", type=int, default=1, help="image groups pipelined over two streams")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--cpu-sample", type=int, default=64, help="images timed for the CPU baseline (0 = skip)")
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="repeat the CPU sample until this much time is spent")
    ap.add_argument("--min-seconds", type=float, default=0.25, help="the warm-up continues until this much device time is covered, "
                                                                    "so that the K timed steps run at sustained clocks")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the detections of the last timed step to DIR as .npy "
                                                                        "files (see dump_outputs)")
    ap.add_argument("--no-extras", action="store_true", help="skip the other configs' numbers")
    ap.add_argument("--inflight", type=int, default=0, help="0 = automatic (3 on one GPU, 2 with the exchange at N>1).  ""steps in flight: each step's chain is a CUDA graph; step i runs on stream "
                                                            "i %% inflight with its own workspace and output rows, so the latency-bound "
                                                            "kernels of a step run under the streaming pass of the next ones (1 = serial)")
    args = ap.parse_args()
    claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)
    if world > 1:
        # With the exchange in the step the register-staged flag kernel measured best (it uses no shared memory, the bulk-copy push
        # of the exchange lives in it): 8 GPUs 268 us per step against 300-356 us with the TMA flag kernel (profiles/r2_summary.md).
        # Read once when the library loads, so set before anything touches it.
        os.environ.setdefault("YL_FLAG", "ldg")

    import torch
    import torch.distributed as dist
    import yolov4_b200 as yb
    from yolov4_b200 import _cabi
    from yolov4_b200.synth import synth_head_outputs

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch
    sampler = ClockSampler(local_rank) if rank == 0 else None   # nvidia-smi needs ~0.3 s before its first sample
    raws = synth_head_outputs(B, IMG, C, seed=rank, device=dev)
    # NP postprocessors (own workspace, output rows and CUDA graph each, the same read-only inputs), one per step in flight
    NP = max(1, min(int(args.inflight), 8)) if args.inflight > 0 else (3 if world == 1 else 2)
    if world > 1:
        NP = max(NP, 2)                                  # the exchange of step i reads rows[i % NP] while step i+1 runs
    hps = [yb.HeadPostprocessor(B, GRIDS, C, CONF, NMS, device=dev, n_groups=args.groups).capture(raws) for _ in range(NP)]
    if world == 1:
        cstreams = [torch.cuda.Stream(device=dev) for _ in range(NP)]
    else:
        # with the exchange in the step the chains run one after the other on ONE stream (two output buffers alternate, the
        # exchange of step i runs under the chain of step i+1 on the side stream): concurrent chains measured slower there
        # (8 GPUs: 342 us per step against 268)
        cstreams = [torch.cuda.Stream(device=dev)] * NP
    hp = hps[0]
    res = hp.results()                                   # validates capacities; also the first parity-visible output
    rows_per_step = sum(0 if r is None else r.shape[0] for r in res)

    ex = None
    pipe = None
    if world > 1:
        from yolov4_b200.sharded import DetectionExchange
        ex = DetectionExchange(B, hp.cap_out, dev, slots=NP)
        side = torch.cuda.Stream(device=dev, priority=int(os.environ.get("YL_XCHG_PRIO", "0")))
        ev_done = [torch.cuda.Event() for _ in range(NP)]
        ev_pushed = [torch.cuda.Event() for _ in range(NP)]
        for e in ev_pushed:
            e.record()
        # (YL_BENCH_XGRAPH=1: the exchange of a slot -- push / wait / release -- as a CUDA graph of its own, one host call per step
        # instead of three kernel launches through ctypes; measured no faster, the eager launches are the default)
        xgraphs = []
        for p_ in range(NP if os.environ.get("YL_BENCH_XGRAPH") == "1" else 0):
            with torch.cuda.stream(side):
                ex.push(hps[p_].rows, hps[p_].meta, p_)          # eager once on every rank: consistent epochs, warm kernels
                ex.wait(p_)
                ex.release(p_)
            torch.cuda.synchronize()
            g_ = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g_, stream=side):
                ex.push(hps[p_].rows, hps[p_].meta, p_)
                ex.wait(p_)
                ex.release(p_)
            xgraphs.append(g_)
        pipe = True

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    state = {"i": 0}

    def step():
        """One step = the chain of one batch (a CUDA graph), on stream i % NP with postprocessor i % NP: NP steps are in flight, so the
        emit / NMS / gather kernels of a step run under the streaming pass of the following ones.  At N>1 the step's exchange (push
        the kept rows into every rank's window, wait for everybody's rows of that slot, release it) follows on the side stream,
        and the step that reuses rows[i % NP] waits for it."""
        p = state["i"] % NP
        cs = cstreams[p]
        if pipe is not None:
            cs.wait_event(ev_pushed[p])
        with torch.cuda.stream(cs):
            hps[p].replay()
            if pipe is not None:
                ev_done[p].record(cs)
        if pipe is not None:
            side.wait_event(ev_done[p])
            with torch.cuda.stream(side):
                if xgraphs:
                    xgraphs[p].replay()
                else:
                    ex.push(hps[p].rows, hps[p].meta, p)
                    ex.wait(p)
                    ex.release(p)
                ev_pushed[p].record(side)
        state["i"] += 1

    def begin():
        """The streams of the pipeline start behind everything enqueued on the current stream (the start event of a timed round)."""
        cur = torch.cuda.current_stream(dev)
        for cs in cstreams:
            cs.wait_stream(cur)

    def drain():
        """The timed region ends when every step in flight has finished and (N>1) its exchange has been delivered everywhere."""
        cur = torch.cuda.current_stream(dev)
        for cs in cstreams:
            cur.wait_stream(cs)
        if pipe is not None:
            cur.wait_stream(side)
            return (state["i"] - 1) % NP
        return None

    def warm(n):
        begin()
        for _ in range(n):
            step()
        drain()
        barrier()

    # clocks are sampled from here through the timed steps and the per-kernel timing below
    warm(args.warmup)
    # K timed steps are a few milliseconds: the warm-up goes on until min_seconds of device time are covered, so that they run at
    # the clocks of sustained load.  The ranks agree on the count (at N>1 every step is matched by the exchange).
    n_sustain = 0
    if args.min_seconds > 0:
        t0 = time.perf_counter()
        warm(16)
        per_step = (time.perf_counter() - t0) / 16
        n_sustain = int(min(20000, math.ceil(args.min_seconds / max(per_step, 1e-7))))
        if world > 1:
            t = torch.tensor([n_sustain], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            n_sustain = int(t.item())
        warm(n_sustain)
        n_sustain += 16

    # ---- the timed region: exactly K steps ---------------------------------------------------------------------------------
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    state["i"] = 0
    barrier()
    ev0.record()
    begin()
    for _ in range(args.steps):
        step()
    last_slot = drain()
    ev1.record()
    barrier()
    sec = ev0.elapsed_time(ev1) / 1e3
    if world > 1:
        t = torch.tensor([sec], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec = float(t.item())
    value = world * B * args.steps / sec
    if args.dump_outputs and rank == 0:
        # what the caller of the timed path receives for the last step: this GPU's images, or at N>1 every rank's after the exchange
        dump_outputs(args.dump_outputs, ex.results(last_slot) if world > 1 else hps[(args.steps - 1) % NP].results())

    # ---- one step alone (serial replays of one graph): the latency of a step, next to the pipelined throughput above --------
    for _ in range(3):
        hp.replay()
    barrier()
    ev0.record()
    for _ in range(args.steps):
        hp.replay()
    ev1.record()
    barrier()
    sec_serial = ev0.elapsed_time(ev1) / 1e3

    # ---- multi-GPU: what the exchange costs, and that its result is right -------------------------------------------------
    xchg = None
    if world > 1:
        # the same K pipelined steps without the exchange: what the collective-free path does
        pipe_saved, pipe = pipe, None
        begin()
        for _ in range(NP):
            step()
        drain()
        barrier()
        ev0.record()
        begin()
        for _ in range(args.steps):
            step()
        drain()
        ev1.record()
        barrier()
        pipe = pipe_saved
        sec_nox = ev0.elapsed_time(ev1) / 1e3
        t = torch.tensor([sec_nox], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec_nox = float(t.item())
        rps = torch.tensor([rows_per_step], device=dev, dtype=torch.int64)
        dist.all_reduce(rps)
        rows_all_ranks = int(rps.item())
        bytes_in = (world - 1) * (rows_per_step * 28 + B * 4)                # what reaches this rank per step (every form)
        bytes_out = bytes_in if "multicast" not in ex.mode else rows_per_step * 28 + B * 4    # multicast: the switch replicates
        # parity: the gathered rows of two other ranks' shards, recomputed on this GPU from their seeds, bit for bit
        got = ex.results(last_slot)
        checked = []
        ok = True
        for r in sorted({(rank + 1) % world, (rank + world // 2) % world} - {rank}):
            want = yb.detect_raw(synth_head_outputs(B, IMG, C, seed=r, device=dev), C, CONF, NMS)
            ok = ok and rows_equal(got[r * B:(r + 1) * B], want)
            checked.append(r)
        ok = ok and rows_equal(got[rank * B:(rank + 1) * B], res)
        flag = torch.tensor([0 if ok else 1], device=dev)
        dist.all_reduce(flag)
        if int(flag.item()) != 0:
            raise SystemExit("exchange parity FAILED: gathered rows differ from the recomputed shards")
        xchg = {"kind": "%s (yl_xchg_push/wait/release), exchange of step i under the kernels of step i+1, counts stay on the "
                        "device" % ex.mode,
                "value_without_exchange": world * B * args.steps / sec_nox, "ms_per_step_without_exchange": 1e3 * sec_nox / args.steps,
                "nvlink_bytes_out_per_rank_per_step": bytes_out, "nvlink_bytes_in_per_rank_per_step": bytes_in,
                "rows_per_step_all_ranks": rows_all_ranks,
                "nvlink_out_gbs_per_rank": bytes_out / (sec / args.steps) / 1e9,
                "nvlink_in_gbs_per_rank": bytes_in / (sec / args.steps) / 1e9,
                "parity_checked_ranks_on_rank0": checked, "parity": "gathered rows == recomputed shards, bit-exact, on every rank",
                "status": ex.status()}

    # ---- BASELINE config 5 at N>1: batch 1024 sharded by image over the ranks, exchange included ---------------------------
    config5 = None
    if world > 1 and 1024 % world == 0 and not args.no_extras:
        B5 = 1024 // world
        raws5 = synth_head_outputs(B5, IMG, C, seed=100 + rank, device=dev)
        hps5 = [yb.HeadPostprocessor(B5, GRIDS, C, CONF, NMS, device=dev).capture(raws5) for _ in range(2)]
        rows5 = sum(0 if r is None else r.shape[0] for r in hps5[0].results())
        ex5 = DetectionExchange(B5, hps5[0].cap_out, dev, slots=2)
        evd = [torch.cuda.Event(), torch.cuda.Event()]
        evp = [torch.cuda.Event(), torch.cuda.Event()]
        for e in evp:
            e.record()

        def step5(i):
            s5 = i & 1
            main = torch.cuda.current_stream(dev)
            main.wait_event(evp[s5])
            hps5[s5].replay()
            evd[s5].record(main)
            side.wait_event(evd[s5])
            with torch.cuda.stream(side):
                ex5.push(hps5[s5].rows, hps5[s5].meta, s5)
                ex5.wait(s5)
                ex5.release(s5)
                evp[s5].record(side)

        n5 = max(4, min(args.steps, 20))
        for i in range(4):
            step5(i)
        torch.cuda.current_stream(dev).wait_stream(side)
        barrier()
        ev0.record()
        for i in range(n5):
            step5(i)
        torch.cuda.current_stream(dev).wait_stream(side)
        ev1.record()
        barrier()
        sec5 = ev0.elapsed_time(ev1) / 1e3
        t = torch.tensor([sec5], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec5 = float(t.item())
        got5 = ex5.results((n5 - 1) & 1)
        ok5 = rows_equal(got5[rank * B5:(rank + 1) * B5], hps5[0].results())
        flag = torch.tensor([0 if ok5 else 1], device=dev)
        dist.all_reduce(flag)
        if int(flag.item()) != 0:
            raise SystemExit("config 5: exchanged rows differ from the local rows")
        config5 = {"workload": "batch 1024 @608 conf 1e-4 nms 0.4 sharded by image: %d images per GPU, exchange of all detections included" % B5,
                   "images_per_s": 1024 * n5 / sec5, "ms_per_step": 1e3 * sec5 / n5, "steps": n5, "rows_per_step_this_rank": rows5,
                   "nvlink_in_gbs_per_rank": (world - 1) * rows5 * 28 / (sec5 / n5) / 1e9, "exchange": ex5.mode, "status": ex5.status()}
        ex5.close()
        del hps5, raws5
        torch.cuda.empty_cache()

    # ---- roofline: the dominant kernel alone, CUDA events on its stream ----------------------------------------------------
    L = _cabi.lib()
    st = torch.cuda.current_stream().cuda_stream
    rp = _cabi.ptrs([r.data_ptr() for r in hp._captured_inputs])
    front = os.environ.get("YL_FILTER", "split")
    flag_name = "k_flag_raw" if os.environ.get("YL_FLAG", "tma") == "ldg" else "k_flag_tma"

    def flag_kernel():
        # the streaming pass alone: k_flag_raw reads every raw byte it needs once (one launch covers the three scales)
        # (stages 1 | 4: the flag kernel alone, counters reset as in the step -- the persistent form draws its tiles from them)
        _cabi.check(L.yl_filter_raw_stage(rp, hp.fs, 3, B, C, hp.anch, hp.mask, hp.conf, hp.ws.ptr(), hp.ws.nbytes, hp.M,
                                          hp.cap_seg, 0, B, 5, st))

    n_f = max(20, min(args.steps, 200))
    t_filter = time_events(torch, flag_kernel, n_f, warm=args.warmup)
    clocks = sampler.stop() if sampler else None
    peak, peak_src = measured_peaks()
    achieved = B * BYTES_PER_IMAGE / t_filter / 1e9
    traffic = TRAFFIC_PER_LAUNCH.get(flag_name) if (front == "split" and B == 64) else None

    # ---- e2e: C-ABI host-buffer call, pinned host inputs, H2D + kernels + D2H inside the timed region ------------------
    e2e = None
    if args.e2e_steps > 0:
        host = [r.cpu().pin_memory() for r in raws]
        cap_out = hp.cap_out
        ctx = ctypes.c_void_p()
        _cabi.check(L.yl_context_create(ctypes.byref(ctx), local_rank, B, hp.fs, 3, C, hp.anch, hp.mask, hp.cap_seg, cap_out))
        out_rows = torch.empty((B, cap_out, 7), dtype=torch.float32).pin_memory()
        out_cnt = torch.zeros((B,), dtype=torch.int32).pin_memory()
        hptrs = _cabi.ptrs([h.data_ptr() for h in host])
        for _ in range(3):
            _cabi.check(L.yl_detect_host(ctx, hptrs, hp.conf, hp.nms, out_rows.data_ptr(), out_cnt.data_ptr()))
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            _cabi.check(L.yl_detect_host(ctx, hptrs, hp.conf, hp.nms, out_rows.data_ptr(), out_cnt.data_ptr()))
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        # the platform's ceiling for this leg, measured here: the same pinned buffers uploaded by plain copies, no kernel, all
        # ranks at once (at N>1 the ranks share the host's memory system and PCIe root complexes)
        dev_in = [torch.empty_like(r) for r in raws]
        for h, d in zip(host, dev_in):
            d.copy_(h, non_blocking=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(max(3, args.e2e_steps)):
            for h, d in zip(host, dev_in):
                d.copy_(h, non_blocking=True)
        torch.cuda.synchronize()
        dt_probe = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt_probe], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt_probe = float(t.item())
        h2d_probe_gbs = sum(h.numel() * 4 for h in host) * max(3, args.e2e_steps) / dt_probe / 1e9
        del dev_in
        host_rows = [out_rows[b, :int(out_cnt[b])] if int(out_cnt[b]) else None for b in range(B)]
        assert rows_equal(host_rows, res), "host path and device path disagree"
        h2d = int(sum(h.numel() * 4 for h in host))
        e2e = {"value": world * B * args.e2e_steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(rows_per_step * 28 + 3 * B * 4), "steps": args.e2e_steps,
               "bound": "host-to-device copies (PCIe): %.1f GB/s per rank of pinned uploads inside the timed region" % (h2d * args.e2e_steps / dt / 1e9),
               "h2d_gbs_per_rank": h2d * args.e2e_steps / dt / 1e9,
               "h2d_probe_gbs_per_rank": h2d_probe_gbs,
               "h2d_probe": "the same pinned buffers uploaded by bare copies (no kernels), all %d ranks at once, max over ranks: the "
                            "platform's ceiling for this leg; e2e reaches %.0f %% of it" % (world, 100 * (h2d * args.e2e_steps / dt / 1e9) / h2d_probe_gbs),
               "parity": "rows returned to the host == rows of the device path, bit-exact"}
        _cabi.check(L.yl_context_destroy(ctx))

    # ---- CPU baseline beside it (rank 0, N=1) + parity of the GPU arm against it on the SAME images -----------------------
    cpu = None
    parity = None
    extra = None
    if rank == 0 and world == 1 and args.cpu_sample > 0:
        threads = os.cpu_count() or 1
        # the oracle gets the very tensors the GPU arm processed (the CUDA generator's stream differs from the CPU generator's)
        n_cpu = min(args.cpu_sample, B)
        v, dt, want, passes = cpu_port(n_cpu, threads, min_seconds=args.cpu_seconds, raws=[r.cpu().numpy() for r in raws])
        cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": "the %d images of the GPU arm's batch x %d passes (%.1f s of CPU work on %d threads), oracle C port of "
                         "YOLOLayer x3 + cat + postprocess, OpenMP over images" % (n_cpu, passes, dt, threads)}
        n_chk = n_cpu
        if not rows_equal(res[:n_chk], want[:n_chk]):
            raise SystemExit("parity FAILED: the GPU arm's rows differ from the oracle's on the same images")
        parity = {"parity_checked_images": n_chk, "against": "oracle (C restatement of the reference, pinned to reference goldens)",
                  "result": "counts and row bytes identical", "rows": int(sum(0 if w is None else len(w) for w in want[:n_chk]))}
    if rank == 0 and world == 1 and not args.no_extras:
        for h in hps:
            del h
        torch.cuda.empty_cache()
        extra = extras(torch, yb, dev, peak)

    if rank == 0:
        step_s = sec / args.steps
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * step_s, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD % B,
                       "l2": "inputs (495 MB/step) are larger than L2 (126 MB); no flush needed",
                       "timed": "K steps, each the CUDA-graph replay of the whole chain of one batch (%s + k_emit_flagged + k_segment_nms_bins + "
                                "k_segment_nms_big + k_gather_rows), %d steps in flight on their own streams / workspaces / output rows; the "
                                "timed region ends when the last step has finished%s" % (
                                    flag_name, NP,
                                    "; at N>1 every step also pushes its kept rows into every rank's window (the final exchange) on a side "
                                    "stream, and the last exchange is delivered inside the timed region" if world > 1 else ""),
                       "steps_in_flight": NP, "one_step_alone_ms": 1e3 * sec_serial / args.steps,
                       "sustained_warmup_steps": n_sustain,
                       "rows_per_step": rows_per_step,
                       "parallelism": "images sharded by rank, no collective inside decode/filter/NMS; final exchange by peer stores"},
            "gpu_launches": (hp.launches_per_run + (3 if world > 1 else 0)) * args.steps,
            "e2e": e2e,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic,
                         "frac_physical": (traffic / t_filter / 1e9 / peak) if traffic else None,
                         "kernel": "%s<3> (streaming decode+filter pass over the raw head tensors, one launch per step), timed alone" % flag_name
                                   if front == "split" else "front end '%s' alone (stage 1 of yl_filter_raw_stage)" % front,
                         "us_per_launch": t_filter * 1e6, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": B * BYTES_PER_IMAGE,
                         "note": "frac = algorithmic bytes (all 85 planes, SURVEY 8(d)) / launch time / peak; frac_physical = the kernel's "
                                 "own DRAM traffic (ncu capture under profiles/; it skips the 4 box planes) / the same time / peak; the peak is "
                                 "the driver-measured COPY bandwidth (read + write), which a read-only stream can slightly exceed",
                         "whole_step_frac": (B * BYTES_PER_IMAGE / step_s / 1e9) / peak,
                         "whole_step_frac_one_step_alone": (B * BYTES_PER_IMAGE / (sec_serial / args.steps) / 1e9) / peak},
            "cpu_baseline": cpu,
            "parity": parity,
            "exchange": xchg,
            "extra": extra if extra is not None else ({"config5_b1024_sharded": config5} if config5 else None),
            "clocks": clocks,
        }
        emit(line)
    if world > 1:
        ex.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
