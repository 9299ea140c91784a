"""Measures the fused training loss with iou_loss in {None, giou, diou, ciou} and prints one JSON line.

Workload: B=64 @608, 80 classes, synth_head_outputs (seed 0) with synth_labels (50 GTs per image, seed 1), fp32 and fp16 heads.
For each (dtype, iou_loss):
  forward_graph_us   fused_yolo_loss_components over the three scales (the PDL chain) captured once as a CUDA graph and
                     replayed, CUDA events over many replays
  fwd_bwd_us         fused_yolo_loss + backward (three gradient tensors in the heads' dtype), eager, CUDA events
  k_loss_match_us    median device time of the k_loss_match launches (one per scale) under torch.profiler, in a run of its own
  parity_ok          box component and box gradient of the first two images against tests/iou_loss_spec.py (the bound of
                     DESIGN.md section 1); None runs against the oracle's loss within 1e-5
The card's name and power limit are read in the same run.

  python tools/iou_loss_probe.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

B, IMG, C = 64, 608, 80
KINDS = [None, "giou", "diou", "ciou"]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        name, power = [x.strip() for x in out[torch.cuda.current_device()].split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:  # the reading is informative; the measurement does not depend on it
        return {"name": torch.cuda.get_device_name(), "power_limit": "unknown (%s)" % type(e).__name__}


def time_events(fn, iters, warm=10):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters


def match_kernel_us(fn, iters):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    times = [e.device_time for e in prof.events() if "k_loss_match" in e.name and e.device_time > 0]
    return float(np.median(times)) if times else None


def parity(heads, lab, cfg, kind):
    import iou_loss_spec as spec
    from oracle import oracle as orc
    from yolov4_b200.yololoss import fused_yolo_loss, fused_yolo_loss_components
    h2 = [h[:2].float().contiguous() for h in heads]
    l2 = lab[:2].contiguous()
    raws = [h.cpu().numpy() for h in h2]
    labels = l2.cpu().numpy()
    got = fused_yolo_loss_components(h2, l2, cfg, iou_loss=kind).cpu().numpy()
    if kind is None:
        want = sum(orc.yolo_loss_layer(raws[l], labels, l, C, 0.7)[0] for l in range(3))
        return bool(np.allclose(got, want, rtol=1e-5, atol=1e-6))
    hs = [h.clone().requires_grad_(True) for h in h2]
    fused_yolo_loss(hs, l2, cfg, iou_loss=kind).backward()
    ok, box = True, 0.0
    for l in range(3):
        comps, _, (cells, _, graw, _) = spec.layer_spec(raws[l], labels, l, C, 0.7, kind)
        box += comps[0]
        g = hs[l].grad.cpu().numpy()
        for (b, a, j, i), gr in zip(cells, graw):
            ok &= bool(spec.within_bound(g[b, a * (5 + C):a * (5 + C) + 4, j, i], gr).all())
    return bool(ok and abs(got[0] - box) <= 1e-5 * abs(box) and got[1] == 0.0)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--iters", type=int, default=500)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("iou_loss_probe.py measures on a GPU; there is none here")
    import yolov4_b200 as yb
    from yolov4_b200.synth import synth_head_outputs, synth_labels
    from yolov4_b200.yololoss import fused_yolo_loss, fused_yolo_loss_components
    cfg = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": C}
    heads32 = synth_head_outputs(B, IMG, C, seed=0, device="cuda", fg_prob=0.02, clustered=True)
    lab = synth_labels(B, IMG, n_valid=50, seed=1, device="cuda")
    res = {"probe": "iou_loss_probe", "workload": "B=%d @%d, %d classes, 50 GTs per image" % (B, IMG, C), "gpu": gpu_info(),
           "runs": []}
    for dt in (torch.float32, torch.float16):
        heads = [h.to(dt).contiguous() for h in heads32]
        for kind in KINDS:
            fwd = lambda: fused_yolo_loss_components(heads, lab, cfg, iou_loss=kind)   # noqa: E731
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                fwd()
            torch.cuda.current_stream().wait_stream(s)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                fwd()
            hs = [h.detach().clone().requires_grad_(True) for h in heads]

            def fwd_bwd():
                fused_yolo_loss(hs, lab, cfg, iou_loss=kind).backward()

            res["runs"].append({
                "dtype": str(dt).replace("torch.", ""), "iou_loss": kind,
                "forward_graph_us": round(time_events(graph.replay, args.iters), 2),
                "fwd_bwd_us": round(time_events(fwd_bwd, max(args.iters // 5, 20)), 2),
                "k_loss_match_us": match_kernel_us(fwd, 50),
                "parity_ok": parity(heads, lab, cfg, kind),
            })
    res["parity_ok"] = all(r["parity_ok"] for r in res["runs"])
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if not res["parity_ok"]:
        raise SystemExit("parity check failed")


if __name__ == "__main__":
    main()
