"""Measures the fused training loss on fp32, fp16 and bf16 head tensors and prints one JSON line.

Workload: B=64 @608, 80 classes, 50 GT per image (synth_head_outputs seed 0, synth_labels seed 2, the workload of
tools/loss_probe.py).  The 16-bit heads are the fp32 ones rounded to the 16-bit type.  Every measured quantity is a CUDA-graph
replay timed with CUDA events over many replays; the dtypes are alternated over several rounds and the median per dtype is kept.

For each dtype:
  forward        fused_yolo_loss_components over the three scales (six kernels in one PDL chain)
  forward_backward  fused_yolo_loss and torch.autograd.grad with respect to the three heads (forward, scalar sum, backward)
  backward       the three yl_loss_backward_typed calls alone on the saved tables of one forward: a memset of the gradient
                 (B*M*85*esize bytes: 495 MB fp32, 247 MB 16-bit), the objectness plane and the matched cells
Parity (the script exits non-zero on a failure): the 16-bit components equal those of the fp32 path on the widened heads within
rtol 1e-12, and the 16-bit gradients (forward_backward and backward graphs) equal the fp32 path's gradients on the widened heads
rounded to the dtype, bit for bit (any NaN equals any NaN).

  python tools/amp_loss_probe.py [--out FILE]
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

B, IMG, C, N_GT = 64, 608, 80, 50
DTYPES = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}
CODES = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        name, power = [x.strip() for x in out[torch.cuda.current_device()].split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:  # the reading is informative; the measurement does not depend on it
        return {"name": torch.cuda.get_device_name(), "power_limit": "unknown (%s)" % type(e).__name__}


def capture(fn):
    """fn() warmed up on a side stream, then captured; returns (graph, fn's outputs inside the graph)."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fn()
    return g, out


def time_replays(g, iters, warm=10):
    for _ in range(warm):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / iters


def bit_equal16(a, b):
    na, nb = torch.isnan(a), torch.isnan(b)
    return bool(torch.equal(na, nb) and torch.equal(a.view(torch.int16)[~na], b.view(torch.int16)[~nb]))


class Case:
    """The three graphs of one dtype."""

    def __init__(self, heads, labels, cfg):
        from yolov4_b200 import _cabi
        from yolov4_b200.yololoss import fused_yolo_loss, fused_yolo_loss_components
        self.heads = [h.detach().requires_grad_(True) for h in heads]
        dt = heads[0].dtype
        self.g_fwd, self.comps = capture(lambda: fused_yolo_loss_components(self.heads, labels, cfg, 0.7))

        def fwd_bwd():
            loss = fused_yolo_loss(self.heads, labels, cfg, 0.7)
            return torch.autograd.grad(loss, self.heads)
        self.g_fb, self.grads_fb = capture(fwd_bwd)

        # backward alone: the saved tables of one forward, the three typed backward calls
        loss = fused_yolo_loss(self.heads, labels, cfg, 0.7)
        saved = loss.grad_fn.saved_tensors
        up = torch.ones(1, dtype=torch.float32, device="cuda")
        K = int(labels.shape[1])
        L = _cabi.lib()
        self.grads_b = [torch.empty(h.shape, dtype=dt, device="cuda") for h in self.heads]

        def bwd():
            for l, (h, g) in enumerate(zip(self.heads, self.grads_b)):
                gobj, mcell, mgrad = saved[3 * l:3 * l + 3]
                _cabi.check(L.yl_loss_backward_typed(gobj.data_ptr(), mcell.data_ptr(), mgrad.data_ptr(), up.data_ptr(), B,
                                                     int(h.shape[2]), K, C, g.data_ptr(), CODES[dt],
                                                     torch.cuda.current_stream().cuda_stream))
        self.g_b, _ = capture(bwd)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("amp_loss_probe.py measures on a GPU; there is none here")
    import yolov4_b200 as yb
    from yolov4_b200.synth import synth_head_outputs, synth_labels
    cfg = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": C}
    base = synth_head_outputs(B, IMG, C, seed=0, device="cuda")
    labels = synth_labels(B, IMG, n_valid=N_GT, seed=2, device="cuda")
    cases = {name: Case([r.to(dt) for r in base], labels, cfg) for name, dt in DTYPES.items()}
    times = {name: {"forward": [], "forward_backward": [], "backward": []} for name in DTYPES}
    for _ in range(args.rounds):
        for name, cs in cases.items():
            times[name]["forward"].append(time_replays(cs.g_fwd, args.iters))
            times[name]["forward_backward"].append(time_replays(cs.g_fb, args.iters))
            times[name]["backward"].append(time_replays(cs.g_b, args.iters))
    for cs in cases.values():                      # the outputs of the last replay of every graph
        cs.g_fwd.replay()
        cs.g_fb.replay()
        cs.g_b.replay()
    torch.cuda.synchronize()

    res = {"probe": "amp_loss_probe", "workload": "B=%d @%d, %d classes, %d GT/image, synth seeds 0 / 2" % (B, IMG, C, N_GT),
           "gpu": gpu_info(), "iters": args.iters, "rounds": args.rounds, "per_dtype": {}}
    ok = True
    for name, dt in DTYPES.items():
        cs = cases[name]
        esize = torch.tensor([], dtype=dt).element_size()
        entry = {"grad_bytes": sum(h.numel() for h in cs.heads) * esize, "components": cs.comps.tolist()}
        for k, v in times[name].items():
            entry[k + "_us"] = 1e6 * float(np.median(v))
            entry[k + "_rounds_us"] = [1e6 * t for t in v]
        if name != "fp32":
            # the fp32 path on the widened heads: its own graphs of the same three computations
            wide = Case([h.detach().float() for h in cs.heads], labels, cfg)
            wide.g_fwd.replay()
            wide.g_fb.replay()
            wide.g_b.replay()
            torch.cuda.synchronize()
            comps_ok = bool(np.allclose(cs.comps.cpu().numpy(), wide.comps.cpu().numpy(), rtol=1e-12, atol=0))
            fb_ok = all(g.dtype == dt and bit_equal16(g, w.to(dt)) for g, w in zip(cs.grads_fb, wide.grads_fb))
            b_ok = all(g.dtype == dt and bit_equal16(g, w.to(dt)) for g, w in zip(cs.grads_b, wide.grads_b))
            entry["parity"] = {"components_rtol_1e-12": comps_ok, "forward_backward_grads_bit_equal": fb_ok,
                               "backward_grads_bit_equal": b_ok}
            ok &= comps_ok and fb_ok and b_ok
            del wide
        res["per_dtype"][name] = entry
    res["parity_ok"] = bool(ok)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if not ok:
        raise SystemExit("parity check failed: a 16-bit result differs from the fp32 path on the widened heads")


if __name__ == "__main__":
    main()
