"""Image-group pipelining probe: flag/emit of group g+1 on the main stream next to NMS/gather of group g on a side
stream, as a CUDA graph, for each group count."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import yolov4_b200 as yb
from yolov4_b200.synth import synth_head_outputs
B = 64
raws = synth_head_outputs(B, 608, 80, seed=0, device="cuda")
ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
def timeit(hp, n=100):
    for _ in range(10): hp.replay()
    torch.cuda.synchronize(); ev0.record()
    for _ in range(n): hp.replay()
    ev1.record(); torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) * 1e3 / n
GROUPS = [int(g) for g in os.environ.get("GROUPS", "1,2,4,8").split(",")]
for G in GROUPS:
    hp = yb.HeadPostprocessor(B, [76, 38, 19], 80, 1e-4, 0.4, n_groups=G).capture(raws)
    t = timeit(hp)
    print("groups %2d: %.1f us/step %.0f img/s" % (G, t, B / t * 1e6), flush=True)
