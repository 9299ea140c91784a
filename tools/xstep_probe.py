"""Cross-step pipelining probe: two independent postprocessors (own inputs, workspaces, CUDA graphs) replayed alternately
on one stream (serial) or on two streams (step i+1's streaming flag kernel next to step i's emit / NMS / gather)."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import yolov4_b200 as yb
from yolov4_b200.synth import synth_head_outputs
B = 64
hps = []
NHP = int(os.environ.get('NHP', '2'))
for seed in range(NHP):
    raws = synth_head_outputs(B, 608, 80, seed=seed, device="cuda")
    hp = yb.HeadPostprocessor(B, [76, 38, 19], 80, 1e-4, 0.4)
    hp.ws.buf.zero_()                      # (diagnostic builds that skip a scale leave its flag words untouched)
    hps.append(hp.capture(raws))
N = 200
def run(streams):
    for it in range(N):
        with torch.cuda.stream(streams[it % len(streams)]):
            hps[it % NHP].replay()
for name, prios in (("serial", None), ("%d streams" % NHP, (0,) * NHP)):
    streams = [torch.cuda.Stream()] if prios is None else [torch.cuda.Stream(priority=p) for p in prios]
    run(streams); torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(); 
    for s in streams: s.wait_event(ev0)
    run(streams)
    for s in streams: torch.cuda.current_stream().wait_stream(s)
    ev1.record(); torch.cuda.synchronize()
    t = ev0.elapsed_time(ev1) * 1e3 / N
    print("%s %-18s %.1f us/step %.0f img/s" % (os.environ.get("TAG", ""), name, t, B / t * 1e6), flush=True)
