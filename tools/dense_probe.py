"""Times the dense front end alone (yl_post_reset + yl_filter_dense) at the BASELINE size."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import yolov4_b200 as yb
from yolov4_b200 import _cabi
from yolov4_b200.synth import synth_head_outputs
B, C = int(os.environ.get("B", "64")), 80
cfg = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": C}
raws = synth_head_outputs(B, 608, C, seed=0, device="cuda")
dense = yb.decode_dense_cat(raws, cfg)
del raws
M = dense.shape[1]
L = _cabi.lib()
nb = L.yl_post_workspace_bytes(B, M, C, 1024)
ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
st = torch.cuda.current_stream().cuda_stream
for conf in (1e-4, 0.2):
    def run():
        _cabi.check(L.yl_post_reset(ws.data_ptr(), nb, B, M, C, 1024, st))
        _cabi.check(L.yl_filter_dense(dense.data_ptr(), B, M, C, C, float(torch.tensor(conf, dtype=torch.float32)), ws.data_ptr(), nb, 1024, 0, B, st))
    for _ in range(3): run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20): run()
    e1.record(); torch.cuda.synchronize()
    t = e0.elapsed_time(e1) / 20 * 1e3
    print("conf %g: %.1f us (reset + filter)  %.0f GB/s" % (conf, t, dense.numel() * 4 / t / 1e3))
