"""Per-image detection cap (max_det) on the GPU: every capped result equals cap_spec.cap_detections applied to the uncapped
output and to the oracle's output, bit for bit (rows and counts), on every entry point that takes the cap."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

from oracle import oracle as orc                                     # noqa: E402  (checker only)
import yolov4_b200 as yb                                              # noqa: E402
from yolov4_b200 import _cabi                                         # noqa: E402
from yolov4_b200.synth import synth_head_outputs                      # noqa: E402

from cap_spec import cap_detections                                   # noqa: E402
from test_gpu_half_inputs import assert_lists_bit_equal               # noqa: E402

CFG80 = {"ANCHORS": yb.ANCHORS_PX, "ANCHOR_MASK": yb.ANCHOR_MASK, "N_CLASSES": 80}
KS = (1, 7, 100, 300, 10000)


def check_capped(fn, uncapped, oracle_rows, ks, what=""):
    """fn(max_det) -> list; each must equal the spec applied to the uncapped output and to the oracle's."""
    assert_lists_bit_equal(uncapped, oracle_rows, what=f"{what} uncapped vs oracle")
    for k in ks:
        got = fn(k)
        assert_lists_bit_equal(got, cap_detections(uncapped, k), what=f"{what} max_det {k} vs capped output")
        assert_lists_bit_equal(got, cap_detections(oracle_rows, k), what=f"{what} max_det {k} vs capped oracle")


@pytest.mark.parametrize("clustered,conf,nmst", [(False, 1e-4, 0.4), (True, 1e-4, 0.4), (False, 0.2, 0.5), (True, 0.2, 0.5)])
def test_fused_608(clustered, conf, nmst):
    raws = synth_head_outputs(4, 608, 80, seed=3 if clustered else 4, device="cuda", clustered=clustered,
                              fg_prob=0.02 if clustered else 0.005)
    unc = yb.detect_raw(raws, 80, conf, nmst)
    want = orc.detect([r.cpu().numpy() for r in raws], 80, conf, nmst, nthreads=8)
    check_capped(lambda k: yb.detect_raw(raws, 80, conf, nmst, max_det=k), unc, want, KS, what=f"608 conf {conf}")
    if conf < 0.1:
        assert min(len(u) for u in unc) > 300, "the cap must cut every image at 300"


@pytest.mark.parametrize("img,C,B", [(416, 80, 3), (96, 4, 5), (64, 128, 2)])
def test_fused_other_shapes(img, C, B):
    raws = synth_head_outputs(B, img, C, seed=img + C, device="cuda", fg_prob=0.05, clustered=True)
    for conf, nmst in ((1e-3, 0.45), (0.2, 0.5)):
        unc = yb.detect_raw(raws, C, conf, nmst)
        want = orc.detect([r.cpu().numpy() for r in raws], C, conf, nmst, nthreads=8)
        check_capped(lambda k: yb.detect_raw(raws, C, conf, nmst, max_det=k), unc, want, KS, what=f"{img} C {C}")


def _dense(raws):
    return torch.cat([yb.YOLOLayer(CFG80, l, device="cuda").eval()(r) for l, r in enumerate(raws)], 1)


@pytest.mark.parametrize("conf,nmst", [(1e-4, 0.4), (0.2, 0.5)])
def test_dense_postprocess_608(conf, nmst):
    raws = synth_head_outputs(4, 608, 80, seed=5, device="cuda", clustered=True, fg_prob=0.02)
    dense = _dense(raws)
    unc = yb.postprocess(dense, 80, conf, nmst)
    want = orc.postprocess(dense.cpu().numpy(), 80, conf, nmst, nthreads=8)
    check_capped(lambda k: yb.postprocess(dense, 80, conf, nmst, max_det=k), unc, want, KS, what=f"dense conf {conf}")


def test_dense_postprocess_pathological_values():
    """The inputs of the parity suite's pathological-values test (NaN / inf / negative / duplicates), with a cap."""
    rng = np.random.RandomState(5)
    B, M, C = 2, 600, 6
    pred = np.zeros((B, M, 5 + C), np.float32)
    pred[..., 0:2] = rng.rand(B, M, 2) * 100
    pred[..., 2:4] = rng.rand(B, M, 2) * 40
    pred[..., 4] = rng.rand(B, M)
    pred[..., 5:] = rng.rand(B, M, C) ** 3
    pred[0, 0:20, 2:4] = 0.0
    pred[0, 5:10, 0:2] = pred[0, 0:5, 0:2]
    pred[0, 30, 0] = np.nan
    pred[0, 31, 2] = np.inf
    pred[0, 32, 7] = np.nan
    pred[1, 40, 4] = np.nan
    pred[1, 41, 4] = -0.5
    pred[1, 50:60, :] = pred[1, 60:70, :]
    pred[1, 70:75, 4] = -2.0                                   # negative obj x negative cls: a positive score
    pred[1, 70:75, 5:] = -0.75
    gpu = torch.from_numpy(pred).cuda()
    for conf, nmst in ((0.05, 0.45), (0.3, 0.0001), (0.0, 0.5)):
        unc = yb.postprocess(gpu, C, conf, nmst)
        want = orc.postprocess(pred, C, conf, nmst)
        check_capped(lambda k: yb.postprocess(gpu, C, conf, nmst, max_det=k), unc, want, (1, 3, 10, 50, 200, 5000),
                     what=f"pathological conf {conf} nms {nmst}")


def test_all_ties_across_and_inside_classes():
    """All-zero logits: every score is exactly 0.25, so the cap cuts through one run of ties spanning classes."""
    raws = [torch.zeros(2, 255, f, f, device="cuda") for f in (8, 4, 2)]
    raws[0][1, 4] = -20.0                                      # image 1: the stride-8 boxes drop out
    unc = yb.detect_raw(raws, 80, 0.2, 0.5)
    want = orc.detect([r.cpu().numpy() for r in raws], 80, 0.2, 0.5, nthreads=8)
    per_class = np.bincount(want[0][:, 6].astype(int), minlength=80)
    assert per_class.min() > 1, "every class keeps several tied rows"
    ks = (1, 2, int(per_class[0]) + 1, 100, len(want[0]) - 1, len(want[0]))
    check_capped(lambda k: yb.detect_raw(raws, 80, 0.2, 0.5, max_det=k), unc, want, ks, what="all ties")


def test_rows_beyond_shared_memory_staging():
    """An image with more kept rows than k_select_topk stages in shared memory (16384): the global-memory path."""
    raws = [torch.zeros(2, 255, f, f, device="cuda") for f in (20, 10, 5)]
    raws[0][1, 4] = -20.0
    unc = yb.detect_raw(raws, 80, 0.2, 0.5)
    want = orc.detect([r.cpu().numpy() for r in raws], 80, 0.2, 0.5, nthreads=8)
    assert len(want[0]) > 16384
    check_capped(lambda k: yb.detect_raw(raws, 80, 0.2, 0.5, max_det=k), unc, want, (1, 300, 9999, 16384, len(want[0]) - 1),
                 what="global path")


def test_no_op_caps():
    raws = synth_head_outputs(4, 416, 80, seed=8, device="cuda", clustered=True, fg_prob=0.02)
    unc = yb.detect_raw(raws, 80, 1e-3, 0.45)
    kmax = max(len(u) for u in unc)
    for k in (kmax, kmax + 1, 2 * kmax + 3):
        assert_lists_bit_equal(yb.detect_raw(raws, 80, 1e-3, 0.45, max_det=k), unc, what=f"max_det {k} >= every count")
    # yl_nms_topk(max_det = 0) is yl_nms: same rows, same meta
    L = _cabi.lib()
    Fs = [r.shape[2] for r in raws]
    B, C, M, cap_seg, cap_out = 4, 80, sum(3 * f * f for f in Fs), 1024, 16384
    ws_bytes = L.yl_post_workspace_bytes(B, M, C, cap_seg)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    anch = _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh])
    mask = _cabi.ints([v for m in yb.ANCHOR_MASK for v in m])
    rp = _cabi.ptrs([r.data_ptr() for r in raws])
    st = torch.cuda.current_stream().cuda_stream
    outs = []
    for topk in (False, True):
        rows = torch.full((B, cap_out, 7), 7.0, device="cuda")
        meta = torch.full((3 * B,), -1, dtype=torch.int32, device="cuda")
        _cabi.check(L.yl_post_reset(ws.data_ptr(), ws_bytes, B, M, C, cap_seg, st))
        _cabi.check(L.yl_filter_raw_typed(rp, 0, _cabi.ints(Fs), 3, B, C, anch, mask, float(np.float32(1e-3)), ws.data_ptr(),
                                          ws_bytes, M, cap_seg, 0, B, 3, st))
        if topk:
            _cabi.check(L.yl_nms_topk(ws.data_ptr(), ws_bytes, B, M, C, cap_seg, float(np.float32(0.45)), 0, rows.data_ptr(),
                                      cap_out, meta.data_ptr(), None, 0, B, st))
        else:
            _cabi.check(L.yl_nms(ws.data_ptr(), ws_bytes, B, M, C, cap_seg, float(np.float32(0.45)), rows.data_ptr(), cap_out,
                                 meta.data_ptr(), 0, B, st))
        torch.cuda.synchronize()
        outs.append((rows.cpu().numpy(), meta.cpu().numpy()))
    assert np.array_equal(outs[0][1], outs[1][1])
    assert np.array_equal(outs[0][0].view(np.uint32), outs[1][0].view(np.uint32))


@pytest.mark.parametrize("n_groups,dt", [(1, torch.float32), (2, torch.float32), (1, torch.float16)])
def test_head_postprocessor_run_and_replay(n_groups, dt):
    B, K = 8, 300
    raws = [r.to(dt) for r in synth_head_outputs(B, 608, 80, seed=11, device="cuda")]
    hp = yb.HeadPostprocessor(B, [76, 38, 19], 80, 1e-4, 0.4, n_groups=n_groups, max_det=K)
    assert hp.cap_out == 300
    ref = yb.HeadPostprocessor(B, [76, 38, 19], 80, 1e-4, 0.4, n_groups=n_groups)
    _, meta_unc = ref.run(raws)
    want = yb.detect_raw(raws, 80, 1e-4, 0.4, max_det=K)
    assert_lists_bit_equal(want, cap_detections(yb.detect_raw(raws, 80, 1e-4, 0.4), K))
    hp.run(raws)
    torch.cuda.synchronize()
    assert_lists_bit_equal(hp.results(), want, what="run")
    assert torch.equal(hp.uncapped, meta_unc[:B])
    assert int(hp.meta[:B].max()) == K and int(hp.uncapped.min()) > K
    hp.capture(raws)
    hp.uncapped.zero_()
    hp.replay()
    torch.cuda.synchronize()
    assert_lists_bit_equal(hp.results(), want, what="replay")
    assert torch.equal(hp.uncapped, meta_unc[:B])
    fresh = [r.to(dt) for r in synth_head_outputs(B, 608, 80, seed=12, device="cuda")]
    for dst, src in zip(hp._captured_inputs, fresh):
        dst.copy_(src)
    hp.replay()
    torch.cuda.synchronize()
    assert_lists_bit_equal(hp.results(), yb.detect_raw(fresh, 80, 1e-4, 0.4, max_det=K), what="replay, new inputs")
    ref.run(fresh)
    torch.cuda.synchronize()
    assert torch.equal(hp.uncapped, ref.meta[:B])


@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16])
def test_detect_host_topk(dt):
    L = _cabi.lib()
    B, C, K = 6, 80, 100
    raws = [r.to(dt) for r in synth_head_outputs(B, 416, C, seed=21, fg_prob=0.02, clustered=True)]
    if dt == torch.float32:
        host, code = [r.numpy() for r in raws], 0
    else:
        host, code = [r.view(torch.int16).numpy().view(np.uint16) for r in raws], 2
    gpu = [r.cuda() for r in raws]
    Fs = [r.shape[2] for r in raws]
    ctx = ctypes.c_void_p()
    cap_out = 4096
    anch = _cabi.floats([v for wh in yb.ANCHORS_PX for v in wh])
    mask = _cabi.ints([v for m in yb.ANCHOR_MASK for v in m])
    _cabi.check(L.yl_context_create_typed(ctypes.byref(ctx), 0, B, _cabi.ints(Fs), 3, C, code, anch, mask, 1024, cap_out))
    try:
        rows = np.zeros((B, cap_out, 7), np.float32)
        counts = np.zeros((B,), np.int32)
        ptrs = _cabi.ptrs([h.ctypes.data for h in host])
        assert L.yl_detect_host_topk(ctx, ptrs, 0.001, 0.4, cap_out + 1, rows.ctypes.data, counts.ctypes.data) == 1
        assert L.yl_detect_host_topk(ctx, ptrs, 0.001, 0.4, -1, rows.ctypes.data, counts.ctypes.data) == 1
        for conf, nmst in ((0.001, 0.4), (0.2, 0.5)):
            rows[:] = np.nan
            _cabi.check(L.yl_detect_host_topk(ctx, ptrs, float(np.float32(conf)), float(np.float32(nmst)), K, rows.ctypes.data,
                                              counts.ctypes.data))
            want = yb.detect_raw(gpu, C, conf, nmst, max_det=K)
            got = [rows[b, :counts[b]] if counts[b] else None for b in range(B)]
            assert_lists_bit_equal(got, want, what=f"host path conf {conf}")
            assert all(np.isnan(rows[b, counts[b]:]).all() for b in range(B)), "only the capped rows are copied back"
            if conf < 0.01:
                assert counts.max() == K
    finally:
        _cabi.check(L.yl_context_destroy(ctx))


# ---- exchange sized by the cap ----------------------------------------------------------------------------------------
XB, XIMG, XC, XK = 4, 416, 80, 300


def _capped(seed, dev):
    raws = synth_head_outputs(XB, XIMG, XC, seed=seed, device=dev, fg_prob=0.02, clustered=True)
    hp = yb.HeadPostprocessor(XB, [XIMG // 8, XIMG // 16, XIMG // 32], XC, 1e-3, 0.4, device=dev, max_det=XK)
    rows, meta = hp.run(raws)
    torch.cuda.synchronize(dev)
    return hp, rows, meta, raws


def _xchg_worker(rank, world, port, q):
    try:
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(port)
        dev = torch.device("cuda", rank)
        torch.cuda.set_device(dev)
        if world > 1:
            dist.init_process_group("gloo", rank=rank, world_size=world)
        from yolov4_b200.sharded import DetectionExchange
        ex = DetectionExchange(XB, _capped(0, dev)[0].cap_out, dev, slots=2)
        ok, msg, n_rows = True, "", 0
        for step in range(3):
            slot = step % 2
            _, rows, meta, _ = _capped(100 * step + rank, dev)
            ex.push(rows, meta[:XB], slot)
            ex.wait(slot)
            got = ex.results(slot)
            for r in range(world):
                _, _, _, raws = _capped(100 * step + r, dev)
                want = cap_detections(yb.detect_raw(raws, XC, 1e-3, 0.4), XK)
                for b in range(XB):
                    g, w = got[r * XB + b], want[b]
                    good = (g is None) == (w is None) and (w is None or np.array_equal(
                        g.cpu().numpy().view(np.uint32), w.view(np.uint32)))
                    n_rows += 0 if w is None else len(w)
                    if not good and ok:
                        msg = "step %d source rank %d image %d differs" % (step, r, b)
                    ok = ok and good
            ex.release(slot)
        torch.cuda.synchronize(dev)
        ok = ok and ex.status() == 0 and n_rows > 100
        ex.close()
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        q.put((rank, bool(ok), msg))
    except Exception as e:                                        # pragma: no cover
        q.put((rank, False, repr(e)))


def _xchg_run(world):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_xchg_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert all(r[1] for r in res), res


def test_exchange_sized_by_the_cap_single_rank():
    hp = _capped(0, torch.device("cuda", 0))[0]
    assert hp.cap_out == 300
    _xchg_run(1)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_exchange_sized_by_the_cap_two_ranks():
    _xchg_run(2)
