"""GPU (>= 2 devices for the multi-rank cases; `python -m pytest tests/test_exchange_multigpu.py -m gpu`): the final exchange of the
image-sharded path (yl_xchg_*, sharded.DetectionExchange) -- every rank ends up with the detections of every image, bit for bit
what the owning rank computed, over several steps that reuse the double-buffered slots (epoch / credit protocol), with the
ranks deliberately out of step.  One process per GPU; torch.distributed (gloo) only carries the 64-byte IPC handles.
With one visible GPU the single-rank form (self window) is still exercised."""
import os
import socket
import time

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

B, IMG, C, CONF, NMS = 4, 416, 80, 1e-3, 0.4
STEPS = 5
CAP = 32768


def _detect(seed, dev):
    import yolov4_b200 as yb
    from yolov4_b200.synth import synth_head_outputs
    raws = synth_head_outputs(B, IMG, C, seed=seed, device=dev, fg_prob=0.02, clustered=True)
    hp = yb.HeadPostprocessor(B, [IMG // 8, IMG // 16, IMG // 32], C, CONF, NMS, device=dev, cap_out=CAP)
    rows, meta = hp.run(raws)
    torch.cuda.synchronize(dev)
    return hp, rows, meta


def _worker(rank, world, port, q, backend="gloo"):
    try:
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(port)
        dev = torch.device("cuda", rank)
        torch.cuda.set_device(dev)
        if world > 1:
            if backend == "nccl":
                dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
            else:
                dist.init_process_group("gloo", rank=rank, world_size=world)
        from yolov4_b200.sharded import DetectionExchange
        ex = DetectionExchange(B, CAP, dev, slots=2)
        mode = ex.mode
        ok, n_rows, first_bad = True, 0, ""
        for step in range(STEPS):
            slot = step % 2
            hp, rows, meta = _detect(1000 * step + rank, dev)
            if rank == step % world:
                time.sleep(0.05)                                  # ranks out of step: the wait / credit flags do the ordering
            ex.push(rows, meta[:B], slot)
            ex.wait(slot)
            got = ex.results(slot)
            assert len(got) == world * B
            for r in range(world):
                _, rr, mm = _detect(1000 * step + r, dev)         # recomputed here: images are independent of their rank
                cnt = mm[:B].cpu().numpy()
                for b in range(B):
                    g = got[r * B + b]
                    k = int(cnt[b])
                    if k == 0:
                        good = g is None
                    else:
                        good = g is not None and g.shape[0] == k and \
                            np.array_equal(g.cpu().numpy().view(np.uint32), rr[b, :k].cpu().numpy().view(np.uint32))
                        n_rows += k
                    if not good and ok:
                        first_bad = "step %d slot %d source rank %d image %d: want %d rows, got %s" % (
                            step, slot, r, b, k, None if g is None else tuple(g.shape))
                    ok = ok and good
            ex.release(slot)
        torch.cuda.synchronize(dev)
        st_ = ex.status()
        if st_ != 0 or n_rows <= 100:
            first_bad += " status %d n_rows %d" % (st_, n_rows)
        ok = ok and st_ == 0 and n_rows > 100
        ex.close()
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        q.put((rank, bool(ok), n_rows, first_bad + " [" + mode + "]"))
    except Exception as e:                                        # pragma: no cover
        q.put((rank, False, repr(e)))


def _run(world, backend="gloo"):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, backend)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert all(r[1] for r in res), res
    return res


def test_exchange_single_rank_self_window():
    _run(1)


def test_exchange_single_rank_register_staged_push(monkeypatch):
    monkeypatch.setenv("YL_XCHG_BULK", "0")          # read by yl_xchg_create in the spawned worker
    _run(1)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_exchange_two_ranks_bit_exact_over_reused_slots():
    _run(2)


@pytest.mark.skipif(torch.cuda.device_count() < 4, reason="needs four GPUs")
def test_exchange_four_ranks_bit_exact_over_reused_slots():
    _run(4)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_exchange_two_ranks_multicast_or_its_fallback():
    """With an NCCL group the windows live in torch symmetric memory and the push is one multimem.st per 16 bytes (NVSwitch
    multicast); where the platform has no multicast mapping every rank falls back to the CUDA IPC windows.  Either way: bit-exact."""
    res = _run(2, backend="nccl")
    print("exchange mode:", res[0][3])
