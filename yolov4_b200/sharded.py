"""Image-sharded multi-GPU form of the hot path (SURVEY.md 8(e)).

Images are independent in decode, filter, sort and NMS (utils.py:133 loops per image), so rank r of G simply owns the
contiguous image range shard_range(B, r, G) and runs the single-GPU path on it: no collective on the hot path.
Only the final detections are exchanged: one all-gather of the per-image counts and one of the rows, trimmed to
the largest per-image count so no padding beyond that travels over NVLink.
"""
import torch
import torch.distributed as dist


def shard_range(n_images, rank, world):
    """Contiguous, balanced image range [lo, hi) of rank `rank` (first n_images % world ranks get one extra)."""
    base, extra = divmod(n_images, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def allgather_detections(rows, counts, group=None):
    """rows [B_local, cap, 7] (padded, device or CPU), counts [B_local] int32 -> list over ALL images (rank-major) of
    [K_i, 7] tensors or None, identical on every rank.  All ranks must hold the same B_local (pad the last shard)."""
    world = dist.get_world_size(group)
    b_local = counts.shape[0]
    all_counts = torch.empty((world * b_local,), dtype=counts.dtype, device=counts.device)
    dist.all_gather_into_tensor(all_counts, counts.contiguous(), group=group)
    counts_host = all_counts.cpu()
    k_max = int(counts_host.max()) if counts_host.numel() else 0
    if k_max > rows.shape[1]:
        raise RuntimeError("a rank truncated its rows (count %d > capacity %d)" % (k_max, rows.shape[1]))
    k_max = max(k_max, 1)
    send = rows[:, :k_max].contiguous()
    recv = torch.empty((world * b_local, k_max, 7), dtype=rows.dtype, device=rows.device)
    dist.all_gather_into_tensor(recv, send, group=group)
    out = []
    for i in range(world * b_local):
        k = int(counts_host[i])
        out.append(recv[i, :k] if k else None)
    return out


class DetectionExchange:
    """The final exchange as part of the device path (SURVEY.md 8(e)): kept rows go from the NMS output buffer of every rank
    straight into every rank's gathered buffer by peer stores over NVLink (yl_xchg_*: one window per rank, mapped by the
    peers through CUDA IPC), counts stay on the device, nothing synchronises with the host, and the three kernels of an
    exchange (push / wait / release) are graph-capturable, so the exchange of step i runs under the kernels of step i+1.

        ex = DetectionExchange(B_local, cap_out, device)        # collective: all ranks of `group` (handles are all-gathered)
        ex.push(rows, counts, slot); ex.wait(slot)               # on the current stream
        out = ex.results(slot)                                   # lazily built list over ALL world*B images (one D2H of counts)
        ex.release(slot)                                         # the slot may be pushed into again by every rank

    torch.distributed is used once, for the 64-byte handles; NCCL moves no detection.  world == 1 works (self window)."""

    def __init__(self, b_local, cap_out, device, slots=2, group=None, multicast="auto"):
        import ctypes
        import os

        import numpy as np
        from . import _cabi
        self._cabi, self.L = _cabi, _cabi.lib()
        self.device = torch.device(device)
        self.B, self.cap_out, self.slots = int(b_local), int(cap_out), int(slots)
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.h = ctypes.c_void_p()
        self._views = {}
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.mode = "peer stores into CUDA IPC windows"
        if multicast == "auto":
            multicast = os.environ.get("YL_XCHG_MC", "1") != "0"
        if multicast and self.world > 1 and dist.get_backend(group) == "nccl" and self._try_multicast(dev_index, group):
            return
        _cabi.check(self.L.yl_xchg_create(ctypes.byref(self.h), dev_index, self.rank, self.world, self.B, self.cap_out, self.slots))
        nb = int(self.L.yl_xchg_handle_bytes())
        mine = (ctypes.c_ubyte * nb)()
        _cabi.check(self.L.yl_xchg_local_handle(self.h, mine))
        if self.world > 1:
            local = torch.tensor(list(bytes(mine)), dtype=torch.uint8, device=self.device if dist.get_backend(group) == "nccl" else "cpu")
            allh = torch.empty((self.world * nb,), dtype=torch.uint8, device=local.device)
            dist.all_gather_into_tensor(allh, local, group=group)
            blob = bytes(allh.cpu().numpy().astype(np.uint8).tobytes())
        else:
            blob = bytes(mine)
        buf = (ctypes.c_ubyte * len(blob)).from_buffer_copy(blob)
        _cabi.check(self.L.yl_xchg_connect(self.h, buf))
        if self.world > 1:
            dist.barrier(group=group)                      # every window is mapped before anybody pushes

    def _try_multicast(self, dev_index, group):
        """Windows in torch symmetric memory with an NVSwitch multicast mapping: yl_xchg_push then issues one bulk store to the
        multicast mapping and the switch replicates it (a rank sends 1/world of the bytes).  torch only allocates and maps the
        memory; the kernels are the library's.  All ranks agree on the outcome; any failure falls back to the CUDA IPC windows."""
        import ctypes
        ok, ptrs, mc = 1, None, 0
        try:
            import torch.distributed._symmetric_memory as symm
            nbytes = int(self.L.yl_xchg_window_bytes(self.world, self.B, self.cap_out, self.slots))
            self._symm_buf = symm.empty(nbytes, dtype=torch.uint8, device=self.device)
            hdl = symm.rendezvous(self._symm_buf, dist.group.WORLD if group is None else group)
            ptrs = [int(p) for p in hdl.buffer_ptrs]
            mc = int(hdl.multicast_ptr or 0)
            if mc == 0 or len(ptrs) != self.world:
                ok = 0
            self._symm_hdl = hdl
        except Exception:
            ok = 0
        flag = torch.tensor([ok], device=self.device, dtype=torch.int32)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        if int(flag.item()) == 0:
            self._symm_buf = self._symm_hdl = None
            return False
        arr = (ctypes.c_void_p * self.world)(*ptrs)
        self._cabi.check(self.L.yl_xchg_create_external(ctypes.byref(self.h), dev_index, self.rank, self.world, self.B, self.cap_out,
                                                         self.slots, arr, ctypes.c_void_p(mc)))
        dist.barrier(group=group)                          # every window's flags are zero before anybody pushes
        self.mode = "NVSwitch multicast (multimem.st) into symmetric-memory windows"
        return True

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def push(self, rows, counts, slot):
        if rows.dtype != torch.float32 or not rows.is_cuda or not rows.is_contiguous() or tuple(rows.shape) != (self.B, self.cap_out, 7):
            raise ValueError("rows must be a contiguous float32 CUDA tensor [B, cap_out, 7]")
        if counts.dtype != torch.int32 or not counts.is_cuda or counts.numel() < self.B:
            raise ValueError("counts must be an int32 CUDA tensor with at least B entries")
        self._cabi.check(self.L.yl_xchg_push(self.h, rows.data_ptr(), counts.data_ptr(), int(slot), self._stream()))

    def wait(self, slot):
        self._cabi.check(self.L.yl_xchg_wait(self.h, int(slot), self._stream()))

    def release(self, slot):
        self._cabi.check(self.L.yl_xchg_release(self.h, int(slot), self._stream()))

    def _view(self, ptr, shape, dtype):
        """A torch view of library-owned device memory (no copy) through the CUDA array interface."""
        n = 1
        for s in shape:
            n *= s

        class _Mem:
            pass
        m = _Mem()
        m.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f4" if dtype == torch.float32 else "<i4",
                                      "data": (int(ptr), False), "version": 2}
        return torch.as_tensor(m, device=self.device)

    def gathered(self, slot):
        """(rows [world*B, cap_out, 7], counts [world*B]) device views of this rank's gathered buffers of a slot."""
        if slot not in self._views:
            n = self.world * self.B
            self._views[slot] = (self._view(self.L.yl_xchg_rows(self.h, int(slot)), (n, self.cap_out, 7), torch.float32),
                                 self._view(self.L.yl_xchg_counts(self.h, int(slot)), (n,), torch.int32))
        return self._views[slot]

    def status(self):
        """0 ok; 1 / 2: a push / wait gave up after its time limit (a rank is missing or stuck).  Synchronises."""
        return int(self._view(self.L.yl_xchg_status(self.h), (1,), torch.int32).cpu()[0])

    def results(self, slot):
        """List over all world*B images (rank-major) of [K_i, 7] device views / None, built from the gathered buffers (one D2H
        of the counts).  Call after wait(slot) has been enqueued; the views are valid until release(slot)."""
        rows, counts = self.gathered(slot)
        ch = counts.cpu()
        if self.status() != 0:
            raise RuntimeError("detection exchange timed out (status %d)" % self.status())
        return [rows[i, :int(ch[i])] if int(ch[i]) else None for i in range(rows.shape[0])]

    def close(self):
        if self.h:
            self._views = {}
            self._cabi.check(self.L.yl_xchg_destroy(self.h))
            self.h = None
