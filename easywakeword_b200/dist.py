"""Multi-GPU sharding of a stream bank: one process per GPU, contiguous blocks of stream ids per rank,
no data-path collective (streams are independent — the reference's multiroom shape is N independent
detectors, /root/reference/examples/multiroom_async.py:14-35).  The only exchange is the gather of the
dense 8-byte per-stream result records (score f32, flags u32) that K2/K3 write on the device:
`torch.distributed.all_gather_into_tensor` over NCCL/NVLink on GPUs, gloo on CPU tensors in tests.
"""
from __future__ import annotations

import numpy as np


def shard_range(n_total: int, world: int, rank: int) -> tuple[int, int]:
    """[first, last) global stream ids owned by `rank`: contiguous, sizes differ by at most one."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError("bad world/rank")
    base, rem = divmod(n_total, world)
    first = rank * base + min(rank, rem)
    return first, first + base + (1 if rank < rem else 0)


def owner_of(stream: int, n_total: int, world: int) -> tuple[int, int]:
    """(rank, local index) of a global stream id."""
    base, rem = divmod(n_total, world)
    cut = rem * (base + 1)
    if stream < cut:
        return stream // (base + 1), stream % (base + 1)
    return rem + (stream - cut) // base, (stream - cut) % base


def local_streams(global_streams, n_total: int, world: int, rank: int) -> list[int]:
    """Local indices, in the given order, of the global stream ids that `rank` owns (the rest belong to other ranks)."""
    out = []
    for g in global_streams:
        g = int(g)
        if not 0 <= g < n_total:
            raise ValueError(f"stream {g} outside [0, {n_total})")
        r, i = owner_of(g, n_total, world)
        if r == rank:
            out.append(i)
    return out


def padded_shard(n_total: int, world: int) -> int:
    """Per-rank record count used for the fixed-size all-gather (ceil(n_total / world))."""
    return -(-n_total // world)


class ResultGather:
    """Gathers per-stream result records from every rank into global stream order.

    local records: int32 tensor [padded_shard, 2] on the rank's device (bank kernels write the first
    n_local rows in place when it is installed with Context.set_results_buffer)."""

    def __init__(self, n_total: int, world: int, rank: int, device="cpu"):
        import torch
        self.torch = torch
        self.n_total, self.world, self.rank = n_total, world, rank
        self.first, self.last = shard_range(n_total, world, rank)
        self.n_local = self.last - self.first
        self.pad = padded_shard(n_total, world)
        self.local = torch.zeros(self.pad, 2, dtype=torch.int32, device=device)
        self.gathered = torch.zeros(world * self.pad, 2, dtype=torch.int32, device=device)
        # rows of `gathered` in global stream order
        idx = []
        for r in range(world):
            a, b = shard_range(n_total, world, r)
            idx.extend(range(r * self.pad, r * self.pad + (b - a)))
        self.index = torch.tensor(idx, dtype=torch.long, device=device)

    def gather(self):
        """-> int32 tensor [n_total, 2] (score bits, flags) in global stream order, on every rank."""
        import torch.distributed as dist
        if self.world > 1:
            dist.all_gather_into_tensor(self.gathered, self.local)
        else:
            self.gathered.copy_(self.local)
        return self.gathered.index_select(0, self.index)

    @staticmethod
    def decode(records) -> np.ndarray:
        """int32 [n, 2] -> structured array (score f32, flags u32) like Context.results()."""
        a = records.detach().cpu().numpy().astype(np.int32)
        out = np.empty(len(a), dtype=[("score", "<f4"), ("flags", "<u4")])
        out["score"] = a[:, 0].view(np.float32)
        out["flags"] = a[:, 1].view(np.uint32)
        return out


class ShardedBank:
    """A WakeWordBank over the rank's shard of `n_total` streams plus the result exchange.

    exchange="peer": K2 / K3 store the records and a completion signal into every rank's copy over NVLink
    (PeerResultExchange; needs torch symmetric memory); "nccl": one all-gather per gather() call; "auto": peer when
    available.  gather() returns int32 [n_total, 2] in global stream order either way."""

    def __init__(self, n_total: int, templates, *, world: int, rank: int, device: int, exchange: str = "auto", **bank_kwargs):
        import torch
        from .bank import WakeWordBank
        if exchange not in ("auto", "peer", "nccl"):
            raise ValueError("exchange must be 'auto', 'peer' or 'nccl'")
        self.first, self.last = shard_range(n_total, world, rank)
        self.n_total, self.world, self.rank = n_total, world, rank
        self.bank = WakeWordBank(self.last - self.first, templates, device=device, **bank_kwargs)
        dev = torch.device("cuda", device)
        self.gatherer = ResultGather(n_total, world, rank, device=dev)
        self.bank.ctx.set_results_buffer(self.gatherer.local.data_ptr())
        self.peer = None
        if exchange != "nccl" and world > 1:
            import torch.distributed as dist
            try:
                self.peer = PeerResultExchange(n_total, world, rank, dev)
            except Exception:
                if exchange == "peer":
                    raise
            ok = torch.tensor([1 if self.peer is not None else 0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)           # every rank takes the same path
            if int(ok.item()) == 0:
                if exchange == "peer":
                    raise RuntimeError("peer exchange unavailable on at least one rank")
                self.peer = None
            else:
                self.peer.install(self.bank.ctx)

    def step(self, pcm_local, where=0):
        self.bank.step(pcm_local, where)

    def step_streams(self, global_streams, blocks):
        """WakeWordBank.step_streams over global stream ids: every rank may be called with the whole list and keeps only
        the rows of the streams it owns (dist.local_streams)."""
        streams, rows = [], []
        for g, blk in zip(global_streams, blocks):
            loc = local_streams([g], self.n_total, self.world, self.rank)
            if loc:
                streams.append(loc[0])
                rows.append(blk)
        return self.bank.step_streams(streams, rows)

    def dense_ready(self, global_streams, template_first: int = 0, template_count=None, own_templates: bool = False):
        """WakeWordBank.dense_ready over global stream ids: every rank may be called with the whole list and scores the
        streams it owns (dist.local_streams).  Returns {global stream id: (first hop, float32 [n, T] scores)}."""
        loc = local_streams(global_streams, self.n_total, self.world, self.rank)
        if not loc:
            return {}
        kw = {"own_templates": True} if own_templates else {}
        hop0, rows = self.bank.dense_ready(loc, template_first, template_count, **kw)
        return {self.first + s: (int(h), r) for s, h, r in zip(loc, hop0, rows)}

    def dense_detect(self, global_streams, template_first: int = 0, template_count=None, hold_hops: int = 20,
                     refractory_hops: int = 50, own_templates: bool = False):
        """WakeWordBank.dense_detect over global stream ids: every rank may be called with the whole list and detects on
        the streams it owns (dist.local_streams).  Returns this rank's detections with global stream ids."""
        from . import _lib
        loc = local_streams(global_streams, self.n_total, self.world, self.rank)
        if not loc:
            return np.zeros(0, _lib.DETECTION_DTYPE)
        kw = {"own_templates": True} if own_templates else {}
        det = self.bank.dense_detect(loc, template_first, template_count, hold_hops, refractory_hops, **kw)
        det["stream"] += self.first
        return det

    def gather(self):
        ctx = self.bank.ctx
        if self.peer is not None and ctx.publish_seq() > 0:
            self.peer.wait(ctx)                                  # every rank's records of the latest call have landed
            seqs, timed_out = self.peer.published(ctx)           # (synchronises the context's stream)
            if timed_out:
                raise TimeoutError(f"peer publication: ranks are at calls {seqs.tolist()}, expected {ctx.publish_seq()}")
            return self.peer.records(ctx.publish_parity())
        ctx.join()                        # overlap mode: the records are complete once K3 has been joined
        return self.gatherer.gather()

    def reset(self, global_streams, **overrides):
        """Recycle global streams: every rank is called with the same list and resets the streams it owns
        (WakeWordBank.reset).  Returns this rank's drained events with global stream ids."""
        ev = self.bank.reset(local_streams(global_streams, self.n_total, self.world, self.rank), **overrides)
        ev["stream"] += self.first
        return ev

    def poll_global(self):
        """Local events with global stream ids."""
        ev = self.bank.poll()
        ev["stream"] += self.first
        return ev

    def close(self):
        if self.peer is not None:
            self.bank.ctx.set_results_peers([])
        self.bank.close()


def bind_host_near_gpu(device_index: int):
    """Pins the calling process to the CPUs NVML reports as local to CUDA device `device_index` (its NUMA node /
    PCIe root), so that pinned staging memory allocated afterwards is first-touched next to the GPU and the
    H2D copies of a rank do not cross the socket interconnect when 8 ranks share one host.

    Returns the CPU list that was applied, or None when NVML / the affinity call is unavailable or the mask is
    empty (the process is left as it was: this is a placement hint, never a requirement)."""
    import os
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        p = torch.cuda.get_device_properties(device_index)
        bus = f"{p.pci_domain_id:08x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        ncpu = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        allowed = os.sched_getaffinity(0)
        cpus = sorted(c for c in range(ncpu) if (mask[c // 64] >> (c % 64)) & 1 and c in allowed)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return cpus
    except Exception:
        return None


class PeerResultExchange:
    """The result "gather" done by the producing kernels: every rank owns a symmetric buffer — two parity copies of the
    global record array, int32 [2][world * pad][2], plus a signal row uint64 [2][16] — that all ranks of the NVLink
    domain map (torch symmetric memory: CUDA VMM allocations whose handles are exchanged at rendezvous).  K2 / K3 of
    every rank store each record they write straight into all copies, and the last K3 CTA of a tick call releases the
    call's sequence number into slot `rank` of every signal row (`ewk_set_results_peers`): a put-with-signal.  No
    all-gather and no per-step barrier: a consumer that needs call q of every rank waits for the signals
    (`wait(ctx)` on the device, `published(ctx)` from the host).  `barrier(ctx)` is the lock-step alternative.
    `view(parity)` is this rank's copy; `records(parity)` selects the valid rows in global stream order."""

    SIG = 16                                   # ewk::MAX_PUB slots per signal row

    def __init__(self, n_total: int, world: int, rank: int, device, group=None):
        import torch
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        if world > self.SIG:
            raise ValueError(f"peer publication supports up to {self.SIG} ranks")
        self.torch = torch
        self.n_total, self.world, self.rank = n_total, world, rank
        self.first, self.last = shard_range(n_total, world, rank)
        self.pad = padded_shard(n_total, world)
        self.stride = world * self.pad
        self.device = torch.device(device)
        self.raw = symm.empty((2 * self.stride + 2 * self.SIG,), dtype=torch.int64, device=self.device)
        self.raw.zero_()
        torch.cuda.synchronize(self.device)
        self.hdl = symm.rendezvous(self.raw, group if group is not None else dist.group.WORLD)
        self.ptrs = [int(p) for p in self.hdl.buffer_ptrs]
        if len(self.ptrs) != world or not all(self.ptrs):
            raise RuntimeError("symmetric memory rendezvous returned no peer pointers")
        self.sig_ptrs = [p + 2 * self.stride * 8 for p in self.ptrs]
        self.buf = self.raw[:2 * self.stride].view(torch.int32).view(2, self.stride, 2)
        self.sig = self.raw[2 * self.stride:].view(2, self.SIG)
        idx = []
        for r in range(world):
            a, b = shard_range(n_total, world, r)
            idx.extend(range(r * self.pad, r * self.pad + (b - a)))
        self.index = torch.tensor(idx, dtype=torch.long, device=self.device)
        self._ext = {}
        self.last_stream = None

    def install(self, ctx):
        """Point the context's kernels at every rank's copy (this rank's included) and start a new sequence."""
        self.raw[2 * self.stride:].zero_()
        self.torch.cuda.synchronize(self.device)
        self.hdl.barrier()                     # nobody publishes into a signal row that is still being cleared
        self.torch.cuda.synchronize(self.device)
        ctx.set_results_peers(self.ptrs, stride_records=self.stride, offset_records=self.rank * self.pad,
                              signals=self.sig_ptrs, slot=self.rank)

    def wait(self, ctx, seq=None, timeout_ms=2000):
        """Enqueue on the context's stream a (bounded) wait until every rank's records of call `seq` (default: this
        rank's latest) are in this rank's copy."""
        ctx.wait_published(self.world, ctx.publish_seq() if seq is None else seq, timeout_ms)

    def published(self, ctx, parity=None):
        """Host read: sequence number each rank has completed in the given parity copy (default: the latest)."""
        par = ctx.publish_parity() if parity is None else parity
        return ctx.published_seq(par, self.world)

    def barrier(self, ctx):
        """Lock-step alternative to the signals: a symmetric-memory barrier enqueued on the stream the tick launched K3
        on (the match stream in overlap mode), so the next push and gate do not wait for it."""
        torch = self.torch
        h = ctx.match_stream()
        cur = torch.cuda.current_stream(self.device)
        if not h or h == cur.cuda_stream:
            s = cur
        else:
            s = self._ext.get(h)
            if s is None:
                s = self._ext[h] = torch.cuda.ExternalStream(h, device=self.device)
        with torch.cuda.stream(s):
            self.hdl.barrier()
        self.last_stream = s
        return s

    def finish(self, stream=None):
        """Make `stream` (default: the current one) wait for the latest barrier."""
        if self.last_stream is not None:
            (stream or self.torch.cuda.current_stream(self.device)).wait_stream(self.last_stream)

    def view(self, parity: int):
        """int32 [world * pad, 2] records of the tick call that published with `parity` (ctx.publish_parity())."""
        return self.buf[parity]

    def records(self, parity: int):
        """-> int32 [n_total, 2] in global stream order."""
        return self.buf[parity].index_select(0, self.index)
