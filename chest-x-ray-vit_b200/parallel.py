"""Data-parallel gradient synchronisation for the batch-sharded training path.

The reference trains 8 replicas with gradients averaged implicitly inside the XLA optimizer
step (/root/reference/ViT-Training.py:106,165,170; HF trainer.py:1760,1796).  Here every rank
owns one GPU, the batch is sharded by rank, and the only collective of the path is an
all-reduce (mean) of the flat fp32 gradient buffer, issued bucket by bucket while backward is
still running: the weight gradients of adjacent encoder layers are contiguous in the flat layout
(28.3 MB per ViT-B layer) and are coalesced into buckets of ``layers_per_bucket`` layers (default
3; a sequence such as (3, 3, 3, 2, 1) tapers them) in the order backward finishes them, then one
bucket for everything else.  NCCL runs the buckets on its own stream over NVLink/NVSwitch; the
compute stream only waits after the last bucket, right before the optimizer needs the gradients.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist


class GradSync:
    def __init__(self, layer_ranges: Sequence[Tuple[int, int]], rest_ranges: Sequence[Tuple[int, int]],
                 process_group: Optional[dist.ProcessGroup] = None, layers_per_bucket=3):
        self.layer_ranges = list(layer_ranges)
        self.rest_ranges = list(rest_ranges)
        self.pg = process_group
        self.world = dist.get_world_size(process_group) if dist.is_initialized() else 1
        # int: uniform buckets; sequence: bucket sizes in the order the layers finish (top layer first), the last
        # entry repeating — e.g. (3, 3, 3, 2, 1) tapers the buckets so the all-reduce left after backward is short
        sizes = [layers_per_bucket] if isinstance(layers_per_bucket, int) else list(layers_per_bucket)
        self.bucket_sizes = [max(1, int(x)) for x in sizes] or [3]
        self.bucket_index = 0
        self.flat: Optional[torch.Tensor] = None
        self.works: List = []
        self.pending: List[int] = []
        self.bytes_reduced = 0
        self.collectives = 0
        self._deferred: Optional[Tuple[int, int]] = None
        self._after = None                # event after which the ranges being reduced are complete (None: current stream)
        self._aux: Optional[torch.cuda.Stream] = None

    @classmethod
    def attach(cls, model, process_group=None, layers_per_bucket=3) -> "GradSync":
        gs = cls(model.layout.layer_range, model.layout.rest_ranges, process_group, layers_per_bucket)
        eng = model.engine()
        eng.grad_sync = gs
        eng.arenas.clear()          # launch plans bake the SM budget left to the collective
        return gs

    # called by Engine.backward ------------------------------------------------
    def begin(self, model_or_flat) -> None:
        """Called by Engine.backward with the buffer this backward writes (the flat gradient buffer, or the staging
        buffer when ``param.grad`` is already populated)."""
        self.flat = model_or_flat if isinstance(model_or_flat, torch.Tensor) else model_or_flat.flat_grads()
        self.works, self.pending = [], []
        self.bucket_index = 0
        self._deferred = None

    def layer_ready(self, l: int, after=None) -> None:
        """Layer ``l``'s weight gradients are enqueued on the current stream (layers finish in
        descending order) — or, with ``after`` (a CUDA event), are complete once that event has fired.  Adjacent layers
        are coalesced into one contiguous bucket."""
        self._after = after
        self.pending.append(l)
        size = self.bucket_sizes[min(self.bucket_index, len(self.bucket_sizes) - 1)]
        if len(self.pending) >= size or l == 0:
            lo, hi = min(self.pending), max(self.pending)
            rng = (self.layer_ranges[lo][0], self.layer_ranges[hi][1])
            if l == 0:
                # the bucket that ends with layer 0 finishes only a few kernels before everything else (embeddings,
                # biases): it is reduced together with those in rest_ready — fewer, larger operations in the part of the
                # all-reduce that no backward work is left to hide
                self._deferred = rng
            else:
                self._reduce(*rng)
            self.pending = []
            self.bucket_index += 1

    def bucket_end_layers(self) -> set:
        """Layers whose ``layer_ready`` call completes a bucket (layers finish in descending order).  The engine only
        needs a host callback — i.e. a break in its CUDA-graph segments — at these; the others are replayed for free."""
        ends, pending, bi = set(), 0, 0
        for l in reversed(range(len(self.layer_ranges))):
            pending += 1
            if pending >= self.bucket_sizes[min(bi, len(self.bucket_sizes) - 1)] or l == 0:
                ends.add(l)
                pending, bi = 0, bi + 1
        return ends

    def layers_ready(self, lo: int, hi: int, after=None) -> None:
        """Layers lo … hi (inclusive; a whole bucket) have their weight gradients enqueued on the current stream, or are
        complete once the event ``after`` has fired (the engine's launch plan records it between the bucket's last
        weight-gradient GEMM and the next layer; as an external event it is a node of the backward CUDA graph)."""
        for l in range(hi, lo - 1, -1):
            self.layer_ready(l, after)

    def _final_ranges(self) -> List[Tuple[int, int]]:
        """The deferred last layer bucket and the non-layer ranges, adjacent ones coalesced."""
        rs = sorted(([self._deferred] if self._deferred is not None else []) + [r for r in self.rest_ranges if r[1] > r[0]])
        self._deferred = None
        out: List[Tuple[int, int]] = []
        for s, e in rs:
            if out and out[-1][1] == s:
                out[-1] = (out[-1][0], e)
            else:
                out.append((s, e))
        return out

    def rest_ready(self, after=None) -> None:
        self._after = after
        self._reduce_many(self._final_ranges())
        self.wait()

    def _reduce_many(self, ranges: List[Tuple[int, int]]) -> None:
        for s, e in ranges:
            self._reduce(s, e)

    def wait(self) -> None:
        for w in self.works:
            w.wait()
        self.works = []

    # ---------------------------------------------------------------------------
    def _reduce(self, start: int, end: int) -> None:
        if self.world == 1 or end <= start:
            return
        t = self.flat[start:end]
        self.bytes_reduced += t.numel() * t.element_size()
        self.collectives += 1
        if t.is_cuda:
            if self._after is not None:
                # issue from an auxiliary stream that waits for the bucket's event: NCCL's own stream then depends on the
                # event, not on everything the main stream has been given since (the rest of backward)
                if self._aux is None:
                    self._aux = torch.cuda.Stream(device=t.device)
                self._aux.wait_event(self._after)
                with torch.cuda.stream(self._aux):
                    self.works.append(dist.all_reduce(t, op=dist.ReduceOp.AVG, group=self.pg, async_op=True))
            else:
                self.works.append(dist.all_reduce(t, op=dist.ReduceOp.AVG, group=self.pg, async_op=True))
        else:   # gloo (CPU tests) has no AVG
            w = dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.pg, async_op=True)
            w.wait()
            t.mul_(1.0 / self.world)


class PeerGradSync(GradSync):
    """The same bucket schedule with the all-reduce done over NVLink PEER MEMORY by the copy engines instead of NCCL.

    Why: NCCL's ring all-reduce runs as a 32-CTA kernel next to the backward GEMMs.  Those are persistent 148-CTA
    cluster kernels with a static tile schedule and 227 KB of shared memory per CTA — an SM held by NCCL cannot take a
    GEMM CTA, the CTA pairs that found no SM at launch start a whole tile late, and the step loses about as much time as
    the all-reduce lasts (7.74 → 8.27 ms at 2 GPUs, NCCL_DEBUG: "Algo RING proto SIMPLE channel 0..31").  Here the
    gradient buffer lives in symmetric memory (every rank maps every peer's buffer), and a bucket is reduced as

        barrier                         all ranks have finished computing the bucket
        pull   (copy engines)           my 1/N shard of the bucket from each of the N−1 peers into scratch
        vitk_shard_mean                 my shard ← mean over ranks (HBM-bound, two CTAs per SM for ≈70 µs per 85 MB bucket,
                                        fixed summation order)
        barrier                         every owner has reduced its shard
        pull   (copy engines)           the other N−1 reduced shards from their owners into my gradient buffer

    on a highest-priority communication stream, overlapped with the rest of backward; the SMs only ever see the short mean
    kernel and two one-CTA barrier kernels per bucket.  Wire bytes per GPU are those of a ring all-reduce, 2·(N−1)/N of the
    buffer.  Every rank ends up with the owner's bits, so replicas stay bit-identical."""

    def __init__(self, model, process_group=None, layers_per_bucket=3):
        import torch.distributed._symmetric_memory as symm_mem
        super().__init__(model.layout.layer_range, model.layout.rest_ranges, process_group, layers_per_bucket)
        if self.world < 2:
            raise ValueError("PeerGradSync needs an initialised process group with world size >= 2")
        self.rank = dist.get_rank(process_group)
        group = process_group if process_group is not None else dist.group.WORLD
        dev = model.flat_parameters().device
        total = model.layout.total
        # shards are cut at multiples of 4 elements (16-byte vectors); pad the buffer so every shard of every bucket exists
        self.padded = (total + 4 * self.world + 3) // 4 * 4
        sym = symm_mem.empty(self.padded, dtype=torch.float32, device=dev)
        sym.zero_()
        self.hdl = symm_mem.rendezvous(sym, group)
        self.sym = sym
        self.peer_bufs = {p: self.hdl.get_buffer(p, (self.padded,), torch.float32, 0) for p in range(self.world) if p != self.rank}
        model.set_flat_grads(sym[:total])
        longest = max([e - s for s, e in self.layer_ranges] + [e - s for s, e in self.rest_ranges])
        per_bucket = max(self.bucket_sizes) * longest
        self.max_shard = (per_bucket + self.world - 1) // self.world // 4 * 4 + 4
        self.scratch = torch.empty((self.world - 1) * self.max_shard, dtype=torch.float32, device=dev)
        # highest stream priority: the persistent backward GEMMs keep every SM busy (227 KB of shared memory per CTA leaves no
        # room for a second CTA), so the small mean / barrier kernels only get SMs at kernel boundaries — and must get them
        # FIRST there, or they starve (measured: 485 µs for a 20 µs kernel at default priority)
        self.comm = torch.cuda.Stream(device=dev, priority=-1)
        self._chan = 0
        self._last = None
        self.timeout_ms = 20000           # a protocol bug traps after 20 s instead of hanging the GPUs
        self.timing = None                # set to [] to collect (start, end, [events], t_host) per bucket (diagnostics)

    @classmethod
    def attach(cls, model, process_group=None, layers_per_bucket=3) -> "PeerGradSync":
        gs = cls(model, process_group, layers_per_bucket)
        eng = model.engine()
        eng.grad_sync = gs
        eng.arenas.clear()
        return gs

    def begin(self, model_or_flat) -> None:
        flat = model_or_flat if isinstance(model_or_flat, torch.Tensor) else model_or_flat.flat_grads()
        if flat.data_ptr() != self.sym.data_ptr():
            raise NotImplementedError("PeerGradSync reduces the symmetric gradient buffer only: a backward that finds param.grad "
                                      "already populated writes a staging buffer — call zero_grad(set_to_none=True) between steps "
                                      "(for micro-batch accumulation, detach the sync for all but the last micro-batch)")
        super().begin(flat)

    def _barrier(self) -> None:
        self.hdl.barrier(channel=self._chan, timeout_ms=self.timeout_ms)
        self._chan = (self._chan + 1) % 4

    def _shard(self, start: int, end: int, r: int) -> Tuple[int, int]:
        c = ((end - start + self.world - 1) // self.world + 3) // 4 * 4
        lo = min(start + r * c, end)
        return lo, min(lo + c, end)

    def _reduce(self, start: int, end: int) -> None:
        self._reduce_many([(start, end)])

    def _reduce_many(self, ranges: List[Tuple[int, int]]) -> None:
        """One barrier / pull / mean / barrier / pull round over one or several ranges of the buffer."""
        ranges = [(s, e) for s, e in ranges if e > s]
        if not ranges:
            return
        from . import ops
        flat = self.sym
        self.bytes_reduced += sum(e - s for s, e in ranges) * 4
        self.collectives += 1
        if self._after is not None:
            ready = self._after
        else:
            ready = torch.cuda.Event(enable_timing=self.timing is not None)
            ready.record(torch.cuda.current_stream())
        self.comm.wait_event(ready)
        marks = []

        def mark():
            if self.timing is not None:
                e = torch.cuda.Event(enable_timing=True)
                e.record(self.comm)
                marks.append(e)
        peers = sorted(self.peer_bufs)
        with torch.cuda.stream(self.comm):
            mark()
            self._barrier()                                           # every rank's copy of these ranges is complete
            mark()
            mine, off = [], 0
            for start, end in ranges:                                 # pull my shard of every range from every peer
                lo, hi = self._shard(start, end, self.rank)
                n = hi - lo
                if n <= 0:
                    continue
                if (len(peers) - 1) * self.max_shard + off + n > self.scratch.numel():
                    raise RuntimeError("PeerGradSync: scratch too small for this set of ranges")
                for i, p in enumerate(peers):
                    self.scratch[i * self.max_shard + off:i * self.max_shard + off + n].copy_(self.peer_bufs[p][lo:hi], non_blocking=True)
                mine.append((lo, n, off))
                off += n
            mark()
            for lo, n, o in mine:
                ops.shard_mean(flat[lo:lo + n], self.scratch[o:], self.max_shard, self.world - 1, 1.0 / self.world)
            mark()
            self._barrier()                                           # every owner has reduced its shards
            mark()
            for start, end in ranges:                                 # pull the other ranks' reduced shards
                for p in peers:
                    plo, phi = self._shard(start, end, p)
                    if phi > plo:
                        flat[plo:phi].copy_(self.peer_bufs[p][plo:phi], non_blocking=True)
            mark()
            self._last = torch.cuda.Event()
            self._last.record(self.comm)
        if self.timing is not None:
            self.timing.append((ranges[0][0], ranges[0][0] + sum(e - s for s, e in ranges), ready, marks))

    def rest_ready(self, after=None) -> None:
        self._after = after
        self._reduce_many(self._final_ranges())
        with torch.cuda.stream(self.comm):
            self._barrier()       # nobody may reuse (zero, overwrite) its gradient buffer while a peer still pulls from it
            self._last = torch.cuda.Event()
            self._last.record(self.comm)
        self.wait()

    def wait(self) -> None:
        if self._last is not None:
            torch.cuda.current_stream().wait_event(self._last)
            self._last = None


def broadcast_parameters(model, src: int = 0, process_group=None) -> None:
    """Identical replicas: rank ``src``'s flat fp32 parameters overwrite everyone else's."""
    if dist.is_initialized() and dist.get_world_size(process_group) > 1:
        dist.broadcast(model.flat_parameters(), src=src, group=process_group)
        model.invalidate_shadow()       # the bf16 GEMM weights must be re-derived from the received masters


def shard_batch(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous equal shards of a global batch (rank r owns images [r·n/world, (r+1)·n/world))."""
    if n % world:
        raise ValueError(f"global batch {n} is not divisible by world size {world}: the mean-loss gradient "
                         "average is only exact for equal shards")
    per = n // world
    return rank * per, (rank + 1) * per
