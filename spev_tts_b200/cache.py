"""Log-mel training-cache builder: the B200 replacement of the mel lines of the reference's
cache loop (``/root/reference/spev_real_metrics.py:330-426``; mel statements ``:363-367``,
stored layout ``'mel': mel.T`` ``:421``).

* ``shard_utterances``  -- length-balanced (greedy LPT) assignment of utterances to ranks.  The
  path is embarrassingly data-parallel: no collective runs inside or between kernels.
* ``build_logmel_cache`` -- host buffers in, host buffers out: chunked H2D copy / fused kernel /
  D2H copy on three streams with double buffering (this is the end-to-end path a caller with
  wavs in host memory uses; ``bench.py`` times it as ``e2e``).
* ``gather_shards``      -- the only cross-GPU step: variable-length gather of the ``[F_r, 80]``
  shards (NCCL on GPUs over NVLink; gloo in the CPU tests).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib, spectral
from .batch import HOP, Context, aligned_offsets, make_batch


# ---------------------------------------------------------------------------------------------
# host placement: pinned staging buffers should live on the NUMA node the GPU hangs off
# ---------------------------------------------------------------------------------------------
def _parse_cpulist(text: str):
    cpus = []
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.extend(range(int(a), int(b or a) + 1))
    return cpus


def bind_to_gpu_numa_node(device) -> dict:
    """Pin the calling process to the CPUs of the NUMA node that `device`'s PCIe root belongs to
    (Linux sysfs).  Call it BEFORE allocating pinned host buffers: first-touch then places them on
    that node, so that H2D/D2H copies of several ranks do not cross sockets.  Best effort: returns
    what it did and never raises."""
    import os
    info = {"bound": False}
    try:
        dev = torch.device(device)
        idx = dev.index if dev.index is not None else torch.cuda.current_device()
        props = torch.cuda.get_device_properties(idx)
        bdf = f"{props.pci_domain_id:04x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        info.update(pci=bdf, numa_node=node)
        if node < 0:
            return info
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set(_parse_cpulist(f.read())) & set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            info.update(bound=True, n_cpus=len(cpus))
    except Exception as e:   # sysfs layout / permissions differ: keep going unbound
        info["error"] = repr(e)
    return info


# ---------------------------------------------------------------------------------------------
# sharding (host logic; CPU-testable)
# ---------------------------------------------------------------------------------------------
def frames_of(n_samples) -> np.ndarray:
    return 1 + np.asarray(n_samples, dtype=np.int64) // HOP


def shard_utterances(n_samples: Sequence[int], world_size: int) -> List[np.ndarray]:
    """Greedy longest-processing-time assignment balancing the number of frames per rank.
    Returns, per rank, the sorted utterance indices it owns.  Deterministic."""
    fr = frames_of(n_samples)
    order = np.argsort(-fr, kind="stable")
    loads = np.zeros(world_size, dtype=np.int64)
    owner = np.empty(len(fr), dtype=np.int64)
    for i in order:
        r = int(np.argmin(loads))
        owner[i] = r
        loads[r] += fr[i]
    return [np.sort(np.nonzero(owner == r)[0]) for r in range(world_size)]


@dataclass
class CachePlan:
    """Chunks of consecutive utterances sized to ~``chunk_samples`` samples."""
    n_samples: np.ndarray
    sample_off: np.ndarray      # [U+1] item starts in the host buffer (last = end of buffer)
    frame_off: np.ndarray       # [U+1]
    chunks: List[Tuple[int, int]]   # (first utt, last utt exclusive)


def plan_chunks(n_samples: Sequence[int], chunk_samples: int = 1 << 26,
                sample_off: Optional[np.ndarray] = None) -> CachePlan:
    ns = np.asarray(n_samples, dtype=np.int64)
    so = np.concatenate([[0], np.cumsum(ns)]) if sample_off is None else np.asarray(sample_off, dtype=np.int64)
    assert so.shape == (len(ns) + 1,) and np.all(so[1:] - so[:-1] >= ns)
    fo = np.concatenate([[0], np.cumsum(frames_of(ns))])
    chunks, a = [], 0
    while a < len(ns):
        b = int(np.searchsorted(so, so[a] + chunk_samples, side="right")) - 1
        b = max(b, a + 1)
        b = min(b, len(ns))
        chunks.append((a, b))
        a = b
    return CachePlan(ns, so, fo, chunks)


# ---------------------------------------------------------------------------------------------
# end-to-end builder: pinned host -> device -> pinned host, pipelined
# ---------------------------------------------------------------------------------------------
class LogMelCacheBuilder:
    """Reusable pipelined builder (device staging buffers and streams are allocated once)."""

    def __init__(self, device, *, sr=22050, n_mels=80, chunk_samples: int = 1 << 26, n_buffers: int = 2):
        self.device = torch.device(device)
        self.sr, self.n_mels = sr, n_mels
        self.chunk_samples = chunk_samples
        self.n_buffers = n_buffers
        self.ctx = Context.get(self.device, sr=sr, n_mels=n_mels)
        self.copy_in = torch.cuda.Stream(self.device)
        self.compute = torch.cuda.Stream(self.device)
        self.copy_out = torch.cuda.Stream(self.device)
        self._pcm: List[Optional[torch.Tensor]] = [None] * n_buffers
        self._in: List[Optional[torch.Tensor]] = [None] * n_buffers
        self._out: List[Optional[torch.Tensor]] = [None] * n_buffers
        # per-buffer "free again" events live across build() calls: a second build() enqueued without a host
        # synchronise must not start copying into a staging buffer the previous build's kernels still read
        self._in_free: List[Optional[torch.cuda.Event]] = [None] * n_buffers    # compute finished reading buffer i
        self._out_free: List[Optional[torch.cuda.Event]] = [None] * n_buffers   # D2H finished reading buffer i
        self.launches = 0

    def _buf(self, pool, i, n, dtype=torch.float32):
        if pool[i] is None or pool[i].numel() < n:
            pool[i] = torch.empty(max(n, 1), dtype=dtype, device=self.device)
        return pool[i]

    def build(self, samples_host: torch.Tensor, n_samples: Sequence[int],
              out_host: Optional[torch.Tensor] = None, plan: Optional[CachePlan] = None,
              sample_off: Optional[np.ndarray] = None):
        """``samples_host``: flat host tensor (pinned for full copy speed) holding the utterances at
        ``sample_off`` (default: packed back to back; ``aligned_offsets`` gives the fast layout),
        either float32 or **int16 PCM** (shipped as 2 bytes/sample and widened to ``pcm/32768`` on the
        device -- the exact values a 16-bit wav decodes to); returns ``(out_host [F, n_mels] pinned,
        frame_off)``."""
        pcm = samples_host.dtype == torch.int16
        if not pcm and samples_host.dtype != torch.float32:
            raise ValueError("samples_host must be float32 or int16 PCM")
        if plan is None:
            plan = plan_chunks(n_samples, self.chunk_samples, sample_off)
        F = int(plan.frame_off[-1])
        if out_host is None:
            out_host = torch.empty((F, self.n_mels), dtype=torch.float32).pin_memory()
        nb = self.n_buffers
        in_free, out_free = self._in_free, self._out_free
        max_in = max(int(plan.sample_off[b] - plan.sample_off[a]) for a, b in plan.chunks)
        max_out = max(int(plan.frame_off[b] - plan.frame_off[a]) for a, b in plan.chunks) * self.n_mels
        for i in range(nb):
            self._buf(self._in, i, max_in)
            self._buf(self._out, i, max_out)
            if pcm:
                self._buf(self._pcm, i, max_in, torch.int16)
        # descriptors are tiny; build them all up front so the loop only enqueues
        batches = [make_batch(self.ctx, n_samples=plan.n_samples[a:b],
                              sample_off=plan.sample_off[a:b] - plan.sample_off[a]) for a, b in plan.chunks]
        tables_up = torch.cuda.Event()
        tables_up.record(torch.cuda.current_stream(self.device))   # descriptor uploads and staging allocations ran here
        self.compute.wait_event(tables_up)
        self.copy_in.wait_event(tables_up)                         # (a re-used allocation may still be in use upstream)
        self.copy_out.wait_event(tables_up)
        for ci, (a, b) in enumerate(plan.chunks):
            i = ci % nb
            s0, s1 = int(plan.sample_off[a]), int(plan.sample_off[b])
            f0, f1 = int(plan.frame_off[a]), int(plan.frame_off[b])
            d_in = self._in[i][: s1 - s0]
            d_out = self._out[i][: (f1 - f0) * self.n_mels].view(f1 - f0, self.n_mels)
            with torch.cuda.stream(self.copy_in):
                if in_free[i] is not None:          # also set by a previous build()
                    self.copy_in.wait_event(in_free[i])
                (self._pcm[i][: s1 - s0] if pcm else d_in).copy_(samples_host[s0:s1], non_blocking=True)
                ready = torch.cuda.Event()
                ready.record(self.copy_in)
            with torch.cuda.stream(self.compute):
                self.compute.wait_event(ready)
                if out_free[i] is not None:
                    self.compute.wait_event(out_free[i])
                if pcm:
                    _lib.check(self.ctx.lib.spev_pcm16_to_f32(self._pcm[i].data_ptr(), s1 - s0, d_in.data_ptr(),
                                                              self.compute.cuda_stream), "spev_pcm16_to_f32")
                    self.launches += 1
                spectral.logmel_flat(d_in, plan.n_samples[a:b], sr=self.sr, n_mels=self.n_mels,
                                     out=d_out, batch=batches[ci])
                self.launches += 1
                in_free[i] = torch.cuda.Event()
                in_free[i].record(self.compute)
                done = torch.cuda.Event()
                done.record(self.compute)
            with torch.cuda.stream(self.copy_out):
                self.copy_out.wait_event(done)
                out_host[f0:f1].copy_(d_out, non_blocking=True)
                out_free[i] = torch.cuda.Event()
                out_free[i].record(self.copy_out)
        fin = torch.cuda.Event()
        fin.record(self.copy_out)
        torch.cuda.current_stream(self.device).wait_event(fin)
        self._keep = batches
        return out_host, plan.frame_off


def build_logmel_cache(samples_host: torch.Tensor, n_samples: Sequence[int], device=None,
                       sample_off: Optional[np.ndarray] = None, **kw):
    """One-shot convenience wrapper around ``LogMelCacheBuilder`` (synchronises before returning)."""
    device = spectral.default_device() if device is None else torch.device(device)
    out, fo = LogMelCacheBuilder(device, **kw).build(samples_host, n_samples, sample_off=sample_off)
    torch.cuda.synchronize(device)
    return out, fo


# ---------------------------------------------------------------------------------------------
# the one cross-rank step: gather the shards
# ---------------------------------------------------------------------------------------------
def gather_shards(local: torch.Tensor, dst: int = 0, group=None):
    """Variable-length gather of ``[F_r, n_mels]`` shards to rank ``dst``.
    Returns ``(list of per-rank tensors on dst | None elsewhere, frames_per_rank)``.
    Uses an all_gather of the row counts followed by point-to-point transfers (NCCL has no
    gatherv); works on the NCCL (GPU, NVLink) and gloo (CPU tests) backends."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    n = torch.tensor([local.shape[0]], dtype=torch.int64, device=local.device)
    counts = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(counts, n, group=group)
    counts = [int(c.item()) for c in counts]
    if rank == dst:
        parts = [local if r == dst else torch.empty((counts[r], local.shape[1]), dtype=local.dtype,
                                                    device=local.device) for r in range(world)]
        ops = [dist.P2POp(dist.irecv, parts[r], r, group) for r in range(world) if r != dst and counts[r]]
        if ops:
            for q in dist.batch_isend_irecv(ops):   # one grouped NCCL launch: transfers run concurrently
                q.wait()
        return parts, counts
    if local.shape[0]:
        for q in dist.batch_isend_irecv([dist.P2POp(dist.isend, local.contiguous(), dst, group)]):
            q.wait()
    return None, counts


def copy_segments(src: torch.Tensor, dst: torch.Tensor, src_row, dst_row, n_rows) -> None:
    """``dst[dst_row[i] : dst_row[i] + n_rows[i]] = src[src_row[i] : src_row[i] + n_rows[i]]`` for runs of rows of two
    row-major 2-D CUDA tensors with equal row size, in one launch (``spev_copy_segments``)."""
    if not (src.is_cuda and dst.is_cuda and src.is_contiguous() and dst.is_contiguous()):
        raise RuntimeError("copy_segments needs contiguous CUDA tensors (no CPU path)")
    rb = src.shape[1] * src.element_size()
    if rb != dst.shape[1] * dst.element_size():
        raise ValueError("row sizes differ")
    n_rows = np.asarray(n_rows, dtype=np.int64)
    keep = n_rows > 0
    nb = n_rows[keep] * rb
    if nb.size == 0:
        return
    lib = _lib.load()
    piece = lib.spev_copy_segments_piece_bytes()
    npieces = (nb + piece - 1) // piece
    poff = np.cumsum(npieces) - npieces
    table = np.stack([np.asarray(src_row, dtype=np.int64)[keep] * rb, np.asarray(dst_row, dtype=np.int64)[keep] * rb, nb, poff])
    t = torch.from_numpy(np.ascontiguousarray(table)).pin_memory().to(src.device, non_blocking=True)
    n = int(nb.size)
    with torch.cuda.device(src.device):
        _lib.check(lib.spev_copy_segments(src.data_ptr(), dst.data_ptr(), t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(),
                                          t[3].data_ptr(), n, int(npieces.sum()),
                                          torch.cuda.current_stream(src.device).cuda_stream), "spev_copy_segments")
    t.record_stream(torch.cuda.current_stream(src.device))


def assemble(parts: Sequence[torch.Tensor], shards: Sequence[np.ndarray], n_samples: Sequence[int]):
    """Re-order gathered shards into corpus order.  Returns ``(cache [F, n_mels], frame_off)``
    such that utterance ``u`` is ``cache[frame_off[u]:frame_off[u+1]]`` -- i.e. the tensor each
    ``cache_stable/u_%05d.pt`` would hold under ``'mel'`` (``spev_real_metrics.py:419-425``)."""
    fr = frames_of(n_samples)
    fo = np.concatenate([[0], np.cumsum(fr)])
    out = torch.empty((int(fo[-1]), parts[0].shape[1]), dtype=parts[0].dtype, device=parts[0].device)
    for part, idx in zip(parts, shards):
        if len(idx) == 0:
            continue
        loc = np.concatenate([[0], np.cumsum(fr[idx])])
        if out.is_cuda:      # one row-run copy per utterance, all in one launch
            copy_segments(part.contiguous(), out, loc[:-1], fo[idx], fr[idx])
        else:                # host tensors (the gloo tests of the host logic): plain slice copies
            for k, u in enumerate(idx):
                out[fo[u]: fo[u + 1]] = part[loc[k]: loc[k + 1]]
    return out, fo


# ---------------------------------------------------------------------------------------------
# the multi-GPU cache build as one pipelined step: shard -> fused kernel per chunk -> gather
# ---------------------------------------------------------------------------------------------
@dataclass
class ShardPlan:
    """Everything every rank can compute on its own from the corpus' utterance lengths: who owns which utterance,
    where each rank's rows land in the gathered (rank-major) cache, and how each shard is cut into chunks for the
    compute/gather overlap.  No metadata exchange is needed at run time."""
    world: int
    n_samples: np.ndarray            # [U]
    frames: np.ndarray               # [U]
    shards: List[np.ndarray]         # per rank: sorted utterance indices
    row_off: np.ndarray              # [world+1] first row of each rank's block in the gathered cache
    utt_row: np.ndarray              # [U] first row of utterance u in the gathered cache
    chunks: List[List[Tuple[int, int]]]   # per rank: (first, last-exclusive) LOCAL utterance positions per chunk

    def chunk_rows(self, rank: int, k: int) -> Tuple[int, int]:
        """absolute rows [lo, hi) of chunk k of `rank` in the gathered cache"""
        a, b = self.chunks[rank][k]
        idx = self.shards[rank]
        lo = int(self.row_off[rank] + self.frames[idx[:a]].sum())
        return lo, lo + int(self.frames[idx[a:b]].sum())

    @property
    def n_rows(self) -> int:
        return int(self.row_off[-1])


def plan_shards(n_samples: Sequence[int], world: int, n_chunks: int = 4) -> ShardPlan:
    ns = np.asarray(n_samples, dtype=np.int64)
    fr = frames_of(ns)
    shards = shard_utterances(ns, world)
    per_rank = np.array([int(fr[s].sum()) for s in shards], dtype=np.int64)
    row_off = np.concatenate([[0], np.cumsum(per_rank)]).astype(np.int64)
    utt_row = np.empty(len(ns), dtype=np.int64)
    chunks = []
    for r, idx in enumerate(shards):
        loc = np.concatenate([[0], np.cumsum(fr[idx])])
        utt_row[idx] = row_off[r] + loc[:-1]
        k = max(1, min(n_chunks, len(idx)))
        cuts = [int(np.searchsorted(loc, loc[-1] * j / k, side="left")) for j in range(k + 1)]
        cuts[0], cuts[-1] = 0, len(idx)
        chunks.append([(a, b) for a, b in zip(cuts[:-1], cuts[1:]) if b > a] or [(0, len(idx))])
    return ShardPlan(world, ns, fr, shards, row_off, utt_row, chunks)


class GatheredCache:
    """The gathered log-mel cache on the root: one ``[F, n_mels]`` buffer in rank-major row order plus the row of
    every utterance.  ``utterance(u)`` is the tensor ``cache_stable/u_%05d.pt`` holds under ``'mel'``
    (``spev_real_metrics.py:419-425``) as a zero-copy view; ``corpus_order()`` re-packs once (one launch)."""

    def __init__(self, buf: torch.Tensor, plan: ShardPlan):
        self.buf, self.plan = buf, plan

    def utterance(self, u: int) -> torch.Tensor:
        r0 = int(self.plan.utt_row[u])
        return self.buf[r0: r0 + int(self.plan.frames[u])]

    def corpus_order(self):
        fr = self.plan.frames
        fo = np.concatenate([[0], np.cumsum(fr)])
        out = torch.empty_like(self.buf)
        copy_segments(self.buf, out, self.plan.utt_row, fo[:-1], fr)
        return out, fo


class ShardedCacheBuilder:
    """One rank of the utterance-sharded cache build (one process per GPU).  ``build()`` is the whole multi-GPU step:
    this rank's fused STFT->log-mel kernel over its shard, and the gather of all shards into the root's cache --
    the only cross-GPU exchange of the path (NCCL send/recv over NVLink; gloo in the CPU tests).

    ``overlap=True`` cuts every shard into ``plan``'s chunks: the root posts all receives up front (they land
    directly in their final rows -- no staging, no re-ordering pass) and every rank sends chunk k while its kernel
    works on chunk k+1.  The FFT kernels fill whole SMs, so ``reserve_sms`` CTAs are left to NCCL's kernels while a
    transfer is in flight (``spev_set_sm_limit``)."""

    def __init__(self, plan: ShardPlan, rank: int, device, *, dst: int = 0, group=None, sr=22050, n_mels=80,
                 reserve_sms: int = 16, kernel=None, transport: str = "nccl"):
        """``transport``: ``"nccl"`` -- grouped ncclSend/ncclRecv (the default; NCCL's kernels need SMs, see
        ``reserve_sms``) -- or ``"p2p"`` -- the root's cache is a symmetric-memory window mapped into every rank
        (``torch.distributed._symmetric_memory``) and each rank pushes its finished chunks into their final rows with
        copy-engine ``cudaMemcpyAsync`` over NVLink: no SM is taken from the FFT kernels, and a stream-ordered
        signal-pad barrier closes the step.
        ``kernel(samples, out_rows, a, b)``: test hook replacing the CUDA kernel for the local utterances [a, b)
        (the gloo tests of the host logic); the product always runs ``spev_logmel``."""
        if transport not in ("nccl", "p2p"):
            raise ValueError("transport must be 'nccl' or 'p2p'")
        self.transport = transport
        self._window = self._root_view = self._copy_stream = None
        self.plan, self.rank, self.dst, self.group = plan, rank, dst, group
        self.device = torch.device(device)
        self.sr, self.n_mels = sr, n_mels
        self.reserve_sms = reserve_sms
        idx = plan.shards[rank]
        self.lens = plan.n_samples[idx]
        self.sample_off = aligned_offsets(self.lens)
        self.n_rows_local = int(plan.frames[idx].sum())
        self._kernel_hook = kernel
        self.launches = 0
        if kernel is not None:
            self.ctx = None
            return
        # a PRIVATE context: build() changes its SM limit while transfers are in flight, which must not leak into the
        # shared per-device context other callers (threads) get from Context.get
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.ctx = Context(idx, sr, 1024, HOP, 1024, n_mels, 0.0, None)
        self.batch_all = make_batch(self.ctx, n_samples=self.lens, sample_off=self.sample_off)
        self.batch_chunk = [make_batch(self.ctx, n_samples=self.lens[a:b], sample_off=self.sample_off[a:b])
                            for a, b in plan.chunks[rank]]

    # -- layout helpers -------------------------------------------------------------------------
    def alloc_out(self) -> torch.Tensor:
        """root: the gathered cache ``[F_total, n_mels]``; other ranks: their shard ``[F_r, n_mels]``.  With the p2p
        transport every rank holds a full-size symmetric window (rows outside its shard stay unused off the root)."""
        if self.transport == "p2p" and self.plan.world > 1:
            import torch.distributed as dist
            import torch.distributed._symmetric_memory as symm
            try:
                buf = symm.empty((self.plan.n_rows, self.n_mels), dtype=torch.float32, device=self.device)
                self._window = symm.rendezvous(buf, self.group if self.group is not None else dist.group.WORLD)
                self._root_view = self._window.get_buffer(self.dst, (self.plan.n_rows, self.n_mels), torch.float32)
            except Exception as e:     # no silent change of transport: the caller decides
                raise RuntimeError(f"p2p transport unavailable (symmetric-memory rendezvous failed: {e!r})") from e
            self._copy_stream = torch.cuda.Stream(self.device)
            return buf
        rows = self.plan.n_rows if self.rank == self.dst else self.n_rows_local
        return torch.empty((rows, self.n_mels), dtype=torch.float32, device=self.device)

    def local_rows(self, out: torch.Tensor, k: Optional[int] = None) -> torch.Tensor:
        full = self.rank == self.dst or self._window is not None
        base = int(self.plan.row_off[self.rank]) if full else 0
        if k is None:
            return out[base: base + self.n_rows_local]
        lo, hi = self.plan.chunk_rows(self.rank, k)
        off = int(self.plan.row_off[self.rank]) - base
        return out[lo - off: hi - off]

    def _kernel(self, samples: torch.Tensor, out_rows: torch.Tensor, k: Optional[int]) -> None:
        self.launches += 1
        if self._kernel_hook is not None:
            a, b = (0, len(self.lens)) if k is None else self.plan.chunks[self.rank][k]
            self._kernel_hook(samples, out_rows, a, b)
            return
        batch = self.batch_all if k is None else self.batch_chunk[k]
        _lib.check(self.ctx.lib.spev_logmel(self.ctx.handle, batch.desc, samples.data_ptr(), out_rows.data_ptr(), 1,
                                            spectral.REF_LOG_FLOOR, spectral.REF_LOG_LO, spectral.REF_LOG_HI,
                                            torch.cuda.current_stream(self.device).cuda_stream), "spev_logmel")

    def _limit(self, on: bool) -> None:
        if self.ctx is None:
            return
        _lib.check(self.ctx.lib.spev_set_sm_limit(self.ctx.handle, max(1, self._sms() - self.reserve_sms) if on else 0),
                   "spev_set_sm_limit")

    def _sms(self) -> int:
        return torch.cuda.get_device_properties(self.device).multi_processor_count

    # -- the step ---------------------------------------------------------------------------------
    def build(self, samples: torch.Tensor, out: torch.Tensor, *, gather: bool = True, overlap: bool = True):
        """``samples``: this rank's shard, utterances at ``self.sample_off`` (device float32).  Enqueues everything on
        the current stream (plus NCCL's own stream) and returns without a host synchronisation; afterwards the root's
        ``out`` holds every rank's rows (``GatheredCache(out, plan)``)."""
        import torch.distributed as dist
        plan, rank, dst = self.plan, self.rank, self.dst
        if not gather or plan.world == 1:
            self._kernel(samples, self.local_rows(out), None)
            return out
        peers = [r for r in range(plan.world) if r != dst]
        if self._window is not None:
            return self._build_p2p(samples, out, overlap)
        if not overlap:
            self._kernel(samples, self.local_rows(out), None)
            if rank == dst:
                ops = [dist.P2POp(dist.irecv, out[int(plan.row_off[r]): int(plan.row_off[r + 1])], r, self.group)
                       for r in peers if plan.row_off[r + 1] > plan.row_off[r]]
            else:
                ops = [dist.P2POp(dist.isend, self.local_rows(out), dst, self.group)] if self.n_rows_local else []
            for w in (dist.batch_isend_irecv(ops) if ops else []):
                w.wait()
            return out
        works = []
        self._limit(True)
        try:
            if rank == dst:
                kmax = max(len(plan.chunks[r]) for r in peers)
                for k in range(kmax):             # all receives first: chunk k of every peer is one grouped launch
                    ops = []
                    for r in peers:
                        if k < len(plan.chunks[r]):
                            lo, hi = plan.chunk_rows(r, k)
                            if hi > lo:
                                ops.append(dist.P2POp(dist.irecv, out[lo:hi], r, self.group))
                    if ops:
                        works += dist.batch_isend_irecv(ops)
                for k in range(len(plan.chunks[rank])):
                    self._kernel(samples, self.local_rows(out, k), k)
            else:
                for k in range(len(plan.chunks[rank])):
                    rows = self.local_rows(out, k)
                    self._kernel(samples, rows, k)
                    if rows.shape[0]:
                        works += dist.batch_isend_irecv([dist.P2POp(dist.isend, rows, dst, self.group)])
        finally:
            self._limit(False)
        for w in works:
            w.wait()                              # stream-level join (non-blocking on the host for NCCL)
        return out

    def _build_p2p(self, samples: torch.Tensor, out: torch.Tensor, overlap: bool):
        """Copy-engine transport: chunk k is pushed into the root's window (its final rows) on a side stream while the
        kernel of chunk k+1 runs on all SMs; a signal-pad barrier (stream-ordered, no host sync) ends the step."""
        plan, rank = self.plan, self.rank
        cur = torch.cuda.current_stream(self.device)
        # The FFT CTAs fill whole SMs; one SM is left free so that the (single-CTA) barrier kernels below can run
        # beside them instead of queueing behind a whole shard.
        _lib.check(self.ctx.lib.spev_set_sm_limit(self.ctx.handle, max(1, self._sms() - 1)), "spev_set_sm_limit") \
            if self.ctx is not None else None
        # The window is one-sided: nothing may land in it before the root's earlier work on it (a consumer of the
        # previous step's cache, a fill) has finished.  The root arrives at this barrier on ITS stream, i.e. after that
        # work; the other ranks wait for it on their copy stream only, so their kernels start at once.
        if rank == self.dst:
            self._window.barrier(channel=1)
        else:
            with torch.cuda.stream(self._copy_stream):
                self._copy_stream.wait_stream(cur)
                self._window.barrier(channel=1)
        ks = range(len(plan.chunks[rank])) if overlap else [None]
        for k in ks:
            rows = self.local_rows(out, k)
            self._kernel(samples, rows, k)
            if rank != self.dst and rows.shape[0]:
                if k is None:
                    lo, hi = int(plan.row_off[rank]), int(plan.row_off[rank + 1])
                else:
                    lo, hi = plan.chunk_rows(rank, k)
                ev = torch.cuda.Event()
                ev.record(cur)
                with torch.cuda.stream(self._copy_stream):
                    self._copy_stream.wait_event(ev)
                    self._root_view[lo:hi].copy_(rows, non_blocking=True)
        cur.wait_stream(self._copy_stream)
        self._window.barrier(channel=0)           # every rank's pushes are complete and visible on the root
        self._limit(False)
        return out
