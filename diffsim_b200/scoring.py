"""Batched scoring on top of the C ABI: Q/K/V caches, triplet / pair scoring with host or device inputs,
all-pairs retrieval matrices and their row-block sharding across ranks.

This is the layer the benchmark drivers of the reference would call once per BATCH instead of once per pair
(cute_main.py:111-132 calls DiffSim.diffsim twice per triplet and syncs on every comparison, :196-205).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import torch

from . import ops


@dataclass
class QKVCache:
    """Q, K, V of N images as (N,B,H,S,D) views over (N,B,S,H*D) memory -- the reference's per-image layout
    (diffsim/hacked_attn.py:74-77) with an image axis in front.  What DiffSim.diffsim_value returns per image
    (diffsim/diffsim.py:201-258), stacked."""

    q: torch.Tensor
    k: torch.Tensor
    v: torch.Tensor

    @property
    def n_images(self) -> int:
        return self.q.shape[0]

    @property
    def shape(self) -> Tuple[int, int, int, int]:
        return tuple(self.q.shape[1:])

    @property
    def bytes_per_image(self) -> int:
        B, H, S, D = self.shape
        return 3 * B * H * S * D * self.q.element_size()

    @staticmethod
    def empty(n: int, B: int, H: int, S: int, D: int, dtype=torch.float16, device="cuda", pin: bool = False) -> "QKVCache":
        def mk():
            mem = torch.empty((n, B, S, H * D), dtype=dtype, device=device, pin_memory=pin)
            return mem.view(n, B, S, H, D).permute(0, 1, 3, 2, 4)

        return QKVCache(mk(), mk(), mk())

    @staticmethod
    def from_images(images: Sequence[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]], device=None) -> "QKVCache":
        from .synth import stack_cache

        return QKVCache(*stack_cache(images, device))

    def memory(self) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """The underlying (N,B,S,H*D) buffers (contiguous), for copies and collectives."""
        def mem(t):
            n, B, H, S, D = t.shape
            return t.permute(0, 1, 3, 2, 4).reshape(n, B, S, H * D)

        return mem(self.q), mem(self.k), mem(self.v)

    def slice(self, i0: int, i1: int) -> "QKVCache":
        return QKVCache(self.q[i0:i1], self.k[i0:i1], self.v[i0:i1])

    def to(self, device, non_blocking: bool = False) -> "QKVCache":
        outs = []
        for m, t in zip(self.memory(), (self.q, self.k, self.v)):
            n, B, H, S, D = t.shape
            d = m.to(device, non_blocking=non_blocking)
            outs.append(d.view(n, B, S, H, D).permute(0, 1, 3, 2, 4))
        return QKVCache(*outs)


def score_pairs(cache: QKVCache, pairs, similarity: str = "cosine", scale: Optional[float] = None) -> torch.Tensor:
    """DiffSim.diffsim for every (a,b) in pairs (diffsim/diffsim.py:177-197).  float32 [P] on the device."""
    return ops.aas_pairs(cache.q, cache.k, cache.v, pairs, similarity, scale)


def score_triplets(cache: QKVCache, triplets, similarity: str = "cosine", scale: Optional[float] = None,
                   round_scores: bool = False):
    """(ab, ac, counts, flags) for 2AFC triplets (ref, left, right); see ops.aas_triplets."""
    return ops.aas_triplets(cache.q, cache.k, cache.v, triplets, similarity, scale, round_scores)


class HostTripletScorer:
    """End-to-end scorer for HOST-resident Q/K/V: pinned host buffers -> chunked, double-buffered H2D copies
    on a copy stream overlapped with the fused kernels on the compute stream -> decision counts back on the host.

    Triplet t uses images (3t, 3t+1, 3t+2) of the host cache (reference, left, right).
    """

    def __init__(self, shape: Tuple[int, int, int, int], dtype=torch.float16, device="cuda", chunk_triplets: int = 96,
                 similarity: str = "cosine"):
        self.shape, self.dtype, self.device = shape, dtype, torch.device(device)
        self.chunk = chunk_triplets
        self.similarity = similarity
        B, H, S, D = shape
        self.bufs = [QKVCache.empty(3 * chunk_triplets, B, H, S, D, dtype, device) for _ in range(2)]
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.copied = [torch.cuda.Event() for _ in range(2)]
        self.consumed = [torch.cuda.Event() for _ in range(2)]
        self.trips = torch.arange(3 * chunk_triplets, dtype=torch.int32, device=device).view(-1, 3)
        self.h2d_bytes = 0
        self.d2h_bytes = 0

    def score(self, host: QKVCache, n_triplets: int):
        """Returns (correct, correct_2x) as Python ints (one device->host read at the end)."""
        dev = self.device
        compute = torch.cuda.current_stream(dev)
        hm = host.memory()
        totals = torch.zeros(2, dtype=torch.int32, device=dev)
        n_chunks = (n_triplets + self.chunk - 1) // self.chunk
        for c in range(n_chunks):
            t0, t1 = c * self.chunk, min(n_triplets, (c + 1) * self.chunk)
            nb = c % 2
            buf = self.bufs[nb]
            with torch.cuda.stream(self.copy_stream):
                if c >= 2:
                    self.copy_stream.wait_event(self.consumed[nb])
                for src, dst in zip(hm, buf.memory()):
                    dst[: 3 * (t1 - t0)].copy_(src[3 * t0: 3 * t1], non_blocking=True)
                    self.h2d_bytes += src[3 * t0: 3 * t1].numel() * src.element_size()
                self.copied[nb].record(self.copy_stream)
            compute.wait_event(self.copied[nb])
            _, _, counts, _ = ops.aas_triplets(buf.q, buf.k, buf.v, self.trips[: t1 - t0], self.similarity,
                                               want_flags=False)
            totals += counts
            self.consumed[nb].record(compute)
        out = totals.cpu()  # the step's result read: device -> host
        self.d2h_bytes += out.numel() * out.element_size()
        return int(out[0]), int(out[1])


def project_cache(hidden: torch.Tensor, weight: torch.Tensor, heads: int, bias: Optional[torch.Tensor] = None,
                  out: Optional[QKVCache] = None) -> QKVCache:
    """Hook inputs -> Q/K/V cache: hidden (N,B,S,C) x [W_q; W_k; W_v] (3C', C) -> three (N,B,H,S,D) views over
    (N,B,S,C') memory, the capture step of the reference (diffsim/hacked_attn.py:61-69,74-77) for N images in one
    tcgen05 GEMM (ops.qkv_project).  `out`: a cache to fill (its first N images)."""
    n, B, S, _ = hidden.shape
    c_out = weight.shape[0] // 3
    D = c_out // heads
    if out is None:
        out = QKVCache.empty(n, B, heads, S, D, hidden.dtype, hidden.device)
    mems = [m[:n] for m in out.memory()]
    ops.qkv_project(hidden, weight, bias, 3, out=mems)
    return out.slice(0, n) if out.n_images != n else out


class HostHiddenTripletScorer:
    """End-to-end scorer at the HOOK-INPUT boundary: pinned host hidden states of the target attention layer
    (what `register_forward_pre_hook` hands the reference's hook, diffsim/diffsim.py:43-56) -> chunked,
    double-buffered H2D copies on a copy stream -> QKV projection (K4) + fused AAS scoring (K1) on the compute
    stream -> decision counts back on the host.  A third of the bytes of HostTripletScorer's Q/K/V boundary.

    Triplet t uses images (3t, 3t+1, 3t+2) of the host buffer (reference, left, right)."""

    def __init__(self, shape: Tuple[int, int, int, int], weight: torch.Tensor, bias: Optional[torch.Tensor] = None,
                 dtype=torch.float16, device="cuda", chunk_triplets: int = 96, similarity: str = "cosine"):
        self.shape, self.dtype, self.device = shape, dtype, torch.device(device)
        self.chunk = chunk_triplets
        self.similarity = similarity
        self.weight, self.bias = weight, bias
        B, H, S, D = shape
        c_in = weight.shape[1]
        self.hid = [torch.empty(3 * chunk_triplets, B, S, c_in, dtype=dtype, device=device) for _ in range(2)]
        self.cache = QKVCache.empty(3 * chunk_triplets, B, H, S, D, dtype, device)
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.copied = [torch.cuda.Event() for _ in range(2)]
        self.consumed = [torch.cuda.Event() for _ in range(2)]
        self.trips = torch.arange(3 * chunk_triplets, dtype=torch.int32, device=device).view(-1, 3)
        self.h2d_bytes = 0
        self.d2h_bytes = 0

    def score(self, host_hidden: torch.Tensor, n_triplets: int):
        """host_hidden: (>= 3 n_triplets, B, S, C) pinned host tensor.  Returns (correct, correct_2x) as Python ints
        (one device->host read at the end)."""
        dev = self.device
        H = self.shape[1]
        compute = torch.cuda.current_stream(dev)
        totals = torch.zeros(2, dtype=torch.int32, device=dev)
        n_chunks = (n_triplets + self.chunk - 1) // self.chunk
        for c in range(n_chunks):
            t0, t1 = c * self.chunk, min(n_triplets, (c + 1) * self.chunk)
            nb = c % 2
            n_img = 3 * (t1 - t0)
            with torch.cuda.stream(self.copy_stream):
                if c >= 2:
                    self.copy_stream.wait_event(self.consumed[nb])
                src = host_hidden[3 * t0: 3 * t1]
                self.hid[nb][:n_img].copy_(src, non_blocking=True)
                self.h2d_bytes += src.numel() * src.element_size()
                self.copied[nb].record(self.copy_stream)
            compute.wait_event(self.copied[nb])
            cache = project_cache(self.hid[nb][:n_img], self.weight, H, self.bias, out=self.cache)
            self.consumed[nb].record(compute)   # the hidden-state buffer is free once the projection has read it
            _, _, counts, _ = ops.aas_triplets(cache.q, cache.k, cache.v, self.trips[: t1 - t0], self.similarity,
                                               want_flags=False)
            totals += counts
        out = totals.cpu()  # the step's result read: device -> host
        self.d2h_bytes += out.numel() * out.element_size()
        return int(out[0]), int(out[1])


# --------------------------------------------------------------------------------------------------------
# all-pairs retrieval
# --------------------------------------------------------------------------------------------------------
def row_block(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous row block [r0, r1) of rank `rank` when n rows are split over `world` ranks."""
    base, rem = divmod(n, world)
    r0 = rank * base + min(rank, rem)
    return r0, r0 + base + (1 if rank < rem else 0)


def aas_matrix_local(rows: QKVCache, cols: QKVCache, similarity: str = "cosine", scale: Optional[float] = None):
    """Directional block Dm[rows, all columns] on this device; differentiable in the caches (ops.aas_matrix) when one
    of them requires grad."""
    return ops.aas_matrix(rows.q, rows.k, rows.v, cols.k, cols.v, similarity, scale)


@torch.no_grad()
def aas_matrix_sharded(local: QKVCache, similarity: str = "cosine", scale: Optional[float] = None, group=None,
                       gather_to_all: bool = True, timings: Optional[dict] = None) -> torch.Tensor:
    """All-pairs directional matrix with the images row-block sharded over the ranks of `group`.

    Each rank holds the Q/K/V of its own images.  K and V are exchanged with one all_gather each (NCCL over
    NVLink on GPUs, gloo on CPU tests), issued asynchronously: while they are in flight the rank already scores its
    rows against its OWN columns; the columns of every peer follow, one kernel call per peer, reading the gathered
    buffer in place (no concatenation copy).  Q and the self attention stay local.  Every rank computes
    Dm[own rows, :] and the row blocks are gathered at the end.  Per-element arithmetic does not depend on the
    sharding or on how the columns are cut into calls, so the result is bit-identical to the single-device matrix.
    `timings` (optional dict) receives CUDA events: 'start', 'own_done', 'exchange_done', 'block_done', 'end'.
    Forward only: the peers' K and V arrive through all_gather, so a graph built here would silently lack their
    gradients; the blocks run without one.
    """
    import torch.distributed as dist

    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    _, km, vm = local.memory()
    dev = km.device
    B, H, S, D = local.shape
    n_local = torch.tensor([km.shape[0]], dtype=torch.int64, device=dev)
    counts = [torch.zeros_like(n_local) for _ in range(world)]
    dist.all_gather(counts, n_local, group=group)
    counts = [int(c) for c in counts]
    nmax, n_total = max(counts), sum(counts)
    offs = [sum(counts[:r]) for r in range(world)]

    def mark(name):
        if timings is not None and dev.type == "cuda":
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            timings[name] = ev

    def padded(mem):
        if mem.shape[0] == nmax:
            return mem.contiguous()
        return torch.cat([mem, mem.new_zeros((nmax - mem.shape[0],) + tuple(mem.shape[1:]))], 0)

    mark("start")
    k_all = torch.empty((world, nmax, B, S, H * D), dtype=km.dtype, device=dev)
    v_all = torch.empty_like(k_all)
    pending = []
    if nmax > 0:
        pending = [dist.all_gather_into_tensor(k_all.view(world * nmax, B, S, H * D), padded(km), group=group, async_op=True),
                   dist.all_gather_into_tensor(v_all.view(world * nmax, B, S, H * D), padded(vm), group=group, async_op=True)]
    block = torch.zeros((counts[rank], n_total), dtype=torch.float32 if dev.type == "cuda" else torch.float64, device=dev)
    if counts[rank] > 0:
        # own columns first: this work hides the exchange
        block[:, offs[rank]: offs[rank] + counts[rank]] = _matrix_block(local, local.k, local.v, similarity, scale)
    mark("own_done")
    for w in pending:
        w.wait()
    mark("exchange_done")
    view = lambda m: m.view(m.shape[0], B, S, H, D).permute(0, 1, 3, 2, 4)  # noqa: E731
    if counts[rank] > 0:
        for p in range(world):
            if p == rank or counts[p] == 0:
                continue
            block[:, offs[p]: offs[p] + counts[p]] = _matrix_block(local, view(k_all[p, : counts[p]]),
                                                                  view(v_all[p, : counts[p]]), similarity, scale)
    mark("block_done")
    if not gather_to_all:
        mark("end")
        return block
    pad = block
    if block.shape[0] < nmax:
        pad = torch.cat([block, block.new_zeros((nmax - block.shape[0], block.shape[1]))], 0)
    out = torch.empty((world * nmax, n_total), dtype=block.dtype, device=dev)
    if nmax > 0:
        dist.all_gather_into_tensor(out, pad.contiguous(), group=group)
    mark("end")
    return torch.cat([out[r * nmax: r * nmax + c] for r, c in enumerate(counts)], 0)


def _matrix_block(local: QKVCache, k_all: torch.Tensor, v_all: torch.Tensor, similarity, scale):
    """Hook for tests: the per-rank block computation (CUDA kernels)."""
    return ops.aas_matrix(local.q, local.k, local.v, k_all, v_all, similarity, scale)


def symmetrize(dm: torch.Tensor) -> torch.Tensor:
    """S = (Dm + Dm^T)/2: DiffSim.diffsim(i, j) for every pair (diffsim/diffsim.py:197)."""
    return (dm + dm.t()) * 0.5


def ranked_lists(score: torch.Tensor, names: Sequence[str], topk: int = 5, larger_is_closer: bool = True,
                 skip_self: bool = True) -> List[str]:
    """Compact one-line-per-query summary '<query>: <best> <2nd> ...' (for logs).  The per-query result FILES that
    retrieval_vis.py:57-68 parses (one retrieved image per line) are written by retrieval.write_retrieval_results."""
    n = score.shape[0]
    s = score.clone().float()
    if skip_self:
        s.fill_diagonal_(float("-inf") if larger_is_closer else float("inf"))
    idx = torch.topk(s, min(topk, n - (1 if skip_self else 0)), dim=1, largest=larger_is_closer).indices.cpu()
    return [f"{names[i]}: " + " ".join(names[j] for j in idx[i].tolist()) for i in range(n)]
