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

    gather_to_all=False returns the rank's row block Dm[own rows, all columns], differentiable in local.q/k/v when
    grad mode is on and one of them requires grad.  Its backward gathers the row blocks of dL/dDm and the Q, K, V of
    every image, and computes the gradients of the rank's own images with two passes of the matrix backward: its rows
    against all columns (dq, dk_self, dv_self) and all rows against its columns (dk, dv).  No gradient crosses ranks,
    and every rank's gradients are bit for bit those of one device's ops.aas_matrix_bwd with separate self buffers.
    Two requirements, as for DistributedDataParallel: every rank runs the backward (it holds collectives), and a
    rank's loss depends on its own block only (a gradient reaching a peer's block through another path is lost).
    gather_to_all=True is forward only: the gathered matrix has no graph.
    """
    if not gather_to_all and ops.wants_grad(local.q, local.k, local.v):
        return _ShardedMatrixFn.apply(similarity, scale, group, timings, local.q, local.k, local.v)
    with torch.no_grad():
        return _aas_matrix_sharded(local, similarity, scale, group, gather_to_all, timings)[0]


def _shard_counts(n_local: int, group, dev) -> List[int]:
    import torch.distributed as dist

    n = torch.tensor([n_local], dtype=torch.int64, device=dev)
    counts = [torch.zeros_like(n) for _ in range(dist.get_world_size(group))]
    dist.all_gather(counts, n, group=group)
    return [int(c) for c in counts]


def _aas_matrix_sharded(local: QKVCache, similarity, scale, group, gather_to_all, timings):
    """(matrix or row block, image counts per rank) of aas_matrix_sharded, without a graph."""
    import torch.distributed as dist

    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    _, km, vm = local.memory()
    dev = km.device
    B, H, S, D = local.shape
    counts = _shard_counts(km.shape[0], group, dev)
    nmax, n_total = max(counts), sum(counts)
    offs = [sum(counts[:r]) for r in range(world)]

    def mark(name):
        if timings is not None and dev.type == "cuda":
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            timings[name] = ev

    mark("start")
    k_all = torch.empty((world, nmax, B, S, H * D), dtype=km.dtype, device=dev)
    v_all = torch.empty_like(k_all)
    pending = []
    if nmax > 0:
        pending = [dist.all_gather_into_tensor(k_all.view(world * nmax, B, S, H * D), _padded(km, nmax), group=group, async_op=True),
                   dist.all_gather_into_tensor(v_all.view(world * nmax, B, S, H * D), _padded(vm, nmax), group=group, async_op=True)]
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
        return block, counts
    out = _all_gather_rows(block, counts, group)
    mark("end")
    return out, counts


def _padded(mem: torch.Tensor, n: int) -> torch.Tensor:
    """mem (contiguous) with zero rows appended up to n rows: the equal-size piece of an all_gather_into_tensor."""
    if mem.shape[0] == n:
        return mem.contiguous()
    return torch.cat([mem, mem.new_zeros((n - mem.shape[0],) + tuple(mem.shape[1:]))], 0)


def _all_gather_rows(t: torch.Tensor, counts: List[int], group) -> torch.Tensor:
    """The ranks' row blocks t (counts[r] rows on rank r) concatenated in rank order, on every rank."""
    import torch.distributed as dist

    nmax = max(counts)
    out = torch.empty((len(counts) * nmax,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    if nmax > 0:
        dist.all_gather_into_tensor(out, _padded(t, nmax), group=group)
    if all(c == nmax for c in counts):
        return out
    return torch.cat([out[r * nmax: r * nmax + c] for r, c in enumerate(counts)], 0)


class _ShardedMatrixFn(torch.autograd.Function):
    """aas_matrix_sharded's row block with the two-pass sharded matrix backward; saves only the local caches."""

    @staticmethod
    def forward(ctx, similarity, scale, group, timings, q, k, v):
        block, counts = _aas_matrix_sharded(QKVCache(q, k, v), similarity, scale, group, False, timings)
        ctx.save_for_backward(q, k, v)
        ctx.similarity, ctx.scale, ctx.group, ctx.counts = similarity, scale, group, counts
        return block

    @staticmethod
    def backward(ctx, d_block):
        import torch.distributed as dist

        q, k, v = ctx.saved_tensors
        counts, group = ctx.counts, ctx.group
        rank = dist.get_rank(group)
        r0 = sum(counts[:rank])
        r1 = r0 + counts[rank]
        d_full = _all_gather_rows(d_block.contiguous(), counts, group)
        n, B, H, S, D = q.shape
        mems = [_all_gather_rows(m, counts, group) for m in QKVCache(q, k, v).memory()]
        q_all, k_all, v_all = (m.view(m.shape[0], B, S, H, D).permute(0, 1, 3, 2, 4) for m in mems)
        if r1 == r0:
            return (None,) * 4 + tuple(torch.zeros_like(t, dtype=d_block.dtype) for t in (q, k, v))
        dq, dks, dvs, dk, dv = _matrix_grad_block(q_all, k_all, v_all, r0, r1, d_full, ctx.similarity, ctx.scale)
        return (None,) * 4 + (dq, dks + dk, dvs + dv)


def _matrix_block(local: QKVCache, k_all: torch.Tensor, v_all: torch.Tensor, similarity, scale):
    """Hook for tests: the per-rank block computation (CUDA kernels)."""
    return ops.aas_matrix(local.q, local.k, local.v, k_all, v_all, similarity, scale)


def _matrix_grad_block(q_all, k_all, v_all, r0: int, r1: int, d_full: torch.Tensor, similarity, scale):
    """Hook for tests: the per-rank backward (CUDA kernels).  (dq, dk_self, dv_self, dk, dv) of sum(d_full * Dm) for
    the images [r0, r1) of the global caches: the row pass (own rows against all columns) and the column pass (all
    rows against own columns).  Each is bitwise the single-device aas_matrix_bwd's with separate self buffers."""
    own = slice(r0, r1)
    dq, dks, dvs, _, _ = ops.aas_matrix_bwd(q_all[own], k_all[own], v_all[own], k_all, v_all, d_full[own], similarity,
                                            scale, need_cols=False)
    _, _, _, dk, dv = ops.aas_matrix_bwd(q_all, k_all, v_all, k_all[own], v_all[own], d_full[:, own], similarity,
                                         scale, need_rows=False)
    return dq, dks, dvs, dk, dv


def aas_scores_between(a: QKVCache, b: QKVCache, similarity: str = "cosine", scale: Optional[float] = None) -> torch.Tensor:
    """DiffSim scores [Na, Nb] between the images of two caches: (Dm(a->b) + Dm(b->a)^T) / 2, entry (i, j) the value of
    DiffSim.diffsim(a_i, b_j).  The caches may hold different token counts (a query set and a gallery captured at two
    image sizes); B, H, D and the dtype must match.  Differentiable in both caches (ops.aas_matrix) when one of them
    requires grad."""
    ab = ops.aas_matrix(a.q, a.k, a.v, b.k, b.v, similarity, scale)
    ba = ops.aas_matrix(b.q, b.k, b.v, a.k, a.v, similarity, scale)
    return (ab + ba.t()) * 0.5


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
