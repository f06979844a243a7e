"""Torch-facing wrappers of the C ABI.  PyTorch supplies device memory and streams; all
arithmetic runs in libdiffsim_b200.so (hand-written sm_100a kernels).  No fallbacks.

Tensor layouts are consumed as they are: the reference's (B,H,S,D) views over (B,S,H*D)
memory (diffsim/hacked_attn.py:74-77) and DiT's packed qkv (diffsim/diffsim_dit.py:22-23)
are described to the library by their strides, never copied.
"""
from __future__ import annotations

import math
from typing import Optional, Sequence, Tuple

import torch

from . import _native as N

SIM_MODES = {"cosine": N.DS_SIM_COSINE, "mse": N.DS_SIM_MSE, "minmax_cosine": N.DS_SIM_MINMAX_COSINE}

_DTYPES = {torch.float16: N.DS_F16, torch.bfloat16: N.DS_BF16, torch.float32: N.DS_F32}

# per-device scratch buffers (grown on demand, reused across calls on the same stream)
_workspaces: dict = {}

# number of diffsim_b200 CUDA kernels launched through this module (bench.py reports it as gpu_launches)
LAUNCHES = 0


def _mode(similarity) -> int:
    if isinstance(similarity, int):
        return similarity
    # the reference treats anything that is not 'cosine' as MSE (diffsim/diffsim.py:182-195)
    return SIM_MODES.get(similarity, N.DS_SIM_MSE)


def _need_cuda(*ts: torch.Tensor) -> torch.device:
    dev = ts[0].device
    for t in ts:
        if not t.is_cuda:
            raise RuntimeError("diffsim_b200 ops need CUDA tensors (there is no CPU path)")
        if t.device != dev:
            raise RuntimeError("all tensors must be on the same device")
    return dev


def _workspace(dev: torch.device, nbytes: int, slot: str = "main") -> torch.Tensor:
    # one buffer per (device, stream, slot): calls issued on two streams must not share partials
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), torch.cuda.current_stream(dev).cuda_stream, slot)
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=dev)
        _workspaces[key] = buf
    return buf


def _dtype_code(t: torch.Tensor) -> int:
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise RuntimeError(f"unsupported dtype {t.dtype}") from None


_DESCRIPTORS = {4: (N.Tensor4, "(B,H,S,D)"), 5: (N.Tensor5, "(N,B,H,S,D)")}


def _desc(t: torch.Tensor, rank: int):
    """The ds_tensor4 / ds_tensor5 descriptor of t (no copy: sizes and strides as they are)."""
    cls, layout = _DESCRIPTORS[rank]
    if t.dim() != rank:
        raise RuntimeError(f"expected a {layout} tensor, got shape {tuple(t.shape)}")
    d = cls()
    d.ptr = t.data_ptr()
    d.size[:] = list(t.shape)
    d.stride[:] = list(t.stride())
    d.dtype = _dtype_code(t)
    return d


def _scale_arg(scale) -> float:
    # the library's softmax scale argument: anything not positive (None, 0, < 0) selects the default 1/sqrt(D)
    return 0.0 if scale is None or not scale > 0 else float(scale)


def _call(name: str, dev: torch.device, *args, launches: int, ws_query: Optional[tuple] = None,
          slot: str = "main") -> None:
    """lib.<name>(*args, ws, ws_bytes, stream) on dev's current stream, with the workspace sized by
    lib.<name>_workspace_bytes(*ws_query); without ws_query, lib.<name>(*args, stream).  An error status raises
    DiffSimError; `launches` (the kernels the call issues) is added to LAUNCHES."""
    global LAUNCHES
    lib = N.load()
    tail = ()
    if ws_query is not None:
        ws = _workspace(dev, getattr(lib, name + "_workspace_bytes")(*ws_query), slot)
        tail = (ws.data_ptr(), ws.numel())
    with torch.cuda.device(dev):
        N.check(getattr(lib, name)(*args, *tail, torch.cuda.current_stream(dev).cuda_stream))
    LAUNCHES += launches


def _i32(x, dev) -> torch.Tensor:
    if isinstance(x, torch.Tensor):
        return x.to(device=dev, dtype=torch.int32).contiguous()
    return torch.as_tensor(x, dtype=torch.int32).to(dev).contiguous()


# --------------------------------------------------------------------------------------
# K1: attention
# --------------------------------------------------------------------------------------
def wants_grad(*ts: torch.Tensor) -> bool:
    """True when autograd records this call: grad mode is on and some input requires grad."""
    return torch.is_grad_enabled() and any(t.requires_grad for t in ts)


def attn_fwd(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, scale: Optional[float] = None,
             out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """softmax(q k^T * scale) v per (b,h) -- F.scaled_dot_product_attention(q,k,v,dropout_p=0.0,is_causal=False)
    (diffsim/hacked_attn.py:81-83, diffsim/diffsim.py:177-180).  Returns (B,H,Sq,D) in q's dtype, laid out like
    the reference's head-split views: memory (B,Sq,H*D).  Differentiable (attn_bwd) when an input requires grad;
    `out` is not accepted then."""
    if wants_grad(q, k, v):
        if out is not None:
            raise RuntimeError("attn_fwd: out= is not supported when an input requires grad")
        return _AttnFn.apply(q, k, v, scale)
    return _attn_fwd(q, k, v, scale, out)


def _attn_fwd(q, k, v, scale=None, out=None) -> torch.Tensor:
    dev = _need_cuda(q, k, v)
    B, H, Sq, D = q.shape
    if out is None:
        out = torch.empty((B, Sq, H, D), dtype=q.dtype, device=dev).permute(0, 2, 1, 3)
    q4, k4 = _desc(q, 4), _desc(k, 4)
    _call("ds_attn_fwd", dev, q4, k4, _desc(v, 4), _scale_arg(scale), _desc(out, 4), ws_query=(q4, k4),
          launches=2)  # meta + attention
    return out


class _AttnFn(torch.autograd.Function):
    """attn_fwd with the K5 backward; saves only the inputs and recomputes the output in backward."""

    @staticmethod
    def forward(ctx, q, k, v, scale):
        ctx.save_for_backward(q, k, v)
        ctx.scale = scale
        return _attn_fwd(q, k, v, scale)

    @staticmethod
    def backward(ctx, dout):
        q, k, v = ctx.saved_tensors
        out = _attn_fwd(q, k, v, ctx.scale)
        dq, dk, dv = attn_bwd(q, k, v, out, dout, ctx.scale)
        return dq, dk, dv, None


def _tma_ok(t: torch.Tensor) -> torch.Tensor:
    # a 16-bit operand the library reads by TMA: unit innermost stride, 16-byte aligned base and rows (autograd hands
    # out expanded or otherwise arbitrary gradients)
    ok = t.stride(-1) == 1 and t.data_ptr() % 16 == 0 and all(
        n == 1 or (s > 0 and s % 8 == 0) for n, s in zip(t.shape[:-1], t.stride()[:-1]))
    return t if ok else t.contiguous()


def _grads_like(ts, grads) -> Tuple[torch.Tensor, ...]:
    if grads is None:
        return tuple(torch.zeros(t.shape, dtype=torch.float32, device=t.device) for t in ts)
    if len(grads) != len(ts) or any(g.dtype != torch.float32 or g.shape != t.shape for g, t in zip(grads, ts)):
        raise RuntimeError("grads must be float32 tensors of the inputs' shapes")
    return tuple(grads)


def attn_bwd(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, out: torch.Tensor, dout: torch.Tensor,
             scale: Optional[float] = None, grads: Optional[Sequence[torch.Tensor]] = None) -> Tuple[torch.Tensor, ...]:
    """Gradients (dq, dk, dv) of attn_fwd for the output gradient dout, in float32 (deterministic: no atomics).
    out: the forward output attn_fwd(q, k, v, scale).  grads: optional float32 (dq, dk, dv) to add into."""
    dev = _need_cuda(q, k, v, out, dout)
    dout = _tma_ok(dout.to(q.dtype))
    dq, dk, dv = _grads_like((q, k, v), grads)
    q4, k4 = _desc(q, 4), _desc(k, 4)
    _call("ds_attn_bwd", dev, q4, k4, _desc(v, 4), _desc(out, 4), _desc(dout, 4), _scale_arg(scale), _desc(dq, 4),
          _desc(dk, 4), _desc(dv, 4), ws_query=(q4, k4), slot="bwd", launches=2)  # dQ + dK/dV
    return dq, dk, dv


def aas_dir_bwd(q_i: torch.Tensor, k_i: torch.Tensor, v_i: torch.Tensor, k_j: torch.Tensor, v_j: torch.Tensor,
                d_dir: torch.Tensor, similarity="cosine", scale: Optional[float] = None,
                grads: Optional[Sequence[torch.Tensor]] = None) -> Tuple[torch.Tensor, ...]:
    """Gradients (dq_i, dk_i, dv_i, dk_j, dv_j) of dir = sim(Attn(q_i,k_j,v_j), Attn(q_i,k_i,v_i)) for dL/ddir = d_dir
    (a one-element tensor on the device; no host sync), in float32.  (B,H,S,D) inputs as for attn_fwd.
    grads: optional float32 tensors to add into (they may alias, e.g. dk_i is dk_j when image i is image j)."""
    dev = _need_cuda(q_i, k_i, v_i, k_j, v_j, d_dir)
    g = d_dir.detach().reshape(-1).to(torch.float32)
    if g.numel() != 1:
        raise RuntimeError("d_dir must have exactly one element")
    out = _grads_like((q_i, k_i, v_i, k_j, v_j), grads)
    q4, kj4 = _desc(q_i, 4), _desc(k_j, 4)
    _call("ds_aas_dir_bwd", dev, q4, _desc(k_i, 4), _desc(v_i, 4), kj4, _desc(v_j, 4), _scale_arg(scale),
          _mode(similarity), g.data_ptr(), *[_desc(t, 4) for t in out], ws_query=(q4, kj4), slot="bwd",
          launches=11)  # 2 x (meta + attention) recompute + partials + coefficients + factors + 2 x (dQ + dK/dV)
    return out


def _pair_dirs(qa, ka, va, qb, kb, vb, similarity, scale):
    """(dir(a->b), dir(b->a)) of one image pair: two aas_groups calls, forward only."""
    one, off = [0], [0, 1]
    d_ab = aas_groups(qa[None], ka[None], va[None], kb[None], vb[None], one, off, one, similarity, scale)
    d_ba = aas_groups(qb[None], kb[None], vb[None], ka[None], va[None], one, off, one, similarity, scale)
    return d_ab, d_ba


def pair_dirs_bwd(qa, ka, va, qb, kb, vb, g_ab, g_ba, similarity="cosine", scale=None) -> Tuple[torch.Tensor, ...]:
    """float32 gradients of (qa, ka, va, qb, kb, vb) for dL/d dir(a->b) = g_ab and dL/d dir(b->a) = g_ba (either may be
    None), accumulated in float32 in a fixed order."""
    grads = _grads_like((qa, ka, va, qb, kb, vb), None)
    dqa, dka, dva, dqb, dkb, dvb = grads
    if g_ab is not None:
        aas_dir_bwd(qa, ka, va, kb, vb, g_ab, similarity, scale, grads=(dqa, dka, dva, dkb, dvb))
    if g_ba is not None:
        aas_dir_bwd(qb, kb, vb, ka, va, g_ba, similarity, scale, grads=(dqb, dkb, dvb, dka, dva))
    return grads


class _PairDirsFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, similarity, scale, qa, ka, va, qb, kb, vb):
        ctx.save_for_backward(qa, ka, va, qb, kb, vb)
        ctx.similarity, ctx.scale = similarity, scale
        return _pair_dirs(qa, ka, va, qb, kb, vb, similarity, scale)

    @staticmethod
    def backward(ctx, g_ab, g_ba):
        return (None, None) + pair_dirs_bwd(*ctx.saved_tensors, g_ab, g_ba, ctx.similarity, ctx.scale)


def pair_dirs(qa, ka, va, qb, kb, vb, similarity="cosine", scale: Optional[float] = None):
    """(dir(a->b), dir(b->a)) of one image pair as float32 (1,) tensors -- two aas_groups launches.  The two images may
    have different token counts (a (B,H,S_a,D) against a (B,H,S_b,D) capture): each direction's self attention runs
    over the query image's own K/V and its cross attention over the other image's.  Differentiable (aas_dir_bwd) when
    an input requires grad; the values are the same either way."""
    if wants_grad(qa, ka, va, qb, kb, vb):
        return _PairDirsFn.apply(similarity, scale, qa, ka, va, qb, kb, vb)
    return _pair_dirs(qa, ka, va, qb, kb, vb, similarity, scale)


def aas_groups(q: torch.Tensor, k_self: torch.Tensor, v_self: torch.Tensor, k: torch.Tensor, v: torch.Tensor,
               group_q, group_off, kv_idx, similarity="cosine", scale: Optional[float] = None) -> torch.Tensor:
    """Directional AAS similarities for grouped (query image, kv image list) work -- see ds_aas_groups.
    q: (Nq,B,H,S_q,D), k_self/v_self: (Nq,B,H,S_self,D); k/v: (Nk,B,H,S_cross,D); the three lengths are independent
    (for AAS S_self = S_q).  Returns float32 [n_entries].  Differentiable in the five
    caches (aas_groups_bwd) when one of them requires grad; the values are the same either way."""
    if wants_grad(q, k_self, v_self, k, v):
        dev = _need_cuda(q)
        return _AASGroupsFn.apply(similarity, scale, _i32(group_q, dev), _i32(group_off, dev), _i32(kv_idx, dev), q,
                                  k_self, v_self, k, v)
    return _aas_groups(q, k_self, v_self, k, v, group_q, group_off, kv_idx, similarity, scale)


def _aas_groups(q, k_self, v_self, k, v, group_q, group_off, kv_idx, similarity="cosine", scale=None) -> torch.Tensor:
    dev = _need_cuda(q, k_self, v_self, k, v)
    gq, go, kv = _i32(group_q, dev), _i32(group_off, dev), _i32(kv_idx, dev)
    n_groups, n_entries = gq.numel(), kv.numel()
    if go.numel() != n_groups + 1:
        raise RuntimeError("group_off must have n_groups + 1 entries")
    dirs = torch.empty(n_entries, dtype=torch.float32, device=dev)
    q5 = _desc(q, 5)
    _call("ds_aas_groups", dev, q5, _desc(k_self, 5), _desc(v_self, 5), _desc(k, 5), _desc(v, 5), gq.data_ptr(),
          go.data_ptr(), n_groups, kv.data_ptr(), n_entries, _scale_arg(scale), _mode(similarity), dirs.data_ptr(),
          ws_query=(q5, n_groups, n_entries), launches=3)  # index validation + attention + finish
    return dirs


def aas_pairs(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, pair_idx, similarity="cosine",
              scale: Optional[float] = None) -> torch.Tensor:
    """score[p] = (dir(a->b) + dir(b->a)) / 2 for pair_idx[p] = (a, b): the value DiffSim.diffsim returns
    (diffsim/diffsim.py:177-197).  q,k,v: (N,B,H,S,D) caches.  Returns float32 [P].  Differentiable in the caches
    (aas_pairs_bwd) when one of them requires grad; the values are the same either way."""
    if wants_grad(q, k, v):
        return _AASPairsFn.apply(similarity, scale, _i32(pair_idx, _need_cuda(q)).reshape(-1, 2), q, k, v)
    return _aas_pairs(q, k, v, pair_idx, similarity, scale)


def _aas_pairs(q, k, v, pair_idx, similarity="cosine", scale=None) -> torch.Tensor:
    dev = _need_cuda(q, k, v)
    pairs = _i32(pair_idx, dev).reshape(-1, 2)
    P = pairs.shape[0]
    scores = torch.empty(P, dtype=torch.float32, device=dev)
    q5 = _desc(q, 5)
    _call("ds_aas_pairs", dev, q5, _desc(k, 5), _desc(v, 5), pairs.data_ptr(), P, _scale_arg(scale), _mode(similarity),
          scores.data_ptr(), ws_query=(q5, P), launches=5)  # setup + index validation + attention + finish + combine
    return scores


def aas_triplets(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, trip_idx, similarity="cosine",
                 scale: Optional[float] = None, round_scores: bool = False, want_flags: bool = True):
    """2AFC triplets (ref, left, right) as the benchmark drivers score them (cute_main.py:111-132,196-205):
    returns (ab, ac, counts, flags) on the device: ab = diffsim(ref,left), ac = diffsim(ref,right) (float32 [T]),
    counts int32[2] = {correct, correct_2x}, flags uint8[T].  One library call, no host sync.  ab and ac are
    differentiable in the caches (aas_triplets_bwd) when one of them requires grad (the rounding of round_scores passes
    straight through); counts and flags are not.  The values are the same either way."""
    if wants_grad(q, k, v):
        trips = _i32(trip_idx, _need_cuda(q)).reshape(-1, 3)
        return _AASTripletsFn.apply(similarity, scale, round_scores, want_flags, trips, q, k, v)
    return _aas_triplets(q, k, v, trip_idx, similarity, scale, round_scores, want_flags)


def _aas_triplets(q, k, v, trip_idx, similarity="cosine", scale=None, round_scores=False, want_flags=True):
    dev = _need_cuda(q, k, v)
    trips = _i32(trip_idx, dev).reshape(-1, 3)
    T = trips.shape[0]
    ab = torch.empty(T, dtype=torch.float32, device=dev)
    ac = torch.empty(T, dtype=torch.float32, device=dev)
    counts = torch.empty(2, dtype=torch.int32, device=dev)
    flags = torch.empty(T, dtype=torch.uint8, device=dev) if want_flags else None
    q5 = _desc(q, 5)
    _call("ds_aas_triplets", dev, q5, _desc(k, 5), _desc(v, 5), trips.data_ptr(), T, _scale_arg(scale),
          _mode(similarity), N.DS_OPT_ROUND_SCORES if round_scores else 0, ab.data_ptr(), ac.data_ptr(),
          counts.data_ptr(), flags.data_ptr() if want_flags else None, ws_query=(q5, T),
          launches=5)  # setup + index validation + attention + finish + combine/decide
    return ab, ac, counts, flags


# Cap on the workspace of one grouped-backward library call: longer lists are cut into chunks of whole groups (pairs,
# triplets), issued in list order.  Every gradient row still receives its terms in entry order, so chunking keeps the
# bitwise contract of ds_aas_groups_bwd.  About 4 MB per entry at the SD-1.5 up0 shape (2, 8, 256, 160).
GROUPS_BWD_WORKSPACE_CAP = 1 << 30


def _grad_buffers(ts, grads):
    """float32 zeros with the strides of each input where it is dense (a head-split view of a (N,B,S,H*D) cache gets its
    gradient in that memory layout), or the caller's `grads` to add into; a repeated input shares one buffer."""
    if grads is not None:
        return _grads_like(ts, grads)
    out = []
    for t in ts:
        same = [o for o, u in zip(out, ts) if u is t]
        out.append(same[0] if same else torch.zeros_like(t, dtype=torch.float32))
    return tuple(out)


def _chunks(n: int, ws_bytes) -> list:
    """[(i0, i1)] cutting n units into runs whose workspace ws_bytes(i1 - i0) stays under GROUPS_BWD_WORKSPACE_CAP."""
    per = max(1, GROUPS_BWD_WORKSPACE_CAP // max(1, ws_bytes(1)))
    return [(i, min(n, i + per)) for i in range(0, n, per)]


def aas_groups_bwd(q: torch.Tensor, k_self: torch.Tensor, v_self: torch.Tensor, k: torch.Tensor, v: torch.Tensor,
                   group_q, group_off, kv_idx, d_dir: torch.Tensor, similarity="cosine", scale: Optional[float] = None,
                   grads: Optional[Sequence[torch.Tensor]] = None) -> Tuple[torch.Tensor, ...]:
    """float32 gradients (dq, dk_self, dv_self, dk, dv) of aas_groups for dL/ddir = d_dir (n_entries values on the device),
    bitwise those of one aas_dir_bwd call per entry in list order (ds_aas_groups_bwd).  When k_self is k (v_self is v)
    the gradient is one buffer: dk_self is dk.  grads: optional float32 tensors to add into (dk_self is dk allowed)."""
    dev = _need_cuda(q, k_self, v_self, k, v, d_dir)
    gq, go, kv = _i32(group_q, dev), _i32(group_off, dev), _i32(kv_idx, dev)
    n_groups, n_entries = gq.numel(), kv.numel()
    if go.numel() != n_groups + 1:
        raise RuntimeError("group_off must have n_groups + 1 entries")
    g = d_dir.detach().reshape(-1).to(torch.float32).contiguous()
    if g.numel() != n_entries:
        raise RuntimeError("d_dir must have one value per entry")
    out = _grad_buffers((q, k_self, v_self, k, v), grads)
    if n_groups == 0 or n_entries == 0:
        return out
    lib = N.load()
    q5, k5 = _desc(q, 5), _desc(k, 5)
    args = (q5, _desc(k_self, 5), _desc(v_self, 5), k5, _desc(v, 5))
    gdesc = [_desc(t, 5) for t in out]
    if lib.ds_aas_groups_bwd_workspace_bytes(q5, k5, n_groups, n_entries) <= GROUPS_BWD_WORKSPACE_CAP:
        spans = [(0, n_groups)]
    else:   # cut into runs of whole groups (needs the group offsets on the host)
        off = go.tolist()
        spans, g0 = [], 0
        for g1 in range(1, n_groups + 1):
            if g1 > g0 + 1 and lib.ds_aas_groups_bwd_workspace_bytes(q5, k5, g1 - g0, off[g1] - off[g0]) > GROUPS_BWD_WORKSPACE_CAP:
                spans.append((g0, g1 - 1))
                g0 = g1 - 1
        spans.append((g0, n_groups))
        go = go.cpu()
    for g0, g1 in spans:
        e0, e1 = (0, n_entries) if len(spans) == 1 else (int(go[g0]), int(go[g1]))
        off = go if len(spans) == 1 else (go[g0:g1 + 1] - e0).to(dev)
        _call("ds_aas_groups_bwd", dev, *args, gq[g0:].data_ptr(), off.data_ptr(), g1 - g0, kv[e0:].data_ptr(), e1 - e0,
              _scale_arg(scale), _mode(similarity), g[e0:].data_ptr(), *gdesc, ws_query=(q5, k5, g1 - g0, e1 - e0),
              slot="bwd", launches=10)  # validation + entry groups + lists + recompute + partials + coefficients
        #                                  + factors + dQ + dK/dV + NaN fill
    return out


def aas_pairs_bwd(q, k, v, pair_idx, d_scores, similarity="cosine", scale=None, grads=None) -> Tuple[torch.Tensor, ...]:
    """float32 gradients (dq, dk, dv) of aas_pairs for dL/dscore = d_scores (ds_aas_pairs_bwd: aas_groups_bwd of the
    pairs' work list), added into `grads` when given."""
    dev = _need_cuda(q, k, v, d_scores)
    pairs = _i32(pair_idx, dev).reshape(-1, 2)
    g = d_scores.detach().reshape(-1).to(torch.float32).contiguous()
    if g.numel() != pairs.shape[0]:
        raise RuntimeError("d_scores must have one value per pair")
    out = _grad_buffers((q, k, v), grads)
    lib, q5 = N.load(), _desc(q, 5)
    args, gdesc = (q5, _desc(k, 5), _desc(v, 5)), [_desc(t, 5) for t in out]
    for p0, p1 in _chunks(pairs.shape[0], lambda n: lib.ds_aas_pairs_bwd_workspace_bytes(q5, n)):
        _call("ds_aas_pairs_bwd", dev, *args, pairs[p0:].data_ptr(), p1 - p0, _scale_arg(scale), _mode(similarity),
              g[p0:].data_ptr(), *gdesc, ws_query=(q5, p1 - p0), slot="bwd", launches=12)  # setup + d_dir + groups_bwd
    return out


def aas_triplets_bwd(q, k, v, trip_idx, d_ab, d_ac, similarity="cosine", scale=None, grads=None) -> Tuple[torch.Tensor, ...]:
    """float32 gradients (dq, dk, dv) of the (ab, ac) of aas_triplets for dL/dab = d_ab and dL/dac = d_ac (either may
    be None: zero) -- ds_aas_triplets_bwd -- added into `grads` when given."""
    dev = _need_cuda(q, k, v)
    trips = _i32(trip_idx, dev).reshape(-1, 3)
    T = trips.shape[0]
    zero = torch.zeros(T, dtype=torch.float32, device=dev)
    gab = zero if d_ab is None else d_ab.detach().reshape(-1).to(torch.float32).contiguous()
    gac = zero if d_ac is None else d_ac.detach().reshape(-1).to(torch.float32).contiguous()
    if gab.numel() != T or gac.numel() != T:
        raise RuntimeError("d_ab and d_ac must have one value per triplet")
    out = _grad_buffers((q, k, v), grads)
    lib, q5 = N.load(), _desc(q, 5)
    args, gdesc = (q5, _desc(k, 5), _desc(v, 5)), [_desc(t, 5) for t in out]
    for t0, t1 in _chunks(T, lambda n: lib.ds_aas_triplets_bwd_workspace_bytes(q5, n)):
        _call("ds_aas_triplets_bwd", dev, *args, trips[t0:].data_ptr(), t1 - t0, _scale_arg(scale), _mode(similarity),
              gab[t0:].data_ptr(), gac[t0:].data_ptr(), *gdesc, ws_query=(q5, t1 - t0), slot="bwd",
              launches=12)  # setup + d_dir + groups_bwd
    return out


def _matrix_spans(nr: int, nc: int, ws_bytes) -> list:
    """[((r0, r1), (c0, c1))] cutting an nr x nc matrix backward into calls whose workspace ws_bytes(rows, cols) stays under
    GROUPS_BWD_WORKSPACE_CAP: blocks of whole rows, in order, and column blocks only when one row does not fit."""
    cap = GROUPS_BWD_WORKSPACE_CAP
    if ws_bytes(nr, nc) <= cap:
        return [((0, nr), (0, nc))]
    if ws_bytes(1, nc) <= cap:
        per = 1
        while per < nr and ws_bytes(per + 1, nc) <= cap:
            per += 1
        return [((r, min(nr, r + per)), (0, nc)) for r in range(0, nr, per)]
    per = 1
    while per < nc and ws_bytes(1, per + 1) <= cap:
        per += 1
    return [((r, r + 1), (c, min(nc, c + per))) for r in range(nr) for c in range(0, nc, per)]


def aas_matrix_bwd(q: torch.Tensor, k_self: torch.Tensor, v_self: torch.Tensor, k: torch.Tensor, v: torch.Tensor,
                   d_Dm: torch.Tensor, similarity="cosine", scale: Optional[float] = None,
                   grads: Optional[Sequence[torch.Tensor]] = None, need_rows: bool = True,
                   need_cols: bool = True) -> Tuple[Optional[torch.Tensor], ...]:
    """float32 gradients (dq, dk_self, dv_self, dk, dv) of aas_matrix for dL/dDm = d_Dm ([Nr, Nc] on the device) --
    ds_aas_matrix_bwd: the grouped backward of the row-major list with each row's self terms folded into one.  When
    k_self is k (v_self is v) the gradient is one buffer.  grads: optional float32 tensors to add into (None in the
    places of a family that is not asked for).

    need_rows / need_cols select the two gradient families: the row terms (dq, dk_self, dv_self) and the column terms
    (dk, dv); a family not asked for is returned as None and not computed.  Each family alone is bitwise what the full
    call gives it when dk_self / dv_self are separate buffers, so the gradients of a set of images can be formed from
    its rows against all columns (need_cols=False) and all rows against its columns (need_rows=False).

    A matrix whose workspace would exceed GROUPS_BWD_WORKSPACE_CAP is cut into blocks of whole rows (columns only when
    one row does not fit; each column block then folds its own self term).  Row blocks are bitwise one call when the
    self gradients are separate buffers; with one shared buffer a block's self terms are added after the block."""
    if not (need_rows or need_cols):
        raise RuntimeError("aas_matrix_bwd: need_rows or need_cols must be set")
    dev = _need_cuda(q, k_self, v_self, k, v, d_Dm)
    nr, nc = q.shape[0], k.shape[0]
    g = d_Dm.detach().to(torch.float32)
    if g.shape != (nr, nc):
        raise RuntimeError(f"d_Dm must have shape ({nr}, {nc}), got {tuple(g.shape)}")
    if (nc > 1 and g.stride(1) != 1) or (nr > 1 and g.stride(0) < nc):
        g = g.contiguous()
    ldd = g.stride(0) if nr > 1 else nc
    if need_rows and need_cols:
        out = _grad_buffers((q, k_self, v_self, k, v), grads)
    else:   # one family: its buffers only (a skipped family's entries of grads are not used)
        want = (need_rows,) * 3 + (need_cols,) * 2
        ts = [t for t, w in zip((q, k_self, v_self, k, v), want) if w]
        got = iter(_grad_buffers(ts, None if grads is None else [t for t, w in zip(grads, want) if w]))
        out = tuple(next(got) if w else None for w in want)
    dq, dks, dvs, dk, dv = out
    lib = N.load()
    ws = lambda r, c: lib.ds_aas_matrix_bwd_workspace_bytes(_desc(q[:r], 5), _desc(k[:c], 5))  # noqa: E731
    spans = _matrix_spans(nr, nc, ws)
    shared = need_rows and need_cols and (dks is dk or dvs is dv)
    null = N.Tensor5()   # ptr 0: a family not asked for
    part = lambda t, i0, i1: null if t is None else _desc(t[i0:i1], 5)  # noqa: E731
    for (r0, r1), (c0, c1) in spans:
        rows = (q[r0:r1], k_self[r0:r1], v_self[r0:r1])
        cols = (k[c0:c1], v[c0:c1])
        gks, gvs = part(dks, r0, r1), part(dvs, r0, r1)
        if shared and len(spans) > 1:   # the C call takes one shared buffer whole, not a block of it
            bks, bvs = torch.zeros_like(dks[r0:r1]), torch.zeros_like(dvs[r0:r1])
            gks, gvs = _desc(bks, 5), _desc(bvs, 5)
        q5, k5 = _desc(rows[0], 5), _desc(cols[0], 5)
        _call("ds_aas_matrix_bwd", dev, q5, _desc(rows[1], 5), _desc(rows[2], 5), k5, _desc(cols[1], 5), _scale_arg(scale),
              _mode(similarity), g[r0:, c0:].data_ptr(), ldd, part(dq, r0, r1), gks, gvs, part(dk, c0, c1),
              part(dv, c0, c1), ws_query=(q5, k5), slot="bwd",
              # setup + lists + recompute + partials + coefficients + fold (+ fold rounding) + dQ (or statistics)
              # + dK/dV; without the row terms nothing is folded, so there is no rounding
              launches=9 if need_rows else 8)
        if shared and len(spans) > 1:
            dks[r0:r1] += bks
            dvs[r0:r1] += bvs
    return out


class _AASMatrixFn(torch.autograd.Function):
    """aas_matrix with the folded grouped K5 backward; saves only the caches."""

    @staticmethod
    def forward(ctx, similarity, scale, q, k_self, v_self, k, v):
        ctx.save_for_backward(q, k_self, v_self, k, v)
        ctx.similarity, ctx.scale = similarity, scale
        return _aas_matrix(q, k_self, v_self, k, v, similarity, scale)

    @staticmethod
    def backward(ctx, d_Dm):
        q, ks, vs, k, v = ctx.saved_tensors
        dq, dks, dvs, dk, dv = aas_matrix_bwd(q, ks, vs, k, v, d_Dm, ctx.similarity, ctx.scale)
        return (None,) * 2 + (dq, None if dks is dk else dks, None if dvs is dv else dvs, dk, dv)


class _AASGroupsFn(torch.autograd.Function):
    """aas_groups with the grouped K5 backward; saves only the caches and the index tensors."""

    @staticmethod
    def forward(ctx, similarity, scale, gq, go, kv, q, k_self, v_self, k, v):
        ctx.save_for_backward(gq, go, kv, q, k_self, v_self, k, v)
        ctx.similarity, ctx.scale = similarity, scale
        return _aas_groups(q, k_self, v_self, k, v, gq, go, kv, similarity, scale)

    @staticmethod
    def backward(ctx, d_dir):
        gq, go, kv, q, ks, vs, k, v = ctx.saved_tensors
        dq, dks, dvs, dk, dv = aas_groups_bwd(q, ks, vs, k, v, gq, go, kv, d_dir, ctx.similarity, ctx.scale)
        # one buffer for a repeated input holds the gradient once: hand it to one of the two slots only
        return (None,) * 5 + (dq, None if dks is dk else dks, None if dvs is dv else dvs, dk, dv)


class _AASPairsFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, similarity, scale, pairs, q, k, v):
        ctx.save_for_backward(pairs, q, k, v)
        ctx.similarity, ctx.scale = similarity, scale
        return _aas_pairs(q, k, v, pairs, similarity, scale)

    @staticmethod
    def backward(ctx, d_scores):
        pairs, q, k, v = ctx.saved_tensors
        return (None,) * 3 + aas_pairs_bwd(q, k, v, pairs, d_scores, ctx.similarity, ctx.scale)


class _AASTripletsFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, similarity, scale, round_scores, want_flags, trips, q, k, v):
        ctx.save_for_backward(trips, q, k, v)
        ctx.similarity, ctx.scale = similarity, scale
        ab, ac, counts, flags = _aas_triplets(q, k, v, trips, similarity, scale, round_scores, want_flags)
        ctx.mark_non_differentiable(*[t for t in (counts, flags) if t is not None])
        return ab, ac, counts, flags

    @staticmethod
    def backward(ctx, d_ab, d_ac, _counts, _flags):
        trips, q, k, v = ctx.saved_tensors
        return (None,) * 5 + aas_triplets_bwd(q, k, v, trips, d_ab, d_ac, ctx.similarity, ctx.scale)


def aas_matrix(q: torch.Tensor, k_self: torch.Tensor, v_self: torch.Tensor, k: torch.Tensor, v: torch.Tensor,
               similarity="cosine", scale: Optional[float] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Directional matrix Dm[r,c] = dir(row image r -> column image c); rows (q,k_self,v_self): (Nr,...),
    columns (k,v): (Nc,...); the columns' token count may differ from the rows' (captures at two resolutions, see
    scoring.aas_scores_between).  Returns float32 [Nr,Nc].  Differentiable in the five caches (aas_matrix_bwd) when one of
    them requires grad and `out` is not given; the values are the same either way."""
    if out is None and wants_grad(q, k_self, v_self, k, v):
        return _AASMatrixFn.apply(similarity, scale, q, k_self, v_self, k, v)
    return _aas_matrix(q, k_self, v_self, k, v, similarity, scale, out)


def _aas_matrix(q, k_self, v_self, k, v, similarity="cosine", scale=None, out=None) -> torch.Tensor:
    dev = _need_cuda(q, k_self, v_self, k, v)
    nr, nc = q.shape[0], k.shape[0]
    if out is None:
        out = torch.empty((nr, nc), dtype=torch.float32, device=dev)
    q5, k5 = _desc(q, 5), _desc(k, 5)
    _call("ds_aas_matrix", dev, q5, _desc(k_self, 5), _desc(v_self, 5), k5, _desc(v, 5), _scale_arg(scale),
          _mode(similarity), out.data_ptr(), out.stride(0), ws_query=(q5, k5), launches=3)  # setup + attention + finish
    return out


# --------------------------------------------------------------------------------------
# K2: reductions
# --------------------------------------------------------------------------------------
def pair_reduce(x: torch.Tensor, y: torch.Tensor, similarity="cosine") -> torch.Tensor:
    """sim(x[p], y[p]) over the flattened trailing dims, for every leading row p.  x, y: (P, ...) tensors whose rows
    are contiguous.  Replaces F.cosine_similarity on flattened tensors / F.mse_loss / min-max + cosine
    (diffsim/diffsim.py:182-195, metrics/diffeats.py:136-140,202-205).  Returns float32 [P].  Differentiable in x and
    y (pair_reduce_bwd) when one of them requires grad; the values are the same either way."""
    if wants_grad(x, y):
        return _PairReduceFn.apply(similarity, x, y)
    return _pair_reduce(x, y, similarity)


def _rows(x: torch.Tensor, y: torch.Tensor):
    """(x, y) as (P, E) views with unit column stride, copied only when the flattened rows are not contiguous."""
    P = x.shape[0]
    x2, y2 = x.reshape(P, -1), y.reshape(P, -1)
    if x2.stride(1) != 1:
        x2 = x2.contiguous()
    if y2.stride(1) != 1:
        y2 = y2.contiguous()
    return x2, y2


def _row_stride(t: torch.Tensor) -> int:
    return t.stride(0) if t.shape[0] > 1 else t.shape[1]


def _pair_reduce(x, y, similarity="cosine") -> torch.Tensor:
    dev = _need_cuda(x, y)
    if x.shape != y.shape or x.dtype != y.dtype:
        raise RuntimeError("x and y must have the same shape and dtype")
    P = x.shape[0]
    if P == 0:
        return torch.empty(0, dtype=torch.float32, device=dev)
    x2, y2 = _rows(x, y)
    E = x2.shape[1]
    out = torch.empty(P, dtype=torch.float32, device=dev)
    _call("ds_pair_reduce", dev, x2.data_ptr(), y2.data_ptr(), P, E, _row_stride(x2), _row_stride(y2), _dtype_code(x2),
          _mode(similarity), out.data_ptr(), ws_query=(P, E), launches=1)
    return out


def pair_reduce_bwd(x: torch.Tensor, y: torch.Tensor, d_out: torch.Tensor, similarity="cosine", need_x: bool = True,
                    need_y: bool = True) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
    """float32 gradients (dx, dy) of pair_reduce(x, y, similarity) for dL/dout = d_out (P values on the device), in
    the shapes of x and y, None where not asked for (and then not computed) -- ds_pair_reduce_bwd: the float64 autograd
    gradients of the reference's expressions, deterministic (no atomics)."""
    dev = _need_cuda(x, y, d_out)
    if x.shape != y.shape or x.dtype != y.dtype:
        raise RuntimeError("x and y must have the same shape and dtype")
    P = x.shape[0]
    g = d_out.detach().reshape(-1).to(torch.float32).contiguous()
    if g.numel() != P:
        raise RuntimeError("d_out must have one value per row")
    dx = torch.empty(x.shape, dtype=torch.float32, device=dev) if need_x else None
    dy = torch.empty(y.shape, dtype=torch.float32, device=dev) if need_y else None
    if P == 0 or (dx is None and dy is None):
        return dx, dy
    x2, y2 = _rows(x, y)
    E = x2.shape[1]
    mode = _mode(similarity)
    _call("ds_pair_reduce_bwd", dev, x2.data_ptr(), y2.data_ptr(), P, E, _row_stride(x2), _row_stride(y2),
          _dtype_code(x2), mode, g.data_ptr(), None if dx is None else dx.data_ptr(), E,
          None if dy is None else dy.data_ptr(), E, ws_query=(P, E), slot="bwd",
          launches=1 if mode == N.DS_SIM_MSE else 2)  # (statistics +) gradient pass
    return dx, dy


class _PairReduceFn(torch.autograd.Function):
    """pair_reduce with the K2 backward; saves only x and y (the backward recomputes the row statistics)."""

    @staticmethod
    def forward(ctx, similarity, x, y):
        ctx.save_for_backward(x, y)
        ctx.similarity = similarity
        return _pair_reduce(x, y, similarity)

    @staticmethod
    def backward(ctx, d_out):
        x, y = ctx.saved_tensors
        return (None,) + pair_reduce_bwd(x, y, d_out, ctx.similarity, ctx.needs_input_grad[1], ctx.needs_input_grad[2])


# --------------------------------------------------------------------------------------
# K3: N x N feature similarity matrix
# --------------------------------------------------------------------------------------
def simmat(rows: torch.Tensor, cols: Optional[torch.Tensor] = None, similarity="cosine",
           out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """C[r,c] = sim(rows[r], cols[c]) for 16-bit feature matrices rows (Nr,L), cols (Nc,L) (default cols = rows)."""
    if cols is None:
        cols = rows
    dev = _need_cuda(rows, cols)
    if rows.dim() != 2 or cols.dim() != 2 or rows.shape[1] != cols.shape[1] or rows.dtype != cols.dtype:
        raise RuntimeError("rows and cols must be 2-D with the same feature length and dtype")
    if rows.stride(1) != 1 or cols.stride(1) != 1:
        raise RuntimeError("feature rows must be contiguous")
    nr, L = rows.shape
    nc = cols.shape[0]
    if out is None:
        out = torch.empty((nr, nc), dtype=torch.float32, device=dev)
    # statistics pass + its finish per operand (one operand when rows is cols: the symmetric call), GEMM, normalise
    symmetric = cols.data_ptr() == rows.data_ptr() and nr == nc and cols.stride(0) == rows.stride(0)
    _call("ds_simmat", dev, rows.data_ptr(), nr, rows.stride(0), cols.data_ptr(), nc, cols.stride(0), L,
          _dtype_code(rows), _mode(similarity), out.data_ptr(), out.stride(0), ws_query=(nr, nc, L),
          launches=4 if symmetric else 6)
    return out


# --------------------------------------------------------------------------------------
# K4: QKV projection of the hooked layer
# --------------------------------------------------------------------------------------
def qkv_project(hidden: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None, n_outputs: int = 3,
                out: Optional[Sequence[torch.Tensor]] = None) -> Tuple[torch.Tensor, ...]:
    """hidden (..., C_in) x weight (n_out, C_in)^T (+ bias) -> n_outputs tensors (..., n_out / n_outputs).

    The capture step of the reference on the hook's input: attn.to_q / to_k / to_v (diffsim/hacked_attn.py:61-69,
    weight = the three nn.Linear weights stacked along dim 0) or DiT's fused module.qkv (diffsim/diffsim_dit.py:21,
    n_outputs = 1: one packed (..., 3C) tensor).  fp32 accumulation on tcgen05, one rounding to the input dtype.
    `out`: optional pre-allocated outputs (row stride may exceed the column count, e.g. slices of a cache).
    Differentiable in hidden, weight and bias (qkv_project_bwd) when one of them requires grad and `out` is not given;
    the outputs are bitwise the same either way.  A call with `out` (a capture into a cache) is forward-only."""
    if out is None and wants_grad(hidden, weight, *(() if bias is None else (bias,))):
        return _QKVProjectFn.apply(n_outputs, 0, hidden, weight, bias)
    return _qkv_project(hidden, weight, bias, n_outputs, out)


def qkv_project_stacked(hidden: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], n_outputs: int,
                        weights: Sequence[torch.Tensor], biases: Sequence[Optional[torch.Tensor]]) -> Tuple[torch.Tensor, ...]:
    """qkv_project on a stacked weight (and bias) built from the equal-sized row blocks `weights` (and `biases`, None
    where a block has none), e.g. a cached [W_q; W_k; W_v] of three nn.Linear modules.  The product runs once on the
    stack; when grad is recorded, the gradients of its row blocks go to `weights` / `biases`, which are the graph's
    inputs (the stack itself receives none)."""
    if len(weights) != len(biases):
        raise RuntimeError("weights and biases must have one entry per row block")
    if wants_grad(hidden, *weights, *[b for b in biases if b is not None]):
        return _QKVProjectFn.apply(n_outputs, len(weights), hidden, weight.detach(),
                                   None if bias is None else bias.detach(), *weights, *biases)
    return _qkv_project(hidden, weight, bias, n_outputs)


def _qkv_project(hidden, weight, bias=None, n_outputs=3, out=None) -> Tuple[torch.Tensor, ...]:
    import ctypes as C

    dev = _need_cuda(hidden, weight)
    if hidden.dtype != weight.dtype or (bias is not None and bias.dtype != hidden.dtype):
        raise RuntimeError("hidden, weight and bias must share one 16-bit dtype")
    c_in = hidden.shape[-1]
    if weight.dim() != 2 or weight.shape[1] != c_in or weight.stride(1) != 1:
        raise RuntimeError(f"weight must be (n_out, {c_in}) with contiguous rows (nn.Linear layout)")
    n_out = weight.shape[0]
    if n_out % n_outputs:
        raise RuntimeError("n_out must be a multiple of n_outputs")
    cols = n_out // n_outputs
    h2 = hidden.reshape(-1, c_in)
    if h2.stride(1) != 1:
        h2 = h2.contiguous()
    rows = h2.shape[0]
    if out is None:
        out = [torch.empty(hidden.shape[:-1] + (cols,), dtype=hidden.dtype, device=dev) for _ in range(n_outputs)]
    if len(out) != n_outputs:
        raise RuntimeError(f"expected {n_outputs} output tensors")
    o2 = []
    for o in out:
        if o.dtype != hidden.dtype or o.device != dev or o.shape[-1] != cols or o.stride(-1) != 1 or o.numel() != rows * cols:
            raise RuntimeError("outputs must be (..., n_out / n_outputs) tensors of the input dtype on the input device")
        o_rows = o.reshape(-1, cols) if o.is_contiguous() else o.view(-1, cols)
        o2.append(o_rows)
    ptrs = (C.c_void_p * n_outputs)(*[o.data_ptr() for o in o2])
    lds = (C.c_int64 * n_outputs)(*[o.stride(0) for o in o2])
    _call("ds_qkv_project", dev, h2.data_ptr(), rows, h2.stride(0), c_in, weight.data_ptr(), weight.stride(0),
          bias.data_ptr() if bias is not None else None, n_out, cols, ptrs, lds, _dtype_code(hidden), launches=1)
    return tuple(out)


def _rows_tma(t: torch.Tensor, rows: int, cols: int) -> torch.Tensor:
    # (rows, cols) view of a 16-bit gradient the library reads by TMA (unit column stride, 16-byte aligned base and rows)
    t2 = t.reshape(rows, cols)
    ok = t2.stride(1) == 1 and t2.data_ptr() % 16 == 0 and (rows == 1 or (t2.stride(0) >= cols and t2.stride(0) % 8 == 0))
    return t2 if ok else t2.contiguous()


def qkv_project_bwd(hidden: torch.Tensor, weight: torch.Tensor, dys: Sequence[torch.Tensor], need_hidden: bool = True,
                    need_weight: bool = True, need_bias: bool = False):
    """Gradients (dhidden, dweight, dbias) of qkv_project(hidden, weight, bias, len(dys)) for the output gradients dys,
    each None where not wanted (and then not computed): dY W, dY^T hidden and the column sums of dY, where dY is the
    dys side by side.  In the input dtype, as an fp16 / bf16 nn.Linear backward returns them: fp32 accumulation, one
    rounding; deterministic (split-K partials added in a fixed order, no atomics).  The dys are read in place."""
    import ctypes as C

    dev = _need_cuda(hidden, weight, *dys)
    c_in = hidden.shape[-1]
    n_out, n_t = weight.shape[0], len(dys)
    if weight.dim() != 2 or weight.shape[1] != c_in or weight.stride(1) != 1 or hidden.dtype != weight.dtype:
        raise RuntimeError(f"weight must be (n_out, {c_in}) with contiguous rows, of hidden's dtype")
    if n_t < 1 or n_out % n_t:
        raise RuntimeError("n_out must be a multiple of the number of output gradients")
    cols = n_out // n_t
    rows = hidden.numel() // c_in
    dx = torch.empty(hidden.shape, dtype=hidden.dtype, device=dev) if need_hidden else None
    dw = torch.empty((n_out, c_in), dtype=hidden.dtype, device=dev) if need_weight else None
    db = torch.empty(n_out, dtype=hidden.dtype, device=dev) if need_bias else None
    if rows == 0:   # nothing to add up: the weight and bias gradients are zero, the input gradient is empty
        return dx, None if dw is None else dw.zero_(), None if db is None else db.zero_()
    if dx is None and dw is None and db is None:
        return dx, dw, db
    d2 = [_rows_tma(d.to(hidden.dtype), rows, cols) for d in dys]
    h2 = hidden.reshape(rows, c_in) if need_weight else None
    if h2 is not None and h2.stride(1) != 1:
        h2 = h2.contiguous()
    ptrs = (C.c_void_p * n_t)(*[d.data_ptr() for d in d2])
    lds = (C.c_int64 * n_t)(*[d.stride(0) if rows > 1 else cols for d in d2])
    _call("ds_qkv_project_bwd", dev, None if h2 is None else h2.data_ptr(), rows, c_in if h2 is None else h2.stride(0),
          c_in, weight.data_ptr(), weight.stride(0), n_out, cols, ptrs, lds, None if dx is None else dx.data_ptr(), c_in,
          None if dw is None else dw.data_ptr(), c_in, None if db is None else db.data_ptr(), _dtype_code(hidden),
          ws_query=(rows, c_in, n_out, cols), slot="bwd",
          launches=2 * sum(g is not None for g in (dx, dw, db)))  # per wanted gradient: product or column sums + finish
    return dx, dw, db


class _QKVProjectFn(torch.autograd.Function):
    """qkv_project with the K4 backward; saves only the inputs.  The product runs on (weight, bias); with n_parts > 0 the
    gradients of their n_parts row blocks go to the trailing inputs (n_parts weights, then n_parts biases or None)."""

    @staticmethod
    def forward(ctx, n_outputs, n_parts, hidden, weight, bias, *parts):
        ctx.save_for_backward(hidden, weight)
        ctx.n_outputs, ctx.n_parts = n_outputs, n_parts
        return _qkv_project(hidden, weight, bias, n_outputs)

    @staticmethod
    def backward(ctx, *dys):
        hidden, weight = ctx.saved_tensors
        need = ctx.needs_input_grad
        n = ctx.n_parts
        w_need, b_need = need[5:5 + n], need[5 + n:]
        dx, dw, db = qkv_project_bwd(hidden, weight, dys, need[2], need[3] or any(w_need), need[4] or any(b_need))
        blk = weight.shape[0] // n if n else 0
        w_parts = [dw[i * blk:(i + 1) * blk] if w_need[i] else None for i in range(n)]
        b_parts = [db[i * blk:(i + 1) * blk] if b_need[i] else None for i in range(n)]
        return (None, None, dx, dw if need[3] else None, db if need[4] else None, *w_parts, *b_parts)


# --------------------------------------------------------------------------------------
# decisions
# --------------------------------------------------------------------------------------
def twoafc(ab: torch.Tensor, ac: torch.Tensor, similarity="cosine") -> Tuple[torch.Tensor, torch.Tensor]:
    """2AFC counts of the benchmark drivers (cute_main.py:196-205).  Returns (counts int32[2] = {correct,
    correct_2x}, flags uint8[n]) on the device -- one launch, no host sync."""
    dev = _need_cuda(ab, ac)
    ab = ab.to(torch.float32).contiguous()
    ac = ac.to(torch.float32).contiguous()
    n = ab.numel()
    counts = torch.empty(2, dtype=torch.int32, device=dev)
    flags = torch.empty(n, dtype=torch.uint8, device=dev)
    _call("ds_twoafc", dev, ab.data_ptr(), ac.data_ptr(), n, _mode(similarity), counts.data_ptr(), flags.data_ptr(),
          launches=1)
    return counts, flags


def profile_enable(on: bool = True) -> None:
    N.check(N.load().ds_profile_enable(1 if on else 0))


def profile_collect() -> Tuple[float, int]:
    """(summed device milliseconds, launches) of the attention kernel since the last call."""
    import ctypes as C

    ms, n = C.c_float(0.0), C.c_int(0)
    N.check(N.load().ds_profile_collect(C.byref(ms), C.byref(n)))
    return float(ms.value), int(n.value)


def default_scale(head_dim: int) -> float:
    return 1.0 / math.sqrt(head_dim)
