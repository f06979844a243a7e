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


def _count(n: int) -> None:
    global LAUNCHES
    LAUNCHES += n


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


def _stream(dev: torch.device) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


def _dtype_code(t: torch.Tensor) -> int:
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise RuntimeError(f"unsupported dtype {t.dtype}") from None


def _t4(t: torch.Tensor) -> N.Tensor4:
    if t.dim() != 4:
        raise RuntimeError(f"expected a (B,H,S,D) tensor, got shape {tuple(t.shape)}")
    d = N.Tensor4()
    d.ptr = t.data_ptr()
    d.size[:] = list(t.shape)
    d.stride[:] = list(t.stride())
    d.dtype = _dtype_code(t)
    return d


def _t5(t: torch.Tensor) -> N.Tensor5:
    if t.dim() != 5:
        raise RuntimeError(f"expected a (N,B,H,S,D) tensor, got shape {tuple(t.shape)}")
    d = N.Tensor5()
    d.ptr = t.data_ptr()
    d.size[:] = list(t.shape)
    d.stride[:] = list(t.stride())
    d.dtype = _dtype_code(t)
    return d


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
    lib = N.load()
    dev = _need_cuda(q, k, v)
    B, H, Sq, D = q.shape
    if out is None:
        out = torch.empty((B, Sq, H, D), dtype=q.dtype, device=dev).permute(0, 2, 1, 3)
    q4, k4 = _t4(q), _t4(k)
    nbytes = lib.ds_attn_fwd_workspace_bytes(q4, k4)
    ws = _workspace(dev, nbytes)
    with torch.cuda.device(dev):
        N.check(lib.ds_attn_fwd(q4, k4, _t4(v), float(scale) if scale else 0.0, _t4(out), ws.data_ptr(), ws.numel(),
                                _stream(dev)))
    _count(2)  # meta + attention
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
    lib = N.load()
    dev = _need_cuda(q, k, v, out, dout)
    dout = _tma_ok(dout.to(q.dtype))
    dq, dk, dv = _grads_like((q, k, v), grads)
    q4, k4 = _t4(q), _t4(k)
    ws = _workspace(dev, lib.ds_attn_bwd_workspace_bytes(q4, k4), "bwd")
    with torch.cuda.device(dev):
        N.check(lib.ds_attn_bwd(q4, k4, _t4(v), _t4(out), _t4(dout), float(scale) if scale else 0.0, _t4(dq), _t4(dk),
                                _t4(dv), ws.data_ptr(), ws.numel(), _stream(dev)))
    _count(2)  # dQ + dK/dV
    return dq, dk, dv


def aas_dir_bwd(q_i: torch.Tensor, k_i: torch.Tensor, v_i: torch.Tensor, k_j: torch.Tensor, v_j: torch.Tensor,
                d_dir: torch.Tensor, similarity="cosine", scale: Optional[float] = None,
                grads: Optional[Sequence[torch.Tensor]] = None) -> Tuple[torch.Tensor, ...]:
    """Gradients (dq_i, dk_i, dv_i, dk_j, dv_j) of dir = sim(Attn(q_i,k_j,v_j), Attn(q_i,k_i,v_i)) for dL/ddir = d_dir
    (a one-element tensor on the device; no host sync), in float32.  (B,H,S,D) inputs as for attn_fwd.
    grads: optional float32 tensors to add into (they may alias, e.g. dk_i is dk_j when image i is image j)."""
    lib = N.load()
    dev = _need_cuda(q_i, k_i, v_i, k_j, v_j, d_dir)
    g = d_dir.detach().reshape(-1).to(torch.float32)
    if g.numel() != 1:
        raise RuntimeError("d_dir must have exactly one element")
    out = _grads_like((q_i, k_i, v_i, k_j, v_j), grads)
    q4, kj4 = _t4(q_i), _t4(k_j)
    ws = _workspace(dev, lib.ds_aas_dir_bwd_workspace_bytes(q4, kj4), "bwd")
    with torch.cuda.device(dev):
        N.check(lib.ds_aas_dir_bwd(q4, _t4(k_i), _t4(v_i), kj4, _t4(v_j), float(scale) if scale else 0.0,
                                   _mode(similarity), g.data_ptr(), *[_t4(t) for t in out], ws.data_ptr(), ws.numel(),
                                   _stream(dev)))
    _count(11)  # 2 x (meta + attention) recompute + partials + coefficients + factors + 2 x (dQ + dK/dV)
    return out


def _pair_dirs(qa, ka, va, qb, kb, vb, similarity, scale):
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
    """(dir(a->b), dir(b->a)) of one image pair as float32 (1,) tensors -- two aas_groups launches.  Differentiable
    (aas_dir_bwd) when an input requires grad; the values are the same either way."""
    if wants_grad(qa, ka, va, qb, kb, vb):
        return _PairDirsFn.apply(similarity, scale, qa, ka, va, qb, kb, vb)
    return _pair_dirs(qa, ka, va, qb, kb, vb, similarity, scale)


def aas_groups(q: torch.Tensor, k_self: torch.Tensor, v_self: torch.Tensor, k: torch.Tensor, v: torch.Tensor,
               group_q, group_off, kv_idx, similarity="cosine", scale: Optional[float] = None) -> torch.Tensor:
    """Directional AAS similarities for grouped (query image, kv image list) work -- see ds_aas_groups.
    q/k_self/v_self: (Nq,B,H,S,D); k/v: (Nk,B,H,S,D).  Returns float32 [n_entries]."""
    lib = N.load()
    dev = _need_cuda(q, k_self, v_self, k, v)
    gq, go, kv = _i32(group_q, dev), _i32(group_off, dev), _i32(kv_idx, dev)
    n_groups, n_entries = gq.numel(), kv.numel()
    if go.numel() != n_groups + 1:
        raise RuntimeError("group_off must have n_groups + 1 entries")
    dirs = torch.empty(n_entries, dtype=torch.float32, device=dev)
    q5 = _t5(q)
    nbytes = lib.ds_aas_groups_workspace_bytes(q5, n_groups, n_entries)
    ws = _workspace(dev, nbytes)
    with torch.cuda.device(dev):
        N.check(lib.ds_aas_groups(q5, _t5(k_self), _t5(v_self), _t5(k), _t5(v), gq.data_ptr(), go.data_ptr(), n_groups,
                                  kv.data_ptr(), n_entries, float(scale) if scale else 0.0, _mode(similarity),
                                  dirs.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev)))
    _count(3)  # index validation + attention + finish
    return dirs


def aas_pairs(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, pair_idx, similarity="cosine",
              scale: Optional[float] = None) -> torch.Tensor:
    """score[p] = (dir(a->b) + dir(b->a)) / 2 for pair_idx[p] = (a, b): the value DiffSim.diffsim returns
    (diffsim/diffsim.py:177-197).  q,k,v: (N,B,H,S,D) caches.  Returns float32 [P]."""
    lib = N.load()
    dev = _need_cuda(q, k, v)
    pairs = _i32(pair_idx, dev).reshape(-1, 2)
    P = pairs.shape[0]
    scores = torch.empty(P, dtype=torch.float32, device=dev)
    q5 = _t5(q)
    nbytes = lib.ds_aas_pairs_workspace_bytes(q5, P)
    ws = _workspace(dev, nbytes)
    with torch.cuda.device(dev):
        N.check(lib.ds_aas_pairs(q5, _t5(k), _t5(v), pairs.data_ptr(), P, float(scale) if scale else 0.0,
                                 _mode(similarity), scores.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev)))
    _count(5)  # setup + index validation + attention + finish + pair combine
    return scores


def aas_triplets(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, trip_idx, similarity="cosine",
                 scale: Optional[float] = None, round_scores: bool = False, want_flags: bool = True):
    """2AFC triplets (ref, left, right) as the benchmark drivers score them (cute_main.py:111-132,196-205):
    returns (ab, ac, counts, flags) on the device: ab = diffsim(ref,left), ac = diffsim(ref,right) (float32 [T]),
    counts int32[2] = {correct, correct_2x}, flags uint8[T].  One library call, no host sync."""
    lib = N.load()
    dev = _need_cuda(q, k, v)
    trips = _i32(trip_idx, dev).reshape(-1, 3)
    T = trips.shape[0]
    ab = torch.empty(T, dtype=torch.float32, device=dev)
    ac = torch.empty(T, dtype=torch.float32, device=dev)
    counts = torch.empty(2, dtype=torch.int32, device=dev)
    flags = torch.empty(T, dtype=torch.uint8, device=dev) if want_flags else None
    q5 = _t5(q)
    nbytes = lib.ds_aas_triplets_workspace_bytes(q5, T)
    ws = _workspace(dev, nbytes)
    with torch.cuda.device(dev):
        N.check(lib.ds_aas_triplets(q5, _t5(k), _t5(v), trips.data_ptr(), T, float(scale) if scale else 0.0,
                                    _mode(similarity), N.DS_OPT_ROUND_SCORES if round_scores else 0, ab.data_ptr(),
                                    ac.data_ptr(), counts.data_ptr(), flags.data_ptr() if want_flags else None,
                                    ws.data_ptr(), ws.numel(), _stream(dev)))
    _count(5)  # setup + index validation + attention + finish + combine/decide
    return ab, ac, counts, flags


def aas_matrix(q: torch.Tensor, k_self: torch.Tensor, v_self: torch.Tensor, k: torch.Tensor, v: torch.Tensor,
               similarity="cosine", scale: Optional[float] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Directional matrix Dm[r,c] = dir(row image r -> column image c); rows (q,k_self,v_self): (Nr,...),
    columns (k,v): (Nc,...).  Returns float32 [Nr,Nc]."""
    lib = N.load()
    dev = _need_cuda(q, k_self, v_self, k, v)
    nr, nc = q.shape[0], k.shape[0]
    if out is None:
        out = torch.empty((nr, nc), dtype=torch.float32, device=dev)
    q5, k5 = _t5(q), _t5(k)
    nbytes = lib.ds_aas_matrix_workspace_bytes(q5, k5)
    ws = _workspace(dev, nbytes)
    with torch.cuda.device(dev):
        N.check(lib.ds_aas_matrix(q5, _t5(k_self), _t5(v_self), k5, _t5(v), float(scale) if scale else 0.0,
                                  _mode(similarity), out.data_ptr(), out.stride(0), ws.data_ptr(), ws.numel(),
                                  _stream(dev)))
    _count(3)  # setup + attention + finish
    return out


# --------------------------------------------------------------------------------------
# K2: reductions
# --------------------------------------------------------------------------------------
def pair_reduce(x: torch.Tensor, y: torch.Tensor, similarity="cosine") -> torch.Tensor:
    """sim(x[p], y[p]) over the flattened trailing dims, for every leading row p.  x, y: (P, ...) tensors whose rows
    are contiguous.  Replaces F.cosine_similarity on flattened tensors / F.mse_loss / min-max + cosine
    (diffsim/diffsim.py:182-195, metrics/diffeats.py:136-140,202-205).  Returns float32 [P]."""
    lib = N.load()
    dev = _need_cuda(x, y)
    if x.shape != y.shape or x.dtype != y.dtype:
        raise RuntimeError("x and y must have the same shape and dtype")
    P = x.shape[0]
    if P == 0:
        return torch.empty(0, dtype=torch.float32, device=dev)
    x2, y2 = x.reshape(P, -1), y.reshape(P, -1)
    if x2.stride(1) != 1:
        x2 = x2.contiguous()
    if y2.stride(1) != 1:
        y2 = y2.contiguous()
    E = x2.shape[1]
    out = torch.empty(P, dtype=torch.float32, device=dev)
    nbytes = lib.ds_pair_reduce_workspace_bytes(P, E)
    ws = _workspace(dev, nbytes)
    with torch.cuda.device(dev):
        N.check(lib.ds_pair_reduce(x2.data_ptr(), y2.data_ptr(), P, E, x2.stride(0) if P > 1 else E,
                                   y2.stride(0) if P > 1 else E, _dtype_code(x2), _mode(similarity), out.data_ptr(),
                                   ws.data_ptr(), ws.numel(), _stream(dev)))
    _count(1)
    return out


# --------------------------------------------------------------------------------------
# K3: N x N feature similarity matrix
# --------------------------------------------------------------------------------------
def simmat(rows: torch.Tensor, cols: Optional[torch.Tensor] = None, similarity="cosine",
           out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """C[r,c] = sim(rows[r], cols[c]) for 16-bit feature matrices rows (Nr,L), cols (Nc,L) (default cols = rows)."""
    lib = N.load()
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
    nbytes = lib.ds_simmat_workspace_bytes(nr, nc, L)
    ws = _workspace(dev, nbytes)
    with torch.cuda.device(dev):
        N.check(lib.ds_simmat(rows.data_ptr(), nr, rows.stride(0), cols.data_ptr(), nc, cols.stride(0), L,
                              _dtype_code(rows), _mode(similarity), out.data_ptr(), out.stride(0), ws.data_ptr(),
                              ws.numel(), _stream(dev)))
    # statistics pass + its finish per operand (one operand when rows is cols: the symmetric call), GEMM, normalise
    _count(4 if (cols.data_ptr() == rows.data_ptr() and nr == nc and cols.stride(0) == rows.stride(0)) else 6)
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
    `out`: optional pre-allocated outputs (row stride may exceed the column count, e.g. slices of a cache)."""
    import ctypes as C

    lib = N.load()
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
    with torch.cuda.device(dev):
        N.check(lib.ds_qkv_project(h2.data_ptr(), rows, h2.stride(0), c_in, weight.data_ptr(), weight.stride(0),
                                   bias.data_ptr() if bias is not None else None, n_out, cols, ptrs, lds,
                                   _dtype_code(hidden), _stream(dev)))
    _count(1)
    return tuple(out)


# --------------------------------------------------------------------------------------
# decisions
# --------------------------------------------------------------------------------------
def twoafc(ab: torch.Tensor, ac: torch.Tensor, similarity="cosine") -> Tuple[torch.Tensor, torch.Tensor]:
    """2AFC counts of the benchmark drivers (cute_main.py:196-205).  Returns (counts int32[2] = {correct,
    correct_2x}, flags uint8[n]) on the device -- one launch, no host sync."""
    lib = N.load()
    dev = _need_cuda(ab, ac)
    ab = ab.to(torch.float32).contiguous()
    ac = ac.to(torch.float32).contiguous()
    n = ab.numel()
    counts = torch.empty(2, dtype=torch.int32, device=dev)
    flags = torch.empty(n, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        N.check(lib.ds_twoafc(ab.data_ptr(), ac.data_ptr(), n, _mode(similarity), counts.data_ptr(), flags.data_ptr(),
                              _stream(dev)))
    _count(1)
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
