"""Float64 gradient oracle of the attention and of the Aligned Attention Score.  TEST INFRASTRUCTURE ONLY.

torch autograd of the T1 formulas of aas_oracle (float64 attention, outputs rounded to the input dtype, float64
reductions), with the rounding passed straight through (its gradient is taken as the identity, as the CUDA backward
does).  Works on any device: the GPU tests evaluate it there at full size.
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import torch


def _st_round(x: torch.Tensor, dtype: Optional[torch.dtype]) -> torch.Tensor:
    """x rounded to dtype in the forward, identity in the backward."""
    if dtype is None:
        return x
    return x + (x.to(dtype).to(x.dtype) - x).detach()


def attention(q, k, v, scale: Optional[float] = None, round_to: Optional[torch.dtype] = None) -> torch.Tensor:
    """softmax(q k^T scale) v in float64, differentiable; optionally rounded (straight through) to round_to."""
    sc = (1.0 / math.sqrt(q.shape[-1])) if scale is None else float(scale)
    s = torch.matmul(q, k.transpose(-1, -2)) * sc
    return _st_round(torch.matmul(torch.softmax(s, dim=-1), v), round_to)


def similarity(x: torch.Tensor, y: torch.Tensor, mode: str = "cosine", eps: float = 1e-8) -> torch.Tensor:
    """Flat cosine with torch's per-norm max(|.|, eps) clamp, or the mean squared difference."""
    x, y = x.reshape(-1), y.reshape(-1)
    if mode == "cosine":
        return (x * y).sum() / (x.norm().clamp_min(eps) * y.norm().clamp_min(eps))
    return ((x - y) ** 2).mean()


def _leaves(*ts):
    return [t.detach().to(torch.float64).requires_grad_(True) for t in ts]


def attn_grads(q, k, v, dout, scale: Optional[float] = None) -> Tuple[torch.Tensor, ...]:
    """(dq, dk, dv) of sum(attention(q, k, v) * dout) in float64."""
    q64, k64, v64 = _leaves(q, k, v)
    out = attention(q64, k64, v64, scale)
    return torch.autograd.grad(out, (q64, k64, v64), dout.to(torch.float64))


def dir_value(q_i, k_i, v_i, k_j, v_j, mode: str = "cosine", scale: Optional[float] = None,
              round_to: Optional[torch.dtype] = None) -> torch.Tensor:
    """sim(Attn(q_i, k_j, v_j), Attn(q_i, k_i, v_i)) on float64 tensors (T1 when round_to is the input dtype)."""
    return similarity(attention(q_i, k_j, v_j, scale, round_to), attention(q_i, k_i, v_i, scale, round_to), mode)


def pair_score_grads(qa, ka, va, qb, kb, vb, mode: str = "cosine", scale: Optional[float] = None,
                     g: float = 1.0) -> Tuple[torch.Tensor, ...]:
    """Float64 gradients of g * (dir(a->b) + dir(b->a)) / 2 with respect to (qa, ka, va, qb, kb, vb): the T1 pair
    score of aas_oracle.aas_pair_score, rounded like the inputs' dtype."""
    rnd = qa.dtype if qa.dtype in (torch.float16, torch.bfloat16) else None
    leaves = _leaves(qa, ka, va, qb, kb, vb)
    a_q, a_k, a_v, b_q, b_k, b_v = leaves
    s = (dir_value(a_q, a_k, a_v, b_k, b_v, mode, scale, rnd) + dir_value(b_q, b_k, b_v, a_k, a_v, mode, scale, rnd)) / 2
    return torch.autograd.grad(s * g, leaves)
