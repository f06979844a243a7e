"""Float64 gradient oracle of the QKV projection (K4 backward).  TEST INFRASTRUCTURE ONLY.

For y = hidden W^T (+ bias) split into column blocks dY = [dy_0 | dy_1 | ...]:
    dhidden = dY W,   dweight = dY^T hidden,   dbias = sum over rows of dY
in float64, with the matching sums of |products| that bound what fp32 accumulation in any order can be off by (the
weight gradient's long sums over all tokens cancel, so a tolerance relative to the result alone would not do).

capture_chain_grads is the float64 chain hook input -> projection (rounded straight through to the input dtype, as K4
rounds) -> head split -> pair score, whose gradients the end-to-end tests compare with.
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import torch

from . import aas_grad_oracle as G


def qkv_bwd(hidden: torch.Tensor, weight: torch.Tensor, dys: Sequence[torch.Tensor]):
    """((dhidden, dweight, dbias), (|dY| |W|, |dY|^T |hidden|, sum |dY|)) in float64; hidden (..., C_in) flattened to
    rows, weight (n_out, C_in), dys the output gradients (..., n_out / len(dys))."""
    c_in = hidden.shape[-1]
    x = hidden.reshape(-1, c_in).to(torch.float64)
    w = weight.to(torch.float64)
    dy = torch.cat([d.reshape(x.shape[0], -1).to(torch.float64) for d in dys], dim=1)
    grads = (dy @ w, dy.t() @ x, dy.sum(0))
    a = dy.abs()
    bounds = (a @ w.abs(), a.t() @ x.abs(), a.sum(0))
    return grads, bounds


def capture_chain_grads(xa: torch.Tensor, xb: torch.Tensor, weights: Sequence[torch.Tensor], heads: int,
                        mode: str = "cosine", g: float = 1.0, biases: Optional[Sequence[torch.Tensor]] = None
                        ) -> Tuple[torch.Tensor, ...]:
    """Float64 gradients (dxa, dxb, dW_q, dW_k, dW_v[, db_q, db_k, db_v]) of g * pair_score for two hook inputs
    (B, S, C) projected by the three weights (and biases): q/k/v rounded to the input dtype straight through, split into
    `heads` heads, then aas_grad_oracle's T1 pair score."""
    rnd = xa.dtype if xa.dtype in (torch.float16, torch.bfloat16) else None
    leaves = G._leaves(xa, xb, *weights, *(biases or ()))
    a, b, ws = leaves[0], leaves[1], leaves[2:5]
    bs = leaves[5:] if biases else [None] * 3

    def qkv(x):
        out = []
        for w, bias in zip(ws, bs):
            y = x @ w.t() + (bias if bias is not None else 0.0)
            y = G._st_round(y, rnd)
            B, S, C = y.shape
            out.append(y.view(B, S, heads, C // heads).transpose(1, 2))
        return out

    qa, ka, va = qkv(a)
    qb, kb, vb = qkv(b)
    s = (G.dir_value(qa, ka, va, kb, vb, mode, None, rnd) + G.dir_value(qb, kb, vb, ka, va, mode, None, rnd)) / 2
    return torch.autograd.grad(s * g, leaves)
