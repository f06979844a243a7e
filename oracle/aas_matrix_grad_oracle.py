"""Float64 model of the matrix backward ds_aas_matrix_bwd.  TEST INFRASTRUCTURE ONLY.

Dm[r, c] = sim(X_rc, Y_r), X_rc = Attn(q_r, k_c, v_c), Y_r = Attn(q_r, k_self_r, v_self_r).  The kernels fold the Nc
self terms of row r into one attention backward with dO = F_r = sum_c coef_self_rc fy_rc.  matrix_grads_rounded forms
the gradients as the kernels do, in float64, rounded where they round: X and Y as K1 stores them (given), fx per entry,
the folded F_r after its per-row power-of-two scale, and P, dS and delta as in aas_grad_oracle.attn_grads_rounded.  With
nothing rounded (float64 inputs, unrounded X and Y) it is the exact gradient of sum(d_Dm * Dm).
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import torch

from . import aas_grad_oracle as G


def _coefs(x: torch.Tensor, y: torch.Tensor, g: float, mode: str) -> Tuple[float, float, float]:
    """(c, k_X, k_Y) of g * sim(x, y) as sim_coef forms them: dX = c (Y - k_X X), dY = c (X - k_Y Y); MSE: k = 0
    and the factors are X - Y, Y - X."""
    if mode != "cosine":
        return 2.0 * g / x.numel(), 0.0, 0.0
    nx, ny = float(x.norm()), float(y.norm())
    cx, cy = max(nx, 1e-8), max(ny, 1e-8)
    cos = float((x * y).sum()) / (cx * cy)
    return g / (cx * cy), (cos * cy / cx if nx > 1e-8 else 0.0), (cos * cx / cy if ny > 1e-8 else 0.0)


def fold_factor(F: torch.Tensor, rnd: Optional[torch.dtype]) -> Tuple[torch.Tensor, float]:
    """(dO, coefficient) of a folded self term: F scaled by 2^-e with max |F| * 2^-e in [0.5, 1), rounded once."""
    m = float(F.abs().max())
    e = min(max(math.frexp(m)[1], -126), 127) if 0.0 < m < math.inf else 0
    return G._round(F * 2.0 ** -e, rnd), 2.0 ** e


def matrix_grads_rounded(q, k_self, v_self, k, v, X, Y, d_Dm, mode: str = "cosine",
                         scale: Optional[float] = None) -> Tuple[torch.Tensor, ...]:
    """(dq, dk_self, dv_self, dk, dv) of sum(d_Dm * Dm) as ds_aas_matrix_bwd forms them, in float64.  q, k_self, v_self:
    (Nr, B, H, S, D); k, v: (Nc, ...); X: (Nr, Nc, B, H, S, D) and Y: (Nr, ...) the attention outputs the kernels
    recompute.  Rounding is to q's dtype (none for float64 inputs)."""
    rnd = G._rounding_of(q)
    nr, nc = q.shape[0], k.shape[0]
    out = [torch.zeros(t.shape, dtype=torch.float64, device=t.device) for t in (q, k_self, v_self, k, v)]
    dq, dks, dvs, dk, dv = out
    for r in range(nr):
        y = Y[r].to(torch.float64)
        F = torch.zeros_like(y)
        for c in range(nc):
            x = X[r, c].to(torch.float64)
            cf, k_x, k_y = _coefs(x, y, float(d_Dm[r, c]), mode)
            fx = G._round(y - k_x * x if mode == "cosine" else x - y, rnd)
            F = F + cf * (x - k_y * y if mode == "cosine" else y - x)
            gq, gk, gv = G.attn_grads_rounded(q[r], k[c], v[c], x, fx, scale, rnd)
            dq[r] += cf * gq
            dk[c] += cf * gk
            dv[c] += cf * gv
        f16, s = fold_factor(F, rnd)
        gq, gk, gv = G.attn_grads_rounded(q[r], k_self[r], v_self[r], y, f16, scale, rnd)
        dq[r] += s * gq
        dks[r] += s * gk
        dvs[r] += s * gv
    return tuple(out)


def matrix_value(q, k_self, v_self, k, v, mode: str = "cosine", scale: Optional[float] = None,
                 round_to: Optional[torch.dtype] = None) -> torch.Tensor:
    """Dm [Nr, Nc] on float64 tensors, differentiable (T1 when round_to is the input dtype)."""
    rows = []
    for r in range(q.shape[0]):
        y = G.attention(q[r], k_self[r], v_self[r], scale, round_to)
        rows.append(torch.stack([G.similarity(G.attention(q[r], k[c], v[c], scale, round_to), y, mode)
                                 for c in range(k.shape[0])]))
    return torch.stack(rows)


def matrix_grads(q, k_self, v_self, k, v, d_Dm, mode: str = "cosine", scale: Optional[float] = None,
                 round_to: Optional[torch.dtype] = None) -> Tuple[torch.Tensor, ...]:
    """Float64 autograd of sum(d_Dm * Dm) w.r.t. (q, k_self, v_self, k, v) (a repeated input gets the sum of its
    slots' gradients in each of them)."""
    leaves = G._leaves(q, k_self, v_self, k, v)
    dm = matrix_value(*leaves, mode, scale, round_to)
    return torch.autograd.grad((dm * d_Dm.to(dm)).sum(), leaves)
