"""Float64 gradient oracle of the similarity reductions (K2 backward).  TEST INFRASTRUCTURE ONLY.

pair_reduce_grads is the closed form of the gradients of out[p] = sim(x[p], y[p]) for dL/dout = g, row by row:
    cosine  s = x.y / (nx ny), n = max(|.|, 1e-8):  dx = g (y / (nx ny) - s x / (nx |x|)), the second term 0 when |x| = 0
    mse     dx = 2 g (x - y) / E,  dy = -dx
    minmax  x^ = (x - m) / (M - m), G = dcos/dx^ by the cosine rule:
            dx = g (G / (M - m) + [x = m] S_m / n_m + [x = M] S_M / n_M),
            S_m = sum G (x^ - 1) / (M - m),  S_M = -sum G x^ / (M - m),  n_m, n_M the numbers of ties
and dy symmetric.  autograd_grads is float64 torch autograd of the reference's own expressions (F.cosine_similarity on
the flattened rows, F.mse_loss, min_max_normalize + cosine), which the closed form must equal.  Both work on any device.
"""
from __future__ import annotations

from typing import Tuple

import torch
import torch.nn.functional as F

EPS = 1e-8


def _cosine_parts(x: torch.Tensor, y: torch.Tensor, unclamped: bool = True):
    """(dcos/dx, dcos/dy) per row of float64 (P, E) tensors.  unclamped=False puts the clamped norm in the second term
    in place of |x| (a wrong form, for the tests' mutants)."""
    ex, ey = x.norm(dim=1), y.norm(dim=1)
    nx, ny = ex.clamp_min(EPS), ey.clamp_min(EPS)
    s = (x * y).sum(1) / (nx * ny)
    axy = 1.0 / (nx * ny)
    zero = torch.zeros_like(s)
    if unclamped:
        axx = torch.where(ex > 0, s / (nx * ex), zero)
        ayy = torch.where(ey > 0, s / (ny * ey), zero)
    else:
        axx, ayy = s / (nx * nx), s / (ny * ny)
    return axy[:, None] * y - axx[:, None] * x, axy[:, None] * x - ayy[:, None] * y


def _minmax_side(t: torch.Tensor, G: torch.Tensor, c: torch.Tensor, th: torch.Tensor, split_ties: bool,
                 minmax_terms: bool) -> torch.Tensor:
    d = G / c[:, None]
    if not minmax_terms:
        return d
    at_min = t == t.amin(1, keepdim=True)
    at_max = t == t.amax(1, keepdim=True)
    s_m = (G * (th - 1)).sum(1) / c
    s_M = -(G * th).sum(1) / c
    n_m = at_min.sum(1) if split_ties else torch.ones_like(c)
    n_M = at_max.sum(1) if split_ties else torch.ones_like(c)
    return d + at_min * (s_m / n_m)[:, None] + at_max * (s_M / n_M)[:, None]


def _grads(x, y, g, mode: str = "cosine", split_ties: bool = True, minmax_terms: bool = True, unclamped: bool = True):
    P = x.shape[0]
    x = x.reshape(P, -1).to(torch.float64)
    y = y.reshape(P, -1).to(torch.float64)
    g = g.reshape(P, 1).to(device=x.device, dtype=torch.float64)
    if mode == "mse":
        dx = 2.0 * g * (x - y) / x.shape[1]
        return dx, -dx
    if mode == "cosine":
        gx, gy = _cosine_parts(x, y, unclamped)
        return g * gx, g * gy
    mx, my = x.amin(1), y.amin(1)
    cx, cy = x.amax(1) - mx, y.amax(1) - my
    xh, yh = (x - mx[:, None]) / cx[:, None], (y - my[:, None]) / cy[:, None]
    gx, gy = _cosine_parts(xh, yh, unclamped)
    return (g * _minmax_side(x, gx, cx, xh, split_ties, minmax_terms),
            g * _minmax_side(y, gy, cy, yh, split_ties, minmax_terms))


def pair_reduce_grads(x: torch.Tensor, y: torch.Tensor, g: torch.Tensor, mode: str = "cosine"
                      ) -> Tuple[torch.Tensor, torch.Tensor]:
    """float64 (dx, dy) of out[p] = sim(x[p], y[p]) for dL/dout = g ([P]); x, y (P, ...) flattened to rows (P, E)."""
    return _grads(x, y, g, mode)


def reference_score(x: torch.Tensor, y: torch.Tensor, mode: str = "cosine") -> torch.Tensor:
    """The reference's expression on one pair of (flattened) rows, differentiable."""
    x, y = x.reshape(-1), y.reshape(-1)
    if mode == "cosine":
        return F.cosine_similarity(x.unsqueeze(0), y.unsqueeze(0))[0]
    if mode == "mse":
        return F.mse_loss(x, y)

    def min_max_normalize(t):   # metrics/diffeats.py:136-140
        return (t - t.min()) / (t.max() - t.min())

    return F.cosine_similarity(min_max_normalize(x).unsqueeze(0), min_max_normalize(y).unsqueeze(0))[0]


def autograd_grads(x: torch.Tensor, y: torch.Tensor, g: torch.Tensor, mode: str = "cosine"
                   ) -> Tuple[torch.Tensor, torch.Tensor]:
    """float64 torch autograd of sum_p g[p] reference_score(x[p], y[p], mode), as (P, E) tensors."""
    P = x.shape[0]
    x64 = x.detach().reshape(P, -1).to(torch.float64).requires_grad_(True)
    y64 = y.detach().reshape(P, -1).to(torch.float64).requires_grad_(True)
    g64 = g.detach().reshape(-1).to(device=x64.device, dtype=torch.float64)
    loss = sum(g64[p] * reference_score(x64[p], y64[p], mode) for p in range(P))
    return torch.autograd.grad(loss, (x64, y64))


# Per-row relative tolerance of the K2 backward against this oracle: |got - ref| / max(|ref|, cross_term_norms) over
# each row of dx and dy (fp32 arithmetic on exact inputs; rows whose reference is NaN must be NaN).  Worst seen over
# tests/test_gpu_reduce_grad.py on a B200: 1.7e-6 (minmax, bf16, 1 x 655 360); cosine 3.7e-7, mse 6e-8.
ROW_TOL = 1e-5


def cross_term_norms(x: torch.Tensor, y: torch.Tensor, g: torch.Tensor, mode: str = "cosine"):
    """Per-row norms of the term of dx (dy) that the other operand drives -- g y / (nx ny) for the cosine, on the
    normalised rows and over (M - m) for minmax, the whole 2 g (x - y) / E for mse: the scale of a row's gradient
    when the gradient itself cancels to ~0 (a row at its maximum similarity).  row_errors' denominator floor."""
    P = x.shape[0]
    x = x.reshape(P, -1).to(torch.float64)
    y = y.reshape(P, -1).to(device=x.device, dtype=torch.float64)
    g = g.reshape(-1).to(device=x.device, dtype=torch.float64).abs()
    if mode == "mse":
        n = 2.0 * g * (x - y).norm(dim=1) / x.shape[1]
        return n, n
    cx = cy = torch.ones_like(g)
    if mode != "cosine":
        cx, cy = x.amax(1) - x.amin(1), y.amax(1) - y.amin(1)
        x, y = (x - x.amin(1, keepdim=True)) / cx[:, None], (y - y.amin(1, keepdim=True)) / cy[:, None]
    ex, ey = x.norm(dim=1), y.norm(dim=1)
    d = ex.clamp_min(EPS) * ey.clamp_min(EPS)
    return g * ey / (d * cx), g * ex / (d * cy)


def row_errors(got: torch.Tensor, ref: torch.Tensor, floor: torch.Tensor = None) -> torch.Tensor:
    """Per-row relative error |got - ref| / max(|ref|, floor) of (P, E) tensors (0 where both rows are 0, inf where
    only the denominator is); rows where ref has a NaN are left out (NaN in the result)."""
    P = ref.shape[0]
    got = got.reshape(P, -1).to(torch.float64)
    ref = ref.reshape(P, -1).to(device=got.device, dtype=torch.float64)
    bad = ref.isnan().any(1)
    err = (got - ref).norm(dim=1)
    den = ref.norm(dim=1)
    if floor is not None:
        den = torch.maximum(den, floor.to(den.device).nan_to_num(0))
    out = torch.where(den > 0, err / den.clamp_min(1e-300), torch.where(err > 0, torch.inf, 0.0))
    return torch.where(bad, torch.nan, out)
