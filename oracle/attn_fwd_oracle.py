"""Float64 model of the K1 attention forward and its fused score epilogue.  TEST INFRASTRUCTURE ONLY.

attention_model follows the arithmetic of aas_attn_kernel (csrc/ds_attn.cu) step by step:
- scale: sl2 = fp32(fp32(scale) * fp32(log2 e)), the default scale 1.0f / sqrtf(D) in fp32;
- S = q k^T in fp32, cut into consecutive 128-column halves of the kv rows;
- the lazy running maximum: half 0 of an item fixes m = fp32(max(s) * sl2); a later half only moves it (rescaling O and
  l by exp2(m - Mh)) when its own maximum Mh exceeds m by more than tau = 14 (fp16) or 30 (bf16), so P reaches 2^tau;
- P = r16(exp2(fp32(s * sl2 - m))), r16 rounding to the input dtype; at D <= 80 the columns c with
  ((c mod 32) >> 1) mod 3 == 0 take the kernel's degree-3 polynomial (emulated bit for bit), the others ex2.approx
  (taken as exact);
- l = sum r16(P) (the tensor core's row sum against a ones tile), O = sum r16(P) v, out = r16(O * fp32(1 / l)).
dir_model adds the score epilogue: the self output is rounded to the input dtype and the norms and the cosine's dot
product take the unrounded outputs; the MSE rounds both.

Everything else is float64, so a correct kernel differs from the model only by fp32 accumulation (in the tensor core and
in the epilogue) and by the occasional 16-bit rounding that an fp32-versus-float64 difference flips.  With float64
inputs nothing is rounded and the model is the exact attention of aas_oracle.  Works on any device: the GPU tests
evaluate it there at full size.
"""
from __future__ import annotations

import math
from typing import Optional

import numpy as np
import torch

KV_HALF = 128                                     # kv columns per S half
TAU = {torch.float16: 14.0, torch.bfloat16: 30.0}  # log2 headroom of the lazy maximum
LOG2E = float(np.float32(1.4426950408889634))
# exp2_poly_f2 (csrc/ds_ptx.cuh): 2^f ~ ((C3 f + C2) f + C1) f + C0 on |f| <= 0.5, coefficients as fp32
POLY = tuple(float(np.float32(c)) for c in (0.05517144873738289, 0.2426108419895172, 0.6932609677314758,
                                            0.9999281167984009))
POLY_MAX_REL = 7.5e-5                             # the polynomial's relative error as the kernel comment states it


def _r32(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.float32).to(torch.float64)


def r16(x: torch.Tensor, dtype: Optional[torch.dtype]) -> torch.Tensor:
    """x rounded to nearest in dtype (None: unchanged), returned in float64."""
    return x if dtype is None else x.to(dtype).to(torch.float64)


def _rounding_of(t: torch.Tensor) -> Optional[torch.dtype]:
    return t.dtype if t.dtype in (torch.float16, torch.bfloat16) else None


def kernel_scale(D: int, scale: Optional[float] = None) -> float:
    """The softmax scale as the host passes it to the kernel: fp32(scale), or 1.0f / sqrtf(D) when scale is None or
    not positive."""
    if scale is None or not scale > 0:
        return float(np.float32(1.0) / np.sqrt(np.float32(D)))
    return float(np.float32(scale))


def exp2_poly(x: torch.Tensor) -> torch.Tensor:
    """exp2_poly_f2 on fp32 values x (held in float64): Cody-Waite split x = j + f with j = round-to-nearest-even(x),
    the Horner steps as fp32 FMAs, 2^j added into the exponent.  Inputs below -126 are clamped as in the kernel."""
    x = x.clamp_min(-126.0)
    j = torch.round(x)
    f = x - j
    c3, c2, c1, c0 = POLY
    p = _r32(f * c3 + c2)
    p = _r32(p * f + c1)
    p = _r32(p * f + c0)
    return torch.ldexp(p, j)


def poly_columns(n: int, D: int, device=None) -> torch.Tensor:
    """Mask of the columns of an n-column S half that K1 exponentiates with the polynomial (head dims <= 80)."""
    c = torch.arange(n, device=device)
    return (((c % 32) >> 1) % 3 == 0) & (D <= 80)


def attention_model(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, scale: Optional[float] = None,
                    *, l_from_fp32_p: bool = False):
    """K1's attention (B,H,Sq,D) x (B,H,Skv,D) as described in the module docstring.  Returns (o, out, rescales):
    o the float64 output before its final rounding, out = r16(o) in float64, rescales the number of times the running
    maximum moved per (b, h, row) (an int64 (B,H,Sq) tensor).  Float64 inputs: no rounding anywhere and exact exp2, so
    o is the exact attention.  l_from_fp32_p takes l from the unrounded P (a kernel mistake the tests must catch)."""
    rnd = _rounding_of(q)
    D, Skv = q.shape[-1], k.shape[-2]
    q64, k64, v64 = (t.to(torch.float64) for t in (q, k, v))
    if rnd is None:
        sl2 = ((1.0 / math.sqrt(D)) if scale is None or not scale > 0 else float(scale)) * (1.0 / math.log(2.0))
        tau, f32 = 14.0, (lambda t: t)  # noqa: E731
    else:
        sl2 = float(np.float32(kernel_scale(D, scale)) * np.float32(LOG2E))
        tau, f32 = TAU[rnd], _r32
    s = f32(torch.matmul(q64, k64.transpose(-1, -2)))
    O = torch.zeros(q.shape[:-1] + (v.shape[-1],), dtype=torch.float64, device=q.device)
    l = torch.zeros(q.shape[:-1], dtype=torch.float64, device=q.device)
    m = None
    rescales = torch.zeros(q.shape[:-1], dtype=torch.int64, device=q.device)
    for h0 in range(0, Skv, KV_HALF):
        sh = s[..., h0:h0 + KV_HALF]
        mh = f32(sh.amax(dim=-1) * sl2)
        if m is None:
            m = mh
        else:
            up = mh > m + tau
            alpha = torch.where(up, torch.exp2(f32(m - mh)), torch.ones_like(m))
            O, l = O * alpha[..., None], l * alpha
            m = torch.where(up, mh, m)
            rescales += up.to(torch.int64)
        x = f32(sh * sl2 - m[..., None])
        e = torch.exp2(x)
        if rnd is not None:
            e = torch.where(x < -126.0, torch.zeros_like(e), e)   # ex2.approx.ftz: subnormal results are flushed
            poly = poly_columns(sh.shape[-1], D, sh.device)
            e = torch.where(poly, exp2_poly(x), e)
        p = r16(e, rnd)
        l = l + (e if l_from_fp32_p else p).sum(dim=-1)
        O = O + torch.matmul(p, v64[..., h0:h0 + KV_HALF, :])
    o = O * (f32(1.0 / l) if rnd is not None else 1.0 / l)[..., None]
    return o, r16(o, rnd), rescales


def scores_from_outputs(xc: torch.Tensor, xc16: torch.Tensor, ys: torch.Tensor, ys16: torch.Tensor, mode: str) -> float:
    """K1's score epilogue on float64 outputs: cosine = sum(xc * ys16) / (max(|xc|, 1e-8) max(|ys|, 1e-8)) with the
    unrounded cross output xc against the rounded self output ys16 and unrounded norms; MSE = mean (xc16 - ys16)^2."""
    if mode == "cosine":
        nx = max(math.sqrt(float(xc.square().sum())), 1e-8)
        ny = max(math.sqrt(float(ys.square().sum())), 1e-8)
        return float((xc * ys16).sum()) / (nx * ny)
    return float((xc16 - ys16).square().sum()) / xc16.numel()


def dir_model(q_i, k_i, v_i, k_j, v_j, mode: str = "cosine", scale: Optional[float] = None) -> float:
    """dir(i -> j) = sim(Attn(q_i, k_j, v_j), Attn(q_i, k_i, v_i)) as K1's score epilogue computes it; k_i and k_j may
    differ in length."""
    xc, xc16, _ = attention_model(q_i, k_j, v_j, scale)
    ys, ys16, _ = attention_model(q_i, k_i, v_i, scale)
    return scores_from_outputs(xc, xc16, ys, ys16, mode)


# ----------------------------------------------------------------------------------------------------------------------
# error metrics shared by the GPU tests and the CPU mutant table
# ----------------------------------------------------------------------------------------------------------------------
MANTISSA = {torch.float16: 10, torch.bfloat16: 7}


def ulp_error(got: torch.Tensor, o: torch.Tensor, dtype: torch.dtype) -> float:
    """Largest |got - o| in 16-bit ulps of max(|o|, 0.1 rms of o's row): o is the model's unrounded output, so a
    correct kernel sits near 0.5 ulp plus flips.  A flip is a P that ex2.approx or the tensor core's fp32 S puts on the
    other side of a 16-bit rounding boundary than the model's: it moves the row by one ulp of that P times v / l, which
    at the small elements of a row with a large P is several ulps of the element (up to 14 observed in fp16)."""
    o = o.to(torch.float64)
    rms = o.square().mean(dim=-1, keepdim=True).sqrt()
    mag = torch.maximum(o.abs(), 0.1 * rms)
    if dtype == torch.float16:
        mag = mag.clamp_min(2.0 ** -14)   # fp16's subnormal range has a fixed ulp
    ulp = torch.exp2(torch.floor(torch.log2(mag.clamp_min(1e-300))) - MANTISSA[dtype])
    err = (got.to(torch.float64) - o).abs()
    return float(torch.where(err == 0, torch.zeros_like(err), err / ulp).max())


def mismatch_fraction(got: torch.Tensor, out: torch.Tensor) -> float:
    """Fraction of elements where got differs from the model's rounded output: a global scale error moves most of them,
    in bf16 too."""
    return float((got.to(torch.float64) != out.to(torch.float64)).double().mean())


def rel_fro(got: torch.Tensor, ref: torch.Tensor) -> float:
    """Relative Frobenius error; an all-zero reference must be matched exactly."""
    e = float((got.to(torch.float64) - ref.to(torch.float64)).norm())
    n = float(ref.to(torch.float64).norm())
    return e / n if n > 0 else (0.0 if e == 0 else float("inf"))


def row_error(got: torch.Tensor, out: torch.Tensor) -> float:
    """Largest per-row relative error |got_r - out_r| / max(|out_r|, 0.1 rms of the row norms) over every (b, h, s)
    row, against the model's rounded output: one wrong row or one ragged tile cannot hide in the norm of the whole
    tensor.  Where the denominator is 0 only an exact match passes."""
    err = (got.to(torch.float64) - out.to(torch.float64)).norm(dim=-1)
    rn = out.to(torch.float64).norm(dim=-1)
    den = rn.clamp_min(0.1 * float(rn.square().mean().sqrt()))
    return float(torch.where(err == 0, torch.zeros_like(err), err / den).max())


OUTPUT_METRICS = ("ulps", "mismatch", "rel", "row")


def output_errors(got: torch.Tensor, o: torch.Tensor, out: torch.Tensor, dtype: torch.dtype):
    """The OUTPUT_METRICS of an attention output against the model's (o, out): the largest error in ulps against o, the
    fraction of elements that differ from out, and the relative Frobenius and largest per-row errors against out (the
    rounded model, so that the 16-bit rounding every element carries does not hide a small error)."""
    return ulp_error(got, o, dtype), mismatch_fraction(got, out), rel_fro(got, out), row_error(got, out)


COS_FLOOR = 1e-2


def score_error(got: float, model: float, mode: str) -> float:
    """Cosine: |got - model| / max(1 - model, COS_FLOOR), the error in the quantity that moves as images grow alike
    (alpha -> 1); MSE: relative error (an exact zero must be matched exactly)."""
    e = abs(float(got) - float(model))
    if mode == "cosine":
        return e / max(1.0 - float(model), COS_FLOOR)
    return e / abs(float(model)) if model != 0 else (0.0 if e == 0 else float("inf"))
