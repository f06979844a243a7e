"""The reference's baseline metrics at the same boundary (tensors captured by the metric hooks in, score out).

Every function takes what the reference's hook left on `module.stores` (metrics/hooks.py:3-38) or the feature
tensors its model returned, and replaces the torch arithmetic that follows with the library's kernels:

    dino_cross_score   metrics/dino.py:120-161     AAS on DINOv2 q,k,v (6 x 64, 257 tokens)    -> fused K1
    clip_cross_score   metrics/clip_i.py:113-159   AAS on CLIP q,k,v with explicit scale and the
                                                   layer's out_proj applied before the cosine  -> K1 store + K4 + K2
    feature_score      metrics/clip_i.py:183, metrics/dino.py:183   flat cosine of two layer outputs   -> K2
    diffeats_score     metrics/diffeats.py:136-140,202-205   min-max normalise + flat cosine   -> K2 (one pass)
    embedding_score    metrics/clip_i.py:92-96, metrics/dino.py:87-91   100 * <x/|x|, y/|y|>   -> K2
    gram_matrix / gram_similarity   metrics/vgg_gram.py:57-81   F F^T, flat cosine of the Grams -> K4 + K2
    ffa_similarity     metrics/foreground_feature_averaging.py:90   cosine of two masked-mean embeddings -> K2
    all_pairs          N x N form of feature_score / diffeats_score                            -> K3

Every score but ffa_similarity (a Python float, as in the reference) and all_pairs is differentiable in its tensor
inputs: the attention (K5), projection (K4) and reduction (K2) backwards run when an input requires grad.

The backbones themselves (CLIP, DINOv2, VGG, CarveKit) are out of scope; none is installed offline.
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import torch

from . import ops

QKV = Tuple[torch.Tensor, torch.Tensor, torch.Tensor]


def _as_ref(score: torch.Tensor, like: torch.Tensor, match_reference_dtype: bool) -> torch.Tensor:
    return score.to(like.dtype) if match_reference_dtype else score


def dino_cross_score(A: QKV, B: QKV, attention_head_size: Optional[int] = None,
                     match_reference_dtype: bool = True) -> torch.Tensor:
    """metrics/dino.py:134-161 on the hooked (q,k,v) of the two images, each (bsz, heads, tokens, head_dim).
    softmax(q k^T / sqrt(attention_head_size)) v per direction, flat cosine against the self attention, mean of the
    two directions -- the AAS pair formula, so it runs on the fused attention kernel."""
    (qa, ka, va), (qb, kb, vb) = A, B
    scale = None if attention_head_size is None else float(attention_head_size) ** -0.5
    d_ab, d_ba = ops._pair_dirs(qa, ka, va, qb, kb, vb, "cosine", scale)
    if match_reference_dtype:
        return (d_ab.to(qa.dtype) + d_ba.to(qa.dtype)) / 2
    return (d_ab + d_ba) * 0.5


def attention_calc(q, k, v, scale: Optional[float], hidden_size_shape: Sequence[int], out_proj_weight: torch.Tensor,
                   out_proj_bias: Optional[torch.Tensor] = None) -> torch.Tensor:
    """metrics/clip_i.py:113-127: SDPA with an explicit scale, heads merged back to (bsz, tgt_len, embed_dim), then the
    layer's out_proj.  The attention output is written by the kernel directly in the merged (bsz, tgt_len, H*D)
    layout (the transpose + reshape of :122-123 become output strides), then one projection GEMM."""
    bsz, tgt_len, embed_dim = (int(x) for x in hidden_size_shape)
    B, H, S, D = q.shape
    if (B, S, H * D) != (bsz, tgt_len, embed_dim):
        raise RuntimeError(f"hidden_size_shape {tuple(hidden_size_shape)} does not match q {tuple(q.shape)}")
    if ops.wants_grad(q, k, v):
        # the differentiable attention allocates its (B,H,S,D) output over (B,S,H*D) memory: merging heads is a view
        merged = ops.attn_fwd(q, k, v, scale).permute(0, 2, 1, 3)
    else:
        merged = torch.empty((B, S, H, D), dtype=q.dtype, device=q.device)
        ops.attn_fwd(q, k, v, scale, out=merged.permute(0, 2, 1, 3))
    (out,) = ops.qkv_project(merged.view(B, S, H * D), out_proj_weight, out_proj_bias, n_outputs=1)
    return out


def clip_cross_score(A: QKV, B: QKV, scale: float, hidden_size_shape: Sequence[int], out_proj_weight: torch.Tensor,
                     out_proj_bias: Optional[torch.Tensor] = None, match_reference_dtype: bool = True) -> torch.Tensor:
    """metrics/clip_i.py:130-159: four attention_calc's and two flat cosines."""
    (qa, ka, va), (qb, kb, vb) = A, B
    args = (scale, hidden_size_shape, out_proj_weight, out_proj_bias)
    a_on_b = attention_calc(qa, kb, vb, *args)
    b_on_a = attention_calc(qb, ka, va, *args)
    self_a = attention_calc(qa, ka, va, *args)
    self_b = attention_calc(qb, kb, vb, *args)
    x = torch.stack([a_on_b.reshape(-1), b_on_a.reshape(-1)])
    y = torch.stack([self_a.reshape(-1), self_b.reshape(-1)])
    d = ops.pair_reduce(x, y, "cosine")
    if match_reference_dtype:
        d = d.to(qa.dtype)
        return (d[0:1] + d[1:2]) / 2
    return (d[0:1] + d[1:2]) * 0.5


def feature_score(a: torch.Tensor, b: torch.Tensor, match_reference_dtype: bool = True) -> torch.Tensor:
    """F.cosine_similarity(a.reshape(-1).unsqueeze(0), b.reshape(-1).unsqueeze(0)) -- metrics/clip_i.py:183,
    metrics/dino.py:183, metrics/vgg_gram.py:81.  Returns shape (1,)."""
    return _as_ref(ops.pair_reduce(a.reshape(1, -1), b.reshape(1, -1), "cosine"), a, match_reference_dtype)


def diffeats_score(a: torch.Tensor, b: torch.Tensor, match_reference_dtype: bool = True) -> torch.Tensor:
    """metrics/diffeats.py:136-140,202-205: (t - min) / (max - min) on each feature map, then the flat cosine; one
    pass over the data (sums, sums of squares, min and max together; the normalisation is applied algebraically)."""
    return _as_ref(ops.pair_reduce(a.reshape(1, -1), b.reshape(1, -1), "minmax_cosine"), a, match_reference_dtype)


def embedding_score(x: torch.Tensor, y: torch.Tensor) -> Tuple[torch.Tensor, int]:
    """metrics/clip_i.py:92-96 / metrics/dino.py:87-91: rows L2-normalised, 100 * row-wise dot, summed over the batch;
    returns (score.sum(0).float(), n) like the reference."""
    if x.dim() == 1:
        x, y = x[None], y[None]
    d = ops.pair_reduce(x, y, "cosine")
    return (100.0 * d).sum(0).float(), x.shape[0]


def gram_matrix(features: torch.Tensor) -> torch.Tensor:
    """metrics/vgg_gram.py:57-69: (b, d, h, w) -> view (b*d, h*w) -> F F^T, in the input dtype (fp32 accumulation,
    one rounding, like torch.mm on 16-bit inputs)."""
    b, d, h, w = features.shape
    f = features.reshape(b * d, h * w)
    if (h * w) % 8 or (b * d) % 8:
        raise RuntimeError("gram_matrix: b*d and h*w must be multiples of 8 (16-byte rows for TMA)")
    (g,) = ops.qkv_project(f, f, None, n_outputs=1)
    return g


def gram_similarity(features_a: torch.Tensor, features_b: torch.Tensor, match_reference_dtype: bool = True) -> torch.Tensor:
    """metrics/vgg_gram.py:71-81 from the VGG feature maps on: cosine of the LAST ROW of each Gram matrix (the reference
    indexes `style_grams[-1]`, i.e. one row, not the last layer -- reproduced as written)."""
    ga, gb = gram_matrix(features_a), gram_matrix(features_b)
    return feature_score(ga[-1], gb[-1], match_reference_dtype)


def ffa_embedding(grid: torch.Tensor, masks: torch.Tensor) -> torch.Tensor:
    """metrics/foreground_feature_averaging.py:110-112: foreground-masked mean of the patch-token grid.
    grid (n, 24, 24, C), masks (n, 1, 24, 24).  Tiny (n x 576 x C); left to torch."""
    return (grid * masks.permute(0, 2, 3, 1)).sum(dim=(1, 2)) / masks.sum(dim=(1, 2, 3)).unsqueeze(-1)


def ffa_similarity(emb_a: torch.Tensor, emb_b: torch.Tensor) -> float:
    """metrics/foreground_feature_averaging.py:90: torch.cosine_similarity(e_a, e_b, dim=0).cpu().item()."""
    return float(ops.pair_reduce(emb_a.reshape(1, -1), emb_b.reshape(1, -1), "cosine")[0])


def all_pairs(features: torch.Tensor, similarity: str = "cosine") -> torch.Tensor:
    """N x N matrix of feature_score / diffeats_score over a set of per-image features (N, ...): the retrieval form
    (tensor-core GEMM + fused normalisation, K3)."""
    return ops.simmat(features.reshape(features.shape[0], -1), None, similarity)
