"""`torch.ops.diffsim_b200.*` -- the C-ABI entry points as torch custom operators (CUDA dispatch key only).

north_star asks for "a thin C-ABI extension (torch custom op) in place of the hacked AttnProcessor and the metrics/
similarity reduction": the library itself knows nothing about torch (include/diffsim_b200.h: plain pointers, sizes,
strides), and this module registers its calls with the dispatcher so that reference-side code can write

    torch.ops.diffsim_b200.attn_fwd(q, k, v)                        # F.scaled_dot_product_attention(q, k, v)   hacked_attn.py:81-83
    torch.ops.diffsim_b200.aas_score(qA, kA, vA, qB, kB, vB, "cosine")   # the tail of DiffSim.diffsim           diffsim.py:177-197
    torch.ops.diffsim_b200.pair_reduce(x, y, "cosine")              # F.cosine_similarity on flattened rows       diffsim.py:187-188

There is no CPU (or any other) kernel behind these operators: called on CPU tensors the dispatcher raises
NotImplementedError -- the loud failure the path requires.  `scale = 0.0` means the default 1/sqrt(D).
attn_fwd and aas_score have autograd kernels (K5 backward); the other operators are forward-only.
"""
from __future__ import annotations

from typing import List

import torch
from torch.library import Library

from . import ops

_lib = Library("diffsim_b200", "DEF")

_lib.define("attn_fwd(Tensor q, Tensor k, Tensor v, float scale=0.0) -> Tensor")
_lib.define("aas_score(Tensor qa, Tensor ka, Tensor va, Tensor qb, Tensor kb, Tensor vb, str similarity='cosine', "
            "float scale=0.0) -> Tensor")
_lib.define("aas_pairs(Tensor q, Tensor k, Tensor v, Tensor pair_idx, str similarity='cosine', float scale=0.0) -> Tensor")
_lib.define("aas_triplets(Tensor q, Tensor k, Tensor v, Tensor trip_idx, str similarity='cosine', float scale=0.0, "
            "bool round_scores=False) -> (Tensor, Tensor, Tensor, Tensor)")
_lib.define("aas_matrix(Tensor q, Tensor k_self, Tensor v_self, Tensor k, Tensor v, str similarity='cosine', "
            "float scale=0.0) -> Tensor")
_lib.define("pair_reduce(Tensor x, Tensor y, str similarity='cosine') -> Tensor")
_lib.define("simmat(Tensor rows, Tensor? cols=None, str similarity='cosine') -> Tensor")
_lib.define("qkv_project(Tensor hidden, Tensor weight, Tensor? bias=None, int n_outputs=3) -> Tensor[]")


def _attn_fwd(q, k, v, scale=0.0):
    return ops.attn_fwd(q, k, v, scale)


def _aas_score(qa, ka, va, qb, kb, vb, similarity="cosine", scale=0.0):
    d_ab, d_ba = ops._pair_dirs(qa, ka, va, qb, kb, vb, similarity, scale)
    return (d_ab + d_ba) * 0.5


def _aas_pairs(q, k, v, pair_idx, similarity="cosine", scale=0.0):
    return ops._aas_pairs(q, k, v, pair_idx, similarity, scale)   # forward only: no autograd registered


def _aas_triplets(q, k, v, trip_idx, similarity="cosine", scale=0.0, round_scores=False):
    return ops._aas_triplets(q, k, v, trip_idx, similarity, scale, round_scores)   # forward only


def _aas_matrix(q, k_self, v_self, k, v, similarity="cosine", scale=0.0):
    return ops._aas_matrix(q, k_self, v_self, k, v, similarity, scale)   # forward only


def _pair_reduce(x, y, similarity="cosine"):
    return ops._pair_reduce(x, y, similarity)   # forward only: no autograd registered


def _simmat(rows, cols=None, similarity="cosine"):
    return ops.simmat(rows, cols, similarity)


def _qkv_project(hidden, weight, bias=None, n_outputs=3) -> List[torch.Tensor]:
    return list(ops._qkv_project(hidden, weight, bias, n_outputs))   # forward only: no autograd registered


for _name, _fn in (("attn_fwd", _attn_fwd), ("aas_score", _aas_score), ("aas_pairs", _aas_pairs),
                   ("aas_triplets", _aas_triplets), ("aas_matrix", _aas_matrix), ("pair_reduce", _pair_reduce),
                   ("simmat", _simmat), ("qkv_project", _qkv_project)):
    _lib.impl(_name, _fn, "CUDA")


# Gradients (K5): attn_fwd and aas_score are differentiable in their tensor inputs.  Only the inputs are saved; the
# backward recomputes what it needs.  The float32 gradients are cast to the input dtype by the autograd engine.
def _setup_inputs(ctx, inputs, output):
    ctx.save_for_backward(*[t for t in inputs if isinstance(t, torch.Tensor)])
    ctx.rest = [x for x in inputs if not isinstance(x, torch.Tensor)]


def _attn_fwd_bwd(ctx, dout):
    q, k, v = ctx.saved_tensors
    (scale,) = ctx.rest or [0.0]
    out = ops.attn_fwd(q, k, v, scale)
    return ops.attn_bwd(q, k, v, out, dout, scale) + (None,)


def _aas_score_bwd(ctx, grad):
    similarity, scale = (ctx.rest + ["cosine", 0.0][len(ctx.rest):])[:2]
    g = grad.reshape(1) * 0.5   # score = (dir(a->b) + dir(b->a)) / 2
    return ops.pair_dirs_bwd(*ctx.saved_tensors, g, g, similarity, scale) + (None, None)


torch.library.register_autograd("diffsim_b200::attn_fwd", _attn_fwd_bwd, setup_context=_setup_inputs, lib=_lib)
torch.library.register_autograd("diffsim_b200::aas_score", _aas_score_bwd, setup_context=_setup_inputs, lib=_lib)
DIFFERENTIABLE = ("attn_fwd", "aas_score")

OPERATORS = ("attn_fwd", "aas_score", "aas_pairs", "aas_triplets", "aas_matrix", "pair_reduce", "simmat", "qkv_project")
