"""Capture machinery at the hooked attention layer -- the replacement of diffsim/hacked_attn.py and of the
forward-pre-hooks in diffsim/diffsim.py:43-56, diffsim_xl.py:11-24, diffsim_dit.py:19-26, metrics/hooks.py.

The reference's pre-hook runs a complete hacked attention processor (projections, a full SDPA and the output
projection whose result is thrown away, diffsim/diffsim.py:48) and then lets the module's normal forward run
again; a new copy of the hook is registered on every call and never removed (diffsim/diffsim.py:144).  Here
the hook computes only the three projections, leaves `module.stores = [q, k, v]` exactly as the reference does
(same shapes, same strides: (B,H,S,D) views over (B,S,H*D) memory), can stop the trunk right after the hooked
layer (StopForward), and is removed by its context manager.
"""
from __future__ import annotations

import contextlib
from typing import Optional

import torch

from . import ops


class StopForward(Exception):
    """Raised by an early-exit hook once q, k, v of the target layer are captured: the reference lets the
    UNet run to the end for nothing (diffsim/diffsim_pipeline.py:213-221)."""


def split_heads(t: torch.Tensor, heads: int) -> torch.Tensor:
    """(B,S,H*D) -> (B,H,S,D) view, as diffsim/hacked_attn.py:74-77."""
    B, S, C = t.shape
    return t.view(B, S, heads, C // heads).transpose(1, 2)


def _stacked_qkv_weight(attn):
    """[W_q; W_k; W_v] (3C, C_in) of a diffusers-style Attention module (+ stacked bias or None), built once per module and
    rebuilt when a weight is replaced or modified in place (tensor identity and version counter)."""
    ws = (attn.to_q.weight, attn.to_k.weight, attn.to_v.weight)
    key = tuple((w.data_ptr(), w._version, w.dtype, w.device) for w in ws)
    cached = getattr(attn, "_ds_qkv_stack", None)
    if cached is None or cached[0] != key:
        weight = torch.cat([w.detach() for w in ws], dim=0).contiguous()
        bs = (attn.to_q.bias, attn.to_k.bias, attn.to_v.bias)
        bias = None
        if any(b is not None for b in bs):
            bias = torch.cat([b.detach() if b is not None else w.new_zeros(w.shape[0]) for b, w in zip(bs, ws)]).contiguous()
        cached = (key, weight, bias)
        attn._ds_qkv_stack = cached
    return cached[1], cached[2]


def _can_fuse(attn, hidden_states) -> bool:
    """The three projections run as ONE ds_qkv_project call (K4, tcgen05) when the layer is a plain self-attention
    on a CUDA device in a 16-bit dtype; otherwise the module's own nn.Linear layers are used (CPU trunks of the tests,
    fp32 trunks, LoRA-wrapped or quantised projections)."""
    lin = torch.nn.Linear
    return (hidden_states.is_cuda and hidden_states.dtype in (torch.float16, torch.bfloat16)
            and all(type(getattr(attn, n, None)) is lin for n in ("to_q", "to_k", "to_v"))
            and attn.to_q.weight.dtype == hidden_states.dtype
            and attn.to_q.in_features == attn.to_k.in_features == attn.to_v.in_features
            and attn.to_q.out_features == attn.to_k.out_features == attn.to_v.out_features
            and attn.to_q.in_features % 8 == 0 and attn.to_q.out_features % 8 == 0)


def project_qkv(attn, hidden_states: torch.Tensor, encoder_hidden_states: Optional[torch.Tensor] = None,
                already_normed: bool = False, fused_qkv: bool = True, out=None):
    """q, k, v of a diffusers-style Attention module (attributes to_q, to_k, to_v, heads; optional group_norm,
    spatial_norm, norm_cross) -- the projection part of hacked_AttnProcessor2_0.__call__
    (diffsim/hacked_attn.py:38-77), without the attention and output projection the reference discards.

    Self-attention on CUDA: one ds_qkv_project call on the stacked weight [W_q; W_k; W_v] (K4) instead of three
    nn.Linear; `out` = three pre-allocated (B,S,H*D) tensors (e.g. a slot of a QKVCache) receives the result in place.
    The fused projection is differentiable: with grad recorded, hidden_states and the to_q / to_k / to_v weights and
    biases get their gradients (ds_qkv_project_bwd).  A capture with `out` is forward-only, like the cache scorers.
    already_normed: the caller (a processor) has applied attn.spatial_norm(hidden_states, temb) itself -- a pre-hook has no
    temb and cannot."""
    if getattr(attn, "spatial_norm", None) is not None and not already_normed:
        raise NotImplementedError("spatial_norm needs temb, which a forward-pre-hook does not see: set a B200AttnProcessor "
                                  "on such layers (it applies the norm and passes already_normed=True)")
    if hidden_states.ndim == 4:
        b, c, h, w = hidden_states.shape
        hidden_states = hidden_states.view(b, c, h * w).transpose(1, 2)
    if getattr(attn, "group_norm", None) is not None:
        hidden_states = attn.group_norm(hidden_states.transpose(1, 2)).transpose(1, 2)
    if encoder_hidden_states is None and fused_qkv and _can_fuse(attn, hidden_states):
        weight, bias = _stacked_qkv_weight(attn)
        if out is None:
            # differentiable in hidden_states and in the three modules' weights and biases (not in the cached stack)
            lins = (attn.to_q, attn.to_k, attn.to_v)
            query, key, value = ops.qkv_project_stacked(hidden_states, weight, bias, 3, [m.weight for m in lins],
                                                        [m.bias for m in lins])
        else:
            query, key, value = ops.qkv_project(hidden_states, weight, bias, 3, out=out)
        return split_heads(query, attn.heads), split_heads(key, attn.heads), split_heads(value, attn.heads)
    query = attn.to_q(hidden_states)
    if encoder_hidden_states is None:
        encoder_hidden_states = hidden_states
    elif getattr(attn, "norm_cross", False):
        encoder_hidden_states = attn.norm_encoder_hidden_states(encoder_hidden_states)
    key = attn.to_k(encoder_hidden_states)
    value = attn.to_v(encoder_hidden_states)
    if out is not None:
        for o, t in zip(out, (query, key, value)):
            o.copy_(t)
        query, key, value = out
    return split_heads(query, attn.heads), split_heads(key, attn.heads), split_heads(value, attn.heads)


def make_sd_pre_hook(early_exit: bool = False, fused_qkv: bool = True, out=None):
    """forward-pre-hook with the contract of sd15_attention_forward_hooked / sdxl_attention_forward_hooked
    (diffsim/diffsim.py:43-56): `module.stores = [query, key, value]`.  fused_qkv: the projections run as one
    ds_qkv_project call (K4) where the layer allows it; out: three (B,S,H*D) tensors to capture into (a cache slot)."""

    def hook(module, input):
        q, k, v = project_qkv(module, input[0], fused_qkv=fused_qkv, out=out)
        module.stores = [q, k, v]
        if early_exit:
            raise StopForward()

    return hook


def make_dit_pre_hook(early_exit: bool = False, fused_qkv: bool = True):
    """forward-pre-hook for a timm-style Attention block (attributes qkv, num_heads, head_dim, q_norm, k_norm):
    the contract of dit_attention_forward_hook (diffsim/diffsim_dit.py:19-26).  q, k, v are views into the packed
    qkv activation (strides (N*3*H*D, D, 3*H*D, 1)); the kernels read them in place.  fused_qkv: module.qkv runs on
    ds_qkv_project (K4, bias included) when it is a plain 16-bit nn.Linear on CUDA."""

    def hook(module, input):
        x = input[0]
        B, N, C = x.shape
        lin = module.qkv
        if (fused_qkv and x.is_cuda and x.dtype in (torch.float16, torch.bfloat16) and type(lin) is torch.nn.Linear
                and lin.weight.dtype == x.dtype and C % 8 == 0 and lin.out_features % 8 == 0):
            packed = ops.qkv_project(x, lin.weight, lin.bias, 1)[0]   # differentiable in x, weight and bias
        else:
            packed = lin(x)
        qkv = packed.reshape(B, N, 3, module.num_heads, module.head_dim).permute(2, 0, 3, 1, 4)
        q, k, v = qkv.unbind(0)
        q, k = module.q_norm(q), module.k_norm(k)
        module.stores = [q, k, v]
        if early_exit:
            raise StopForward()

    return hook


@contextlib.contextmanager
def capture(module, hook):
    """Register `hook` as a forward-pre-hook on `module` for the duration of the block (and remove it: the
    reference accumulates one more hook per call, diffsim/diffsim.py:144)."""
    handle = module.register_forward_pre_hook(hook)
    try:
        yield module
    finally:
        handle.remove()


class B200AttnProcessor:
    """diffusers AttnProcessor protocol (`attn.set_processor(p)`; `p(attn, hidden_states, encoder_hidden_states,
    attention_mask, temb)`) with the hacked return contract of hacked_AttnProcessor2_0 (diffsim/hacked_attn.py:101):
    (hidden_states, query, key, value, residual).  The scaled-dot-product attention runs in the sm_100a kernel (K1, store
    mode) and, with fused_qkv (default), the three projections of a self-attention layer in ONE ds_qkv_project call (K4) on
    the stacked weight -- diffsim/hacked_attn.py:61-77 without a cuBLAS call."""

    def __init__(self, fused_qkv: bool = True):
        self.fused_qkv = fused_qkv

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, temb=None, *args, **kwargs):
        if attention_mask is not None:
            raise NotImplementedError("attention masks are not used on the DiffSim path (hacked_attn.py:81-83 passes None)")
        residual = hidden_states
        if getattr(attn, "spatial_norm", None) is not None:
            hidden_states = attn.spatial_norm(hidden_states, temb)
        input_ndim = hidden_states.ndim
        if input_ndim == 4:
            batch_size, channel, height, width = hidden_states.shape
            hidden_states = hidden_states.view(batch_size, channel, height * width).transpose(1, 2)
        batch_size = hidden_states.shape[0]
        query, key, value = project_qkv(attn, hidden_states, encoder_hidden_states, already_normed=True,
                                        fused_qkv=self.fused_qkv)
        out = ops.attn_fwd(query, key, value)                       # (B,H,S,D) view over (B,S,H*D)
        head_dim = query.shape[-1]
        hidden_states = out.transpose(1, 2).reshape(batch_size, -1, attn.heads * head_dim).to(query.dtype)
        hidden_states = attn.to_out[0](hidden_states)
        hidden_states = attn.to_out[1](hidden_states)
        if input_ndim == 4:
            hidden_states = hidden_states.transpose(-1, -2).reshape(batch_size, channel, height, width)
        if getattr(attn, "residual_connection", False):
            hidden_states = hidden_states + residual
        hidden_states = hidden_states / getattr(attn, "rescale_output_factor", 1.0)
        return hidden_states, query, key, value, residual


class B200IPAdapterAttnProcessor(torch.nn.Module):
    """hacked_IPAdapterAttnProcessor2_0 (diffsim/hacked_attn.py:104-335) with its attentions on the sm_100a kernel.

    Same constructor (`hidden_size, cross_attention_dim, dtype, num_tokens, scale`), the same `to_k_ip` / `to_v_ip`
    ModuleLists (so IP-Adapter state dicts load unchanged) and the hacked 5-tuple return
    `(hidden_states, query, ip_keys, ip_values, residual)` (:335).  `encoder_hidden_states` is the tuple
    `(text_states, [ip_states_i])` (:161-162) or, deprecated, one tensor whose last `num_tokens[0]` rows are the image
    tokens (:163-173).  The text cross-attention and one attention per adapter against its image-prompt tokens
    (kv length 4 / 16: a ragged tail for the kernel) are added with the adapter scales (:311-320).  IP-adapter masks
    (:225-280) are a generation feature the scorer never passes: NotImplementedError, not a silent skip."""

    def __init__(self, hidden_size, cross_attention_dim=None, dtype=torch.float16, num_tokens=(4,), scale=1.0):
        super().__init__()
        self.hidden_size, self.cross_attention_dim = hidden_size, cross_attention_dim
        if not isinstance(num_tokens, (tuple, list)):
            num_tokens = [num_tokens]
        self.num_tokens = num_tokens
        if not isinstance(scale, list):
            scale = [scale] * len(num_tokens)
        if len(scale) != len(num_tokens):
            raise ValueError("`scale` should be a list of integers with the same length as `num_tokens`.")
        self.scale = scale
        mk = lambda: torch.nn.ModuleList([torch.nn.Linear(cross_attention_dim, hidden_size, bias=False, dtype=dtype)  # noqa: E731
                                          for _ in range(len(num_tokens))])
        self.to_k_ip, self.to_v_ip = mk(), mk()

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, temb=None, scale=1.0,
                 ip_adapter_masks=None):
        if attention_mask is not None or ip_adapter_masks is not None:
            raise NotImplementedError("attention / ip-adapter masks are not used on the DiffSim path")
        residual = hidden_states
        ip_hidden_states = None
        if encoder_hidden_states is not None:
            if isinstance(encoder_hidden_states, tuple):
                encoder_hidden_states, ip_hidden_states = encoder_hidden_states
            else:
                end_pos = encoder_hidden_states.shape[1] - self.num_tokens[0]
                encoder_hidden_states, ip_hidden_states = (encoder_hidden_states[:, :end_pos, :],
                                                           [encoder_hidden_states[:, end_pos:, :]])
        if ip_hidden_states is None:
            raise ValueError("the IP-Adapter processor needs image-prompt states in encoder_hidden_states")
        if getattr(attn, "spatial_norm", None) is not None:
            hidden_states = attn.spatial_norm(hidden_states, temb)
        input_ndim = hidden_states.ndim
        if input_ndim == 4:
            batch_size, channel, height, width = hidden_states.shape
            hidden_states = hidden_states.view(batch_size, channel, height * width).transpose(1, 2)
        batch_size = hidden_states.shape[0]
        query, key, value = project_qkv(attn, hidden_states, encoder_hidden_states, already_normed=True)
        head_dim = query.shape[-1]
        merge = lambda o: o.transpose(1, 2).reshape(batch_size, -1, attn.heads * head_dim).to(query.dtype)  # noqa: E731
        hidden_states = merge(ops.attn_fwd(query, key, value))
        ip_keys, ip_values = [], []
        for ip_states, s, to_k_ip, to_v_ip in zip(ip_hidden_states, self.scale, self.to_k_ip, self.to_v_ip):
            if (isinstance(s, list) and all(x == 0 for x in s)) or (not isinstance(s, list) and s == 0):
                continue
            ip_key = split_heads(to_k_ip(ip_states), attn.heads)
            ip_value = split_heads(to_v_ip(ip_states), attn.heads)
            ip_keys.append(ip_key)
            ip_values.append(ip_value)
            hidden_states = hidden_states + s * merge(ops.attn_fwd(query, ip_key, ip_value))
        hidden_states = attn.to_out[0](hidden_states)
        hidden_states = attn.to_out[1](hidden_states)
        if input_ndim == 4:
            hidden_states = hidden_states.transpose(-1, -2).reshape(batch_size, channel, height, width)
        if getattr(attn, "residual_connection", False):
            hidden_states = hidden_states + residual
        hidden_states = hidden_states / getattr(attn, "rescale_output_factor", 1.0)
        return hidden_states, query, ip_keys, ip_values, residual
