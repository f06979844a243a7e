"""Scorers with the reference's call surface: DiffSim (SD-1.5), diffsim_xl (SDXL), diffsim_DiT (DiT-XL/2).

    DiffSim(torch_dtype, device, ip_adapter).diffsim(image_A, image_B, img_size, prompt, target_block,
        target_layer, target_step, ip_adapter=False, seed='2333', device='cuda', similarity='cosine')  -> Tensor
    DiffSim.diffsim_value(image_A, ...) -> (q, k, v)
    diffsim_xl(...).diffsim_score(image_A, image_B, img_size, prompt, target_block, target_layer, target_step,
        similarity, seed)
    diffsim_DiT(img_size, target_step, device, ckpt=None).diffsim_score(... same ...)

(reference: diffsim/diffsim.py:80-258, diffsim/diffsim_xl.py:47-155, diffsim/diffsim_dit.py:29-142).

What stays on PyTorch is the *trunk* -- VAE encode + one noised forward of the UNet / DiT up to the hooked layer.
It sits behind the small `Trunk` interface: `DiffusersTrunk` drives a real diffusers pipeline when diffusers and
weights are available (neither is, offline); `SyntheticTrunk` produces Q/K/V at the hook boundary for tests and
benchmarks.  What is replaced is everything after the hook: the four SDPA calls and the cosine / MSE reductions
(diffsim/diffsim.py:177-197) run as ONE fused sm_100a kernel per direction, reading the hook's strided q/k/v
views in place.
"""
from __future__ import annotations

import hashlib
from typing import Optional, Sequence, Tuple, Union

import torch

from . import ops

QKV = Tuple[torch.Tensor, torch.Tensor, torch.Tensor]


def get_generator(seed, device):
    """diffsim/diffsim.py:16-25 -- note the reference passes the seed through int() implicitly (default '2333')."""
    if seed is None:
        return None
    if isinstance(seed, list):
        return [torch.Generator(device).manual_seed(int(s)) for s in seed]
    return torch.Generator(device).manual_seed(int(seed))


def resolve_sd15_layer(target_layer, compat_layer_collapse: bool = True) -> int:
    """`--target_layer` arrives as a list (argprocess.py nargs='+').  The reference collapses ANY single value to
    layer 0 (diffsim/diffsim.py:99-100), so `--target_layer 5` in ipref_main.sh still scores layer 0.
    compat_layer_collapse=True reproduces that; False gives the documented meaning (the index)."""
    if isinstance(target_layer, int):
        return target_layer
    if len(target_layer) == 1:
        return 0 if compat_layer_collapse else int(target_layer[0])
    raise ValueError("the SD-1.5 scorer takes exactly one target layer")


def aas_score(A: QKV, B: QKV, similarity: str = "cosine", scale: Optional[float] = None,
              match_reference_dtype: bool = True) -> torch.Tensor:
    """The tail of DiffSim.diffsim (diffsim/diffsim.py:177-197) on captured (q,k,v) of two images.

    Two launches of the fused kernel, one per direction; each evaluates the query image's self attention and the
    cross attention against the other image's K/V and reduces them on chip.  Differentiable in all six inputs when one
    of them requires grad (K5 backward, ops.aas_dir_bwd); the score is the same either way.  The q/k/v views are passed as they
    are (unsqueeze(0) adds the image axis without copying).  With match_reference_dtype the result has the
    reference's dtype and shape: input dtype, (1,) for cosine and () for MSE."""
    (qa, ka, va), (qb, kb, vb) = A, B
    d_ab, d_ba = ops.pair_dirs(qa, ka, va, qb, kb, vb, similarity, scale)
    if not match_reference_dtype:
        return (d_ab + d_ba) * 0.5
    dt = qa.dtype
    s = (d_ab.to(dt) + d_ba.to(dt)) / 2          # the reference adds two fp16/bf16 scalars
    return s if similarity == "cosine" else s.reshape(())


def aas_score_ip_adapter(A, B, similarity: str = "cosine", scale: Optional[float] = None,
                         match_reference_dtype: bool = True) -> torch.Tensor:
    """The IP-Adapter ("DiffSim-C") tail of DiffSim.diffsim -- diffsim/diffsim.py:172-175,184-185.

    A = (query, [ip_key_i], [ip_value_i]) as hacked_IPAdapterAttnProcessor2_0 returns them (diffsim/hacked_attn.py:
    306-307,335): the queries of the image's latent tokens and, per loaded adapter, the keys / values of its image-
    prompt tokens (4 for IP-Adapter, 16 for IP-Adapter-Plus).  Per adapter i the cross attention Attn(Q_A, K_B[i],
    V_B[i]) is compared with Attn(Q_A, K_A[i], V_A[i]); the score is the mean over adapters of the flat cosines,
    averaged over the two directions.  One fused launch per (direction, adapter): kv length = #ip tokens, which the
    kernel handles as a ragged tail (zero-filled by TMA, masked to -inf in the softmax).

    The reference's MSE branch for this path cannot run (`[...].sum()` on a Python list, diffsim/diffsim.py:191-192
    raises AttributeError); the same error type is raised here rather than inventing semantics."""
    (qa, ka_l, va_l), (qb, kb_l, vb_l) = A, B
    if similarity != "cosine":
        raise AttributeError("'list' object has no attribute 'sum' (the reference's IP-Adapter MSE branch, "
                             "diffsim/diffsim.py:191-192, is not executable; only similarity='cosine' is defined)")
    if not (len(ka_l) == len(va_l) == len(kb_l) == len(vb_l)) or len(ka_l) == 0:
        raise RuntimeError("both images need the same, non-zero number of ip key/value tensors")
    dirs = [ops.pair_dirs(qa, ka, va, qb, kb, vb, "cosine", scale) for ka, va, kb, vb in zip(ka_l, va_l, kb_l, vb_l)]
    d_ab = [d[0] for d in dirs]
    d_ba = [d[1] for d in dirs]
    if match_reference_dtype:
        dt = qa.dtype   # torch.mean(torch.stack([...], dim=0)) of (1,) fp16 tensors is a 0-d fp16 tensor
        m_ab = torch.mean(torch.stack([d.to(dt) for d in d_ab], dim=0))
        m_ba = torch.mean(torch.stack([d.to(dt) for d in d_ba], dim=0))
        return (m_ab + m_ba) / 2
    return (torch.stack(d_ab).mean() + torch.stack(d_ba).mean()) * 0.5


# --------------------------------------------------------------------------------------------------------
# trunks
# --------------------------------------------------------------------------------------------------------
class Trunk:
    """Everything before the hook: image -> (q, k, v) at the target layer, in two steps that draw from ONE generator in the
    reference's order (diffsim/diffsim.py:109-113 then diffsim_pipeline.py:174-176):
        encode(image)  -> latents      draws the VAE sample
        forward(latents) -> (q, k, v)  draws the noise
    so that a scorer can call encode(A), encode(B), forward(A), forward(B) exactly as DiffSim.diffsim does, and
    extract(image) = forward(encode(image)) serves the cached / batched paths (which, like the reference's own
    diffsim_value, diffsim/diffsim.py:201-258, seed every image afresh)."""

    def encode(self, image, img_size, generator):
        raise NotImplementedError

    def forward(self, latents, prompt, target_block, target_layer, target_step, generator) -> QKV:
        raise NotImplementedError

    def extract(self, image, img_size, prompt, target_block, target_layer, target_step, generator) -> QKV:
        return self.forward(self.encode(image, img_size, generator), prompt, target_block, target_layer, target_step, generator)


class SyntheticTrunk(Trunk):
    """Q/K/V at the hook boundary from diffsim_b200.synth: `image` is any hashable id, or 'concept@alpha' to
    place images of one concept at a chosen similarity.  NOT a model: it never opens the image.  Scorers take it only when
    it is passed explicitly (tests, benchmarks, the synthetic CLI)."""

    def __init__(self, shape=(2, 8, 256, 160), dtype=torch.float16, device="cuda", layout: str = "sd", seed: int = 2334):
        from .synth import SynthModel

        self.model = SynthModel(*shape, seed=seed)
        self.dtype, self.device, self.layout = dtype, device, layout
        self._bases = {}

    def encode(self, image, img_size=512, generator=None):
        return image                                   # the "latents" of the synthetic trunk are the image id itself

    def forward(self, latents, prompt="", target_block="up_blocks", target_layer=0, target_step=0, generator=None) -> QKV:
        concept, _, alpha = str(latents).partition("@")
        alpha = float(alpha) if alpha else 1.0
        h = int(hashlib.sha1(concept.encode()).hexdigest()[:8], 16)
        if concept not in self._bases:
            self._bases[concept] = self.model.new_base(torch.Generator().manual_seed(h))
        g = torch.Generator().manual_seed((h ^ int(alpha * 1e6) ^ (int(target_step) << 8)) & 0x7FFFFFFF)
        q, k, v = self.model.image(self._bases[concept], alpha, self.dtype, self.layout, g)
        mv = lambda t: _to_device_keep_layout(t, self.device)  # noqa: E731
        return mv(q), mv(k), mv(v)

    def extract(self, image, img_size=512, prompt="", target_block="up_blocks", target_layer=0, target_step=0,
                generator=None) -> QKV:
        return self.forward(image, prompt, target_block, target_layer, target_step, generator)

    def extract_ip(self, image, img_size=512, prompt="", target_block="up_blocks", target_layer=0, target_step=0,
                   generator=None, ip_tokens: int = 16, n_adapters: int = 1):
        """(query, [ip_key], [ip_value]) as the hacked IP-Adapter processor returns them (diffsim/hacked_attn.py:
        306-307,335): latent-token queries and the keys / values of `ip_tokens` image-prompt tokens per adapter.
        The prompt tokens are the first rows of the image's own hidden state pushed through the k / v projections --
        like the real ones they are a function of the image only."""
        q, k, v = self.extract(image, img_size, prompt, target_block, target_layer, target_step, generator)
        ks = [k[:, :, i * ip_tokens:(i + 1) * ip_tokens] for i in range(n_adapters)]
        vs = [v[:, :, i * ip_tokens:(i + 1) * ip_tokens] for i in range(n_adapters)]
        return q, ks, vs


def _to_device_keep_layout(t: torch.Tensor, device) -> torch.Tensor:
    """Move a strided (B,H,S,D) view to `device` preserving its strides (the head-split view layout)."""
    out = torch.empty_strided(t.shape, t.stride(), dtype=t.dtype, device=device)
    out.copy_(t)
    return out


class DiffusersTrunk(Trunk):
    """SD-1.5 / SDXL trunk on a diffusers pipeline: VAE encode -> add noise at timesteps[target_step] -> ONE UNet
    forward that stops at the hooked attn1 (diffsim/diffsim.py:92-96,122-155; diffsim_pipeline.py:125-221; SDXL:
    diffsim/diffsim_xl.py:54-63,88-125, diffsim_xl_pipeline.py:195-323).
    Needs `diffusers` and local weights -- neither exists offline, so this class has only ever met the fake pipelines of
    tests/test_trunk_cpu.py (INTEGRATION.md says so).

    kind='sd15': prompt embeddings from pipe.encode_prompt(prompt, device, 1, True, None); VAE in the pipeline dtype.
    kind='sdxl': encode_prompt by keyword (its second positional is prompt_2); the UNet gets
        added_cond_kwargs = {text_embeds: [neg pooled; pooled], time_ids: [ids; ids]} with
        ids = pipe._get_add_time_ids((s, s), (0, 0), (s, s), ...) as diffsim_xl_pipeline.py:237-312 builds them; the VAE
        encodes in float32 and the latents are cast back to the pipeline dtype (diffsim/diffsim_xl.py:58-63)."""

    def __init__(self, pipe, device="cuda", dtype=torch.float16, guidance_scale: float = 7.5, kind: str = "sd15",
                 value_mode: bool = False, fused_qkv: bool = True):
        if kind not in ("sd15", "sdxl"):
            raise ValueError("kind must be 'sd15' or 'sdxl'")
        self.pipe, self.device, self.dtype, self.guidance_scale, self.kind = pipe, device, dtype, guidance_scale, kind
        self.value_mode = value_mode
        self.fused_qkv = fused_qkv
        self._prompt_cache = {}

    def target_module(self, target_block: str, target_layer):
        unet = self.pipe.unet
        if self.kind == "sd15":
            # diffsim() indexes down_blocks[:-1] / up_blocks[1:]; diffsim_value() has the slices swapped
            # (diffsim/diffsim.py:125-145 vs :224-244) -- value_mode reproduces the latter.
            if target_block == "down_blocks":
                blocks = unet.down_blocks[1:] if self.value_mode else unet.down_blocks[:-1]
                return blocks[target_layer].attentions[-1].transformer_blocks[-1].attn1
            if target_block == "mid_blocks":
                return unet.mid_block.attentions[-1].transformer_blocks[-1].attn1
            blocks = unet.up_blocks[:-1] if self.value_mode else unet.up_blocks[1:]
            return blocks[target_layer].attentions[-1].transformer_blocks[-1].attn1
        # SDXL: (block, attention, transformer_block) -- diffsim/diffsim_xl.py:88-107
        if target_block == "down_blocks":
            return unet.down_blocks[1:][target_layer[0]].attentions[target_layer[1]].transformer_blocks[target_layer[2]].attn1
        if target_block == "mid_blocks":
            return unet.mid_block.attentions[target_layer[0]].transformer_blocks[target_layer[1]].attn1
        return unet.up_blocks[:-1][target_layer[0]].attentions[target_layer[1]].transformer_blocks[target_layer[2]].attn1

    @torch.no_grad()
    def encode(self, image, img_size, generator):
        from .imageio import load_image, process_image

        pipe = self.pipe
        self._img_size = img_size
        x = process_image(load_image(image), img_size)
        if self.kind == "sdxl":
            pipe.vae.float()                                                        # diffsim/diffsim_xl.py:59-60
            lat = pipe.vae.encode(x.to(self.device, torch.float32)).latent_dist.sample(generator=generator)
            return (lat * pipe.vae.config.scaling_factor).to(self.dtype)
        x = x.to(self.device, self.dtype)
        return pipe.vae.encode(x).latent_dist.sample(generator=generator) * pipe.vae.config.scaling_factor

    def _conditioning(self, prompt, img_size):
        """(encoder_hidden_states, extra UNet kwargs), cached per prompt (and image size for SDXL's time ids)."""
        key = (prompt, img_size if self.kind == "sdxl" else None)
        if key in self._prompt_cache:
            return self._prompt_cache[key]
        pipe = self.pipe
        if self.kind == "sd15":
            pe, ne = pipe.encode_prompt(prompt, self.device, 1, True, None)[:2]
            cond = (torch.cat([ne, pe]), {})
        else:
            pe, ne, pooled, neg_pooled = pipe.encode_prompt(prompt=prompt, prompt_2=None, device=self.device,
                                                            num_images_per_prompt=1, do_classifier_free_guidance=True,
                                                            negative_prompt=None, negative_prompt_2=None)
            te2 = getattr(pipe, "text_encoder_2", None)
            proj_dim = int(pooled.shape[-1]) if te2 is None else te2.config.projection_dim
            size = (img_size, img_size)
            ids = pipe._get_add_time_ids(size, (0, 0), size, dtype=pe.dtype, text_encoder_projection_dim=proj_dim)
            added = {"text_embeds": torch.cat([neg_pooled, pooled], dim=0).to(self.device),
                     "time_ids": torch.cat([ids, ids], dim=0).to(self.device)}
            cond = (torch.cat([ne, pe], dim=0).to(self.device), {"added_cond_kwargs": added})
        self._prompt_cache[key] = cond
        return cond

    @torch.no_grad()
    def forward(self, latents, prompt, target_block, target_layer, target_step, generator) -> QKV:
        from . import hooks

        pipe = self.pipe
        embeds, extra = self._conditioning(prompt, getattr(self, "_img_size", None))
        pipe.scheduler.set_timesteps(1000, device=self.device)
        t = pipe.scheduler.timesteps[target_step]          # an INDEX into the 1000-step array (diffsim_pipeline.py:153-157)
        noise = torch.randn(latents.shape, generator=generator, device=latents.device, dtype=latents.dtype)
        noisy = pipe.scheduler.add_noise(latents, noise, t.reshape(1))
        module = self.target_module(target_block, target_layer)
        with hooks.capture(module, hooks.make_sd_pre_hook(early_exit=True, fused_qkv=self.fused_qkv)):
            try:
                pipe.unet(pipe.scheduler.scale_model_input(torch.cat([noisy] * 2), t), t, encoder_hidden_states=embeds, **extra)
            except hooks.StopForward:
                pass
        return tuple(module.stores)


def _require_trunk(trunk, who: str):
    if trunk is None:
        raise ValueError(
            f"{who} needs a trunk: pass trunk=DiffusersTrunk(pipe) (a diffusers pipeline with weights) -- or, for tests and "
            "benchmarks only, trunk=SyntheticTrunk(...), which produces Q/K/V from the image NAME and never reads the image. "
            "There is no default: a scorer that silently falls back to synthetic tensors returns plausible but meaningless "
            "scores.")
    return trunk


def _extract_pair(trunk, image_A, image_B, img_size, prompt, target_block, layer, target_step, generator):
    """Both images through the trunk with ONE generator consumed in the reference's order: VAE sample A, VAE sample B,
    noise A, noise B (diffsim/diffsim.py:109-113, diffsim_pipeline.py:174-176)."""
    lat_a = trunk.encode(image_A, img_size, generator)
    lat_b = trunk.encode(image_B, img_size, generator)
    A = trunk.forward(lat_a, prompt, target_block, layer, target_step, generator)
    B = trunk.forward(lat_b, prompt, target_block, layer, target_step, generator)
    return A, B


def _gen_device(trunk, device):
    return "cpu" if isinstance(trunk, SyntheticTrunk) else device


# --------------------------------------------------------------------------------------------------------
# scorers
# --------------------------------------------------------------------------------------------------------
class DiffSim:
    """SD-1.5 scorer -- diffsim/diffsim.py:80-258.  `trunk` is required (see _require_trunk)."""

    def __init__(self, torch_dtype=torch.float16, device="cuda", ip_adapter=False, trunk: Optional[Trunk] = None,
                 match_reference_dtype: bool = True, compat_layer_collapse: bool = True, compat_value_slices: bool = True):
        # ip_adapter=True: the trunk must provide extract_ip() (query + per-adapter ip keys / values).  In the reference
        # the hook that should capture them cannot fire (attn2 receives encoder_hidden_states as a keyword, SURVEY.md
        # section 5); the scoring arithmetic of diffsim/diffsim.py:172-175,184-185 is implemented regardless.
        self.device, self.ip_adapter, self.torch_dtype = device, ip_adapter, torch_dtype
        self.trunk = _require_trunk(trunk, "DiffSim")
        self.match_reference_dtype = match_reference_dtype
        self.compat_layer_collapse = compat_layer_collapse
        self.compat_value_slices = compat_value_slices

    def diffsim(self, image_A, image_B, img_size, prompt, target_block, target_layer, target_step, ip_adapter=False,
                seed="2333", device="cuda", similarity="cosine"):
        layer = resolve_sd15_layer(target_layer, self.compat_layer_collapse)
        generator = get_generator(seed, _gen_device(self.trunk, device))
        if ip_adapter:
            if not hasattr(self.trunk, "extract_ip"):
                raise NotImplementedError("this trunk does not capture IP-Adapter keys / values (extract_ip)")
            A = self.trunk.extract_ip(image_A, img_size, prompt, target_block, layer, target_step, generator)
            B = self.trunk.extract_ip(image_B, img_size, prompt, target_block, layer, target_step, generator)
            return aas_score_ip_adapter(A, B, similarity, None, self.match_reference_dtype)
        A, B = _extract_pair(self.trunk, image_A, image_B, img_size, prompt, target_block, layer, target_step, generator)
        return aas_score(A, B, similarity, None, self.match_reference_dtype)

    def extract(self, image, img_size, prompt, target_block, target_layer, target_step, seed="2333", device="cuda"):
        """(q, k, v) of ONE image at the layer diffsim() scores (same layer indexing) -- what a cache for batched scoring
        holds (drivers.build_cache).  Seeding is per image (a fresh generator: VAE sample, then noise), as in the
        reference's diffsim_value; inside diffsim(A, B) the reference draws A's and B's VAE samples before either noise, so
        image B's tensors there differ from its cached ones for the same seed (SURVEY.md section 5, RNG contract)."""
        layer = resolve_sd15_layer(target_layer, self.compat_layer_collapse)
        generator = get_generator(seed, _gen_device(self.trunk, device))
        return self.trunk.extract(image, img_size, prompt, target_block, layer, target_step, generator)

    def diffsim_value(self, image_A, img_size, prompt, target_block, target_layer, target_step, ip_adapter=False,
                      seed="2333", device="cuda", similarity="cosine"):
        """diffsim/diffsim.py:201-258.  The reference indexes the blocks differently here than in diffsim()
        (down_blocks[1:] / up_blocks[:-1] instead of down_blocks[:-1] / up_blocks[1:], :224-244 vs :125-145), so the same
        --target_layer names another layer; a trunk that knows about it (DiffusersTrunk.value_mode) reproduces that when
        compat_value_slices is set (default), else this is extract()."""
        trunk = self.trunk
        if self.compat_value_slices and getattr(trunk, "value_mode", None) is not None:
            old, trunk.value_mode = trunk.value_mode, True
            try:
                return self.extract(image_A, img_size, prompt, target_block, target_layer, target_step, seed, device)
            finally:
                trunk.value_mode = old
        return self.extract(image_A, img_size, prompt, target_block, target_layer, target_step, seed, device)


class diffsim_xl:  # noqa: N801 (the reference's name)
    """SDXL scorer -- diffsim/diffsim_xl.py:47-155.  target_layer = (block, attention, transformer_block).
    `trunk` is required: DiffusersTrunk(pipe, kind='sdxl'), or a SyntheticTrunk for tests."""

    def __init__(self, torch_dtype=torch.float16, device="cuda", ip_adapter=False, trunk: Optional[Trunk] = None,
                 match_reference_dtype: bool = True):
        if ip_adapter:
            raise NotImplementedError("the IP-Adapter path is not built")
        self.device = device
        self.trunk = _require_trunk(trunk, "diffsim_xl")
        self.match_reference_dtype = match_reference_dtype

    def diffsim_score(self, image_A, image_B, img_size, prompt, target_block, target_layer, target_step, similarity, seed):
        generator = get_generator(seed, _gen_device(self.trunk, self.device))
        A, B = _extract_pair(self.trunk, image_A, image_B, img_size, prompt, target_block, target_layer, target_step, generator)
        return aas_score(A, B, similarity, None, self.match_reference_dtype)

    def diffsim_value(self, image_A, img_size, prompt, target_block, target_layer, target_step, seed="2333", device=None):
        """Per-image (q,k,v) -- not in the reference's SDXL scorer; the batched drivers and caches need it."""
        generator = get_generator(seed, _gen_device(self.trunk, self.device))
        return self.trunk.extract(image_A, img_size, prompt, target_block, target_layer, target_step, generator)


class diffsim_DiT:  # noqa: N801
    """DiT-XL/2 scorer -- diffsim/diffsim_dit.py:29-142.  target_layer[0] = transformer block index (0..27); the hook
    hands over q, k, v as views into the packed qkv activation, which the kernels read in place.  `trunk` is required (a
    DiT trunk needs timm + the vendored DiT + a checkpoint: `ckpt` is accepted for signature compatibility and is the
    trunk's business, not this class's -- it is an error to pass one without a trunk that uses it)."""

    def __init__(self, img_size=256, target_step=0, device="cuda", ckpt=None, trunk: Optional[Trunk] = None,
                 match_reference_dtype: bool = True):
        self.device = device
        self.trunk = _require_trunk(trunk, "diffsim_DiT")
        if ckpt is not None and not hasattr(self.trunk, "load_checkpoint"):
            raise ValueError("ckpt was given but the trunk has no load_checkpoint(): it would be silently ignored")
        if ckpt is not None:
            self.trunk.load_checkpoint(ckpt)
        self.match_reference_dtype = match_reference_dtype

    def diffsim_score(self, image_A, image_B, img_size, prompt, target_block, target_layer, target_step, similarity, seed):
        layer = target_layer[0] if not isinstance(target_layer, int) else target_layer
        generator = get_generator(seed, _gen_device(self.trunk, self.device))
        A, B = _extract_pair(self.trunk, image_A, image_B, img_size, prompt, target_block, layer, target_step, generator)
        return aas_score(A, B, similarity, None, self.match_reference_dtype)

    def diffsim_value(self, image_A, img_size, prompt, target_block, target_layer, target_step, seed="2333", device=None):
        """Per-image (q,k,v) -- not in the reference's DiT scorer; the batched drivers and caches need it."""
        layer = target_layer[0] if not isinstance(target_layer, int) else target_layer
        generator = get_generator(seed, _gen_device(self.trunk, self.device))
        return self.trunk.extract(image_A, img_size, prompt, target_block, layer, target_step, generator)
