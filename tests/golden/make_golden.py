#!/usr/bin/env python
"""Generate tests/golden/aas_golden.pt by RUNNING THE REFERENCE'S OWN CODE in the build container.

    python tests/golden/make_golden.py            (needs /root/reference; not needed at test time)

The reference cannot be imported as shipped: diffusers, timm, seaborn, matplotlib are not installed, there are
no weights and no network.  Everything *around* the hot path is therefore replaced:
  - absent third-party modules are stubbed by an import hook (they are only touched at import time);
  - the pipeline (VAE + UNet trunk) is a fake whose .step() deposits synthetic Q/K/V in `module.stores`,
    exactly where the reference's forward-pre-hook would leave them (diffsim/diffsim.py:43-56,157,169).
The hot path itself is NOT replaced: DiffSim.diffsim (diffsim/diffsim.py:98-197) is executed as is, so the
recorded scores are produced by the reference's lines 177-197 with torch's own SDPA / cosine_similarity /
mse_loss.  Likewise metrics/dino.py:attention_calc and metrics/diffeats.py:min_max_normalize are called from
the imported reference modules.

Inputs come from seeded generators (diffsim_b200.synth, torch.Generator); the file stores their checksums, not the
tensors, so that it stays small and tests can verify they regenerated identical inputs.
"""
import importlib
import importlib.abc
import importlib.machinery
import os
import sys
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("DIFFSIM_REFERENCE", "/root/reference")
sys.path.insert(0, ROOT)

STUB_ROOTS = ("diffusers", "seaborn", "matplotlib", "timm", "lpips", "carvekit", "segment_anything", "megfile",
              "fire")


class _StubMeta(type):
    def __getattr__(cls, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Stub

    def __call__(cls, *a, **k):
        if cls is _Stub:
            return type.__call__(cls)
        return type.__call__(cls, *a, **k)


class _Stub(metaclass=_StubMeta):
    """Universal placeholder: any attribute is a stub, calling it returns a stub; usable as a base class."""

    def __init__(self, *a, **k):
        pass

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Stub

    def __call__(self, *a, **k):
        if len(a) == 1 and callable(a[0]) and not k:
            return a[0]  # behaves as a transparent decorator
        return _Stub()


class _StubModule(types.ModuleType):
    __path__ = []

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Stub


class _StubFinder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    def find_spec(self, fullname, path, target=None):
        if fullname.split(".")[0] in STUB_ROOTS:
            return importlib.machinery.ModuleSpec(fullname, self, is_package=True)
        return None

    def create_module(self, spec):
        return _StubModule(spec.name)

    def exec_module(self, module):
        pass


def import_reference():
    sys.meta_path.insert(0, _StubFinder())
    sys.path.insert(0, REF)
    ref_diffsim = importlib.import_module("diffsim.diffsim")
    return ref_diffsim


# ------------------------------------------------------------------------------------------------
# fake trunk: everything the reference touches before line 172
# ------------------------------------------------------------------------------------------------
class FakeAttn:
    def __init__(self):
        self.stores = None
        self.hooks = []

    def register_forward_pre_hook(self, fn):
        self.hooks.append(fn)


def _block():
    tb = types.SimpleNamespace(attn1=FakeAttn(), attn2=FakeAttn())
    att = types.SimpleNamespace(transformer_blocks=[tb])
    return types.SimpleNamespace(attentions=[att])


class FakePipe:
    """pipe.step() hands out the queued (q,k,v) triples in order: first call = image A, second = image B."""

    def __init__(self):
        self.queue = []
        blocks = [_block() for _ in range(4)]
        self.unet = types.SimpleNamespace(down_blocks=[_block() for _ in range(4)], mid_block=_block(),
                                          up_blocks=blocks)
        lat = types.SimpleNamespace(sample=lambda generator=None: torch.zeros(1, 4, 8, 8))
        self.vae = types.SimpleNamespace(encode=lambda image: types.SimpleNamespace(latent_dist=lat),
                                         config=types.SimpleNamespace(scaling_factor=0.18215))

    def _all_attn(self):
        for blk in list(self.unet.down_blocks) + [self.unet.mid_block] + list(self.unet.up_blocks):
            for a in blk.attentions:
                for tb in a.transformer_blocks:
                    yield tb.attn1
                    yield tb.attn2

    def step(self, **kwargs):
        q, k, v = self.queue.pop(0)
        for m in self._all_attn():
            m.stores = [q, k, v]
        return 0


class _HalfSafe:
    """image.to(device=..., dtype=torch.float16) in prepare_image_latents: keep it a no-op tensor."""


def run_reference_pair(ref_mod, A, B, similarity, target_block="up_blocks"):
    ds = ref_mod.DiffSim.__new__(ref_mod.DiffSim)  # skip __init__ (it loads weights from a NAS path)
    ds.pipe = FakePipe()
    ds.device = "cpu"
    ds.ip_adapter = False
    ds.pipe.queue = [A, B]
    ref_mod.load_image = lambda path: path
    ref_mod.process_image = lambda img, size=512: torch.zeros(1, 3, 8, 8)
    out = ds.diffsim(image_A="A", image_B="B", img_size=512, prompt="p", target_block=target_block, target_layer=[0],
                     target_step=600, ip_adapter=False, seed=2334, device="cpu", similarity=similarity)
    return out


def checksum(t: torch.Tensor) -> int:
    """Order-sensitive integer checksum of the raw 16/32-bit patterns."""
    raw = t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32).to(torch.int64).reshape(-1)
    w = (torch.arange(raw.numel(), dtype=torch.int64) % 1009) + 1
    return int((raw * w).sum().item())


def main():
    from diffsim_b200 import synth

    ref_mod = import_reference()
    golden = {"torch_version": torch.__version__, "cases": []}
    torch.set_num_threads(8)

    def add_case(name, shape, dtype, layout, n_pairs, seed, alphas=None):
        B, H, S, D = shape
        m = synth.SynthModel(B, H, S, D, seed=2334)
        if alphas is None:
            images, pairs = synth.make_pairs(m, n_pairs, dtype, seed=seed, layout=layout)
        else:
            g = torch.Generator().manual_seed(seed)
            base = m.new_base(g)
            images, pairs = [m.image(base, 1.0, dtype, layout, g)], []
            for a in alphas:
                images.append(m.image(base, a, dtype, layout, g))
                pairs.append((0, len(images) - 1))
        case = {"name": name, "shape": shape, "dtype": str(dtype), "layout": layout, "n_pairs": len(pairs), "seed": seed,
                "alphas": alphas, "pairs": pairs, "scores": {}, "checksums": [[checksum(t) for t in im] for im in images]}
        for sim in ("cosine", "mse"):
            native, f32 = [], []
            for a, b in pairs:
                A, Bm = images[a], images[b]
                native.append(float(run_reference_pair(ref_mod, A, Bm, sim)))
                f32.append(float(run_reference_pair(ref_mod, tuple(t.float() for t in A), tuple(t.float() for t in Bm), sim)))
            case["scores"][sim] = {"reference_native_dtype": native, "reference_fp32_math": f32}
        golden["cases"].append(case)
        print(name, {k: [round(x, 5) for x in v["reference_fp32_math"][:4]] for k, v in case["scores"].items()})

    # small
    add_case("small_f32", (2, 2, 64, 40), torch.float32, "sd", 3, 11)
    add_case("small_f16", (2, 2, 64, 40), torch.float16, "sd", 3, 12)
    add_case("small_bf16", (2, 2, 64, 40), torch.bfloat16, "sd", 3, 13)
    add_case("ragged_f16", (1, 3, 50, 64), torch.float16, "sd", 2, 14)           # CLIP-like 50 tokens
    # the benchmark shapes
    add_case("sd15_up0_f16_cute16", (2, 8, 256, 160), torch.float16, "sd", 16, 2334)  # config 1
    add_case("sd15_up0_bf16", (2, 8, 256, 160), torch.bfloat16, "sd", 4, 21)
    add_case("sd15_up0_alpha_sweep", (2, 8, 256, 160), torch.float16, "sd", 0, 22,
             alphas=[1.0, 0.95, 0.8, 0.5, 0.2, 0.0])
    add_case("dit_xl2_f16_packed", (2, 16, 256, 72), torch.float16, "dit", 4, 23)  # config 5
    add_case("sd15_mid_f16", (2, 8, 64, 160), torch.float16, "sd", 3, 24)
    add_case("sdxl_like_f16", (2, 4, 320, 64), torch.float16, "sd", 2, 25)

    # metrics helpers from the reference modules
    extra = {}
    try:
        dino = importlib.import_module("metrics.dino")
        g = torch.Generator().manual_seed(5)
        q, k, v = (torch.randn(1, 6, 257, 64, generator=g) for _ in range(3))
        self_obj = types.SimpleNamespace()
        out = dino.DinoScore.attention_calc(self_obj, q, k, v, 64, torch.nn.Identity()) if hasattr(dino, "DinoScore") else None
        if out is None:
            for name in dir(dino):
                cls = getattr(dino, name)
                if isinstance(cls, type) and hasattr(cls, "attention_calc"):
                    out = cls.attention_calc(self_obj, q, k, v, 64, torch.nn.Identity())
                    break
        extra["dino_attention_calc"] = {"q": q, "k": k, "v": v, "out": out}
        print("dino attention_calc captured", tuple(out.shape))
    except Exception as e:  # pragma: no cover
        print("dino import failed:", repr(e))
    try:
        diffeats = importlib.import_module("metrics.diffeats")
        g = torch.Generator().manual_seed(6)
        fa = torch.randn(2, 256, 320, generator=g) * 1.3 + 0.4
        fb = 0.7 * fa + 0.5 * torch.randn(2, 256, 320, generator=g)
        import torch.nn.functional as F

        na, nb = diffeats.min_max_normalize(fa), diffeats.min_max_normalize(fb)
        cos = F.cosine_similarity(na.reshape(-1).unsqueeze(0), nb.reshape(-1).unsqueeze(0))
        # the features are regenerated from the seed at test time (conftest.diffeats_features)
        extra["diffeats_minmax_cosine"] = {"checksums": [checksum(fa.half()), checksum(fb.half())], "score_fp32_inputs": float(cos),
                                           "score_f16_inputs": float(F.cosine_similarity(
                                               diffeats.min_max_normalize(fa.half().float()).reshape(1, -1),
                                               diffeats.min_max_normalize(fb.half().float()).reshape(1, -1)))}
        print("diffeats min-max cosine", extra["diffeats_minmax_cosine"]["score_f16_inputs"])
    except Exception as e:  # pragma: no cover
        print("diffeats import failed:", repr(e))
    golden["extra"] = extra
    out_path = os.path.join(HERE, "aas_golden.pt")
    torch.save(golden, out_path)
    print("wrote", out_path, os.path.getsize(out_path), "bytes")


if __name__ == "__main__":
    main()
