#!/usr/bin/env python
"""Generate tests/golden/metrics_golden.pt by RUNNING THE REFERENCE'S OWN CODE for the widened rows of the hot path
(SURVEY.md section 8 a2, a6, f3):

    python tests/golden/make_golden_metrics.py     (needs /root/reference; not needed at test time)

  * IP-Adapter AAS: DiffSim.diffsim(..., ip_adapter=True), diffsim/diffsim.py:98-197 -- the list form of lines
    172-175 and 184-185 -- with a fake pipeline that leaves (query, [ip_key], [ip_value]) in `module.stores`;
  * CLIP AAS:  ClipScore-class `clip_cross_score` (metrics/clip_i.py:130-159, calls attention_calc :113-127) executed
    unmodified on a fake `self` whose encoder layer holds the synthetic q,k,v and a real nn.Linear out_proj;
  * DINO AAS:  `dino_cross_score` (metrics/dino.py:134-161, attention_calc :120-131) likewise;
  * Gram:      vgg_gram.gram_matrix (metrics/vgg_gram.py:57-69) and the last-row cosine of :81.
Scores are recorded for fp32 inputs (and fp16 where torch's CPU kernels allow).  Seeded inputs are stored as checksums
(tests/conftest.py regenerates them) so that the GPU tests can verify they feed the kernels the very same inputs.
"""
import importlib
import os
import sys
import types

import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden as MG  # noqa: E402  (stub import hook, FakePipe, checksum)


def _find_class_with(mod, method):
    for name in dir(mod):
        cls = getattr(mod, name)
        if isinstance(cls, type) and hasattr(cls, method):
            return cls
    raise RuntimeError(f"no class with {method} in {mod.__name__}")


class _Layer:
    """An encoder layer as the metric code sees it: hook registration is a no-op, `.stores` is refilled per image."""

    def __init__(self):
        self.stores = None

    def register_forward_hook(self, fn):
        return None


def run_ip_adapter(ref_mod, A, B, similarity="cosine"):
    ds = ref_mod.DiffSim.__new__(ref_mod.DiffSim)
    ds.pipe = MG.FakePipe()
    ds.device = "cpu"
    ds.ip_adapter = True
    ds.pipe.queue = [A, B]
    ref_mod.load_image = lambda path: path
    ref_mod.process_image = lambda img, size=512: torch.zeros(1, 3, 8, 8)
    return ds.diffsim(image_A="A", image_B="B", img_size=512, prompt="p", target_block="up_blocks", target_layer=[0],
                      target_step=600, ip_adapter=True, seed=2334, device="cpu", similarity=similarity)


def ip_images(seed, ip_tokens, n_adapters, alpha):
    """Two images of one concept (alpha 1 and `alpha`) as (query, [ip_key], [ip_value]); SD-1.5 up_blocks shape, fp16."""
    from diffsim_b200 import synth

    m = synth.SynthModel(2, 8, 256, 160, seed=2334)
    g = torch.Generator().manual_seed(seed)
    base = m.new_base(g)
    imgs = []
    for a in (1.0, alpha):
        q, k, v = m.image(base, a, torch.float16, "sd", g)
        ks = [k[:, :, i * ip_tokens:(i + 1) * ip_tokens] for i in range(n_adapters)]
        vs = [v[:, :, i * ip_tokens:(i + 1) * ip_tokens] for i in range(n_adapters)]
        imgs.append((q, ks, vs))
    return imgs


def dino_images():
    """DINOv2-s shaped q,k,v (1, 6, 257, 64) of two images of one concept, fp16; regenerated from the seed by the tests."""
    from diffsim_b200 import synth

    g = torch.Generator().manual_seed(33)
    md = synth.SynthModel(1, 6, 257, 64, seed=78)
    based = md.new_base(g)
    return md.image(based, 1.0, torch.float16, "sd", g), md.image(based, 0.6, torch.float16, "sd", g)


def main():
    from diffsim_b200 import synth

    ref_mod = MG.import_reference()
    out = {"torch_version": torch.__version__}
    torch.set_num_threads(8)

    # ---------------------------------------------------------------- IP-Adapter list form
    ip = {"cases": []}
    for seed, (T_ip, n_ad, alpha) in enumerate(((16, 1, 0.8), (4, 1, 0.5), (16, 2, 0.9)), start=31):
        imgs = ip_images(seed, T_ip, n_ad, alpha)
        f32 = lambda im: (im[0].float(), [t.float() for t in im[1]], [t.float() for t in im[2]])  # noqa: E731
        score32 = float(run_ip_adapter(ref_mod, f32(imgs[0]), f32(imgs[1])))
        try:
            score16 = float(run_ip_adapter(ref_mod, imgs[0], imgs[1]))
        except Exception as e:  # pragma: no cover
            score16 = None
            print("fp16 ip run failed:", repr(e))
        mse_error = None
        try:
            run_ip_adapter(ref_mod, f32(imgs[0]), f32(imgs[1]), "mse")
        except Exception as e:
            mse_error = type(e).__name__
        # inputs are regenerated from the seed at test time (ip_images below); the checksums prove they are identical
        ip["cases"].append({"seed": seed, "ip_tokens": T_ip, "n_adapters": n_ad, "alpha": alpha, "score_fp32_math": score32,
                            "score_native_f16": score16, "mse_error": mse_error,
                            "checksums": [[MG.checksum(im[0])] + [MG.checksum(t) for t in im[1] + im[2]] for im in imgs]})
        print("ip_adapter", T_ip, n_ad, score32, score16, mse_error)
    out["ip_adapter"] = ip

    # ---------------------------------------------------------------- CLIP AAS (ViT-B/32: 12 x 64, 50 tokens)
    clip = importlib.import_module("metrics.clip_i")
    ClipCls = _find_class_with(clip, "clip_cross_score")
    g = torch.Generator().manual_seed(32)
    H, S, D = 12, 50, 64
    mc = synth.SynthModel(1, H, S, D, seed=77)
    basec = mc.new_base(g)
    qa, ka, va = mc.image(basec, 1.0, torch.float16, "sd", g)
    qb, kb, vb = mc.image(basec, 0.7, torch.float16, "sd", g)
    out_proj = torch.nn.Linear(H * D, H * D)
    with torch.no_grad():
        out_proj.weight.copy_((torch.randn(H * D, H * D, generator=g) / (H * D) ** 0.5).half().float())
        out_proj.bias.copy_((0.1 * torch.randn(H * D, generator=g)).half().float())
    scale = D ** -0.5
    layer = _Layer()
    layer.self_attn = types.SimpleNamespace(dropout=0.0, training=False, scale=scale, out_proj=out_proj)
    fake = types.SimpleNamespace()
    fake.model = types.SimpleNamespace(vision_model=types.SimpleNamespace(encoder=types.SimpleNamespace(layers=[layer])))
    fake.attention_calc = types.MethodType(ClipCls.attention_calc, fake)
    feed = [(qa.float(), ka.float(), va.float(), (1, S, H * D)), (qb.float(), kb.float(), vb.float(), (1, S, H * D))]

    def get_image_features(images, norm=True):
        layer.stores = feed[0] if images == ["A"] else feed[1]
        return None

    fake.get_image_features = get_image_features
    score = ClipCls.clip_cross_score(fake, "A", "B", [0])
    a_on_b = ClipCls.attention_calc(fake, feed[0][0], feed[1][1], feed[1][2], 0.0, False, scale, (1, S, H * D), out_proj)
    # inputs are regenerated from the seed at test time (conftest.clip_images); the checksums prove they are identical
    out["clip_cross"] = {"checksums": [[MG.checksum(t) for t in im] for im in
                                       ((qa, ka, va), (qb, kb, vb), (out_proj.weight.detach().half(), out_proj.bias.detach().half()))],
                         "scale": scale, "score_fp32_math": float(score), "attention_calc_a_on_b_fp32": a_on_b.detach()}
    print("clip_cross", float(score))

    # ---------------------------------------------------------------- DINO AAS (DINOv2-s: 6 x 64, 257 tokens)
    dino = importlib.import_module("metrics.dino")
    DinoCls = _find_class_with(dino, "dino_cross_score")
    H, S, D = 6, 257, 64
    (qa, ka, va), (qb, kb, vb) = dino_images()
    att = _Layer()
    att.attention_head_size = D
    att.dropout = torch.nn.Identity()
    fake = types.SimpleNamespace()
    fake.model = types.SimpleNamespace(encoder=types.SimpleNamespace(
        layer=[types.SimpleNamespace(attention=types.SimpleNamespace(attention=att))]))
    fake.attention_calc = types.MethodType(DinoCls.attention_calc, fake)
    feedd = [(qa.float(), ka.float(), va.float()), (qb.float(), kb.float(), vb.float())]

    def get_image_features_d(images, norm=True):
        att.stores = feedd[0] if images == ["A"] else feedd[1]
        return None

    fake.get_image_features = get_image_features_d
    score = DinoCls.dino_cross_score(fake, "A", "B", [0])
    out["dino_cross"] = {"checksums": [[MG.checksum(t) for t in im] for im in ((qa, ka, va), (qb, kb, vb))],
                         "attention_head_size": D, "score_fp32_math": float(score)}
    print("dino_cross", float(score))

    # ---------------------------------------------------------------- Gram matrix + last-row cosine
    vg = importlib.import_module("metrics.vgg_gram")
    g = torch.Generator().manual_seed(34)
    fa = torch.randn(1, 64, 16, 24, generator=g).abs().half()      # ReLU-like features
    fb = (0.6 * fa.float() + 0.4 * torch.randn(1, 64, 16, 24, generator=g).abs()).half()
    fake = types.SimpleNamespace()
    ga = vg.vgg_gram.gram_matrix(fake, fa.float())
    gb = vg.vgg_gram.gram_matrix(fake, fb.float())
    cos = F.cosine_similarity(ga[-1].reshape(-1).unsqueeze(0), gb[-1].reshape(-1).unsqueeze(0))
    # the features are regenerated from the seed at test time (conftest.gram_features)
    out["gram"] = {"checksums": [MG.checksum(fa), MG.checksum(fb)], "gram_a_fp32": ga, "score_fp32_math": float(cos)}
    print("gram", float(cos))

    path = os.path.join(HERE, "metrics_golden.pt")
    torch.save(out, path)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
