import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_PATH = os.path.join(ROOT, "tests", "golden", "aas_golden.pt")
METRICS_GOLDEN_PATH = os.path.join(ROOT, "tests", "golden", "metrics_golden.pt")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200, sm_100a); run with `-m gpu`")


@pytest.fixture(scope="session")
def golden():
    import torch

    return torch.load(GOLDEN_PATH, weights_only=False)


@pytest.fixture(scope="session")
def metrics_golden():
    import torch

    return torch.load(METRICS_GOLDEN_PATH, weights_only=False)


def ip_images(seed, ip_tokens, n_adapters, alpha):
    """The inputs of an IP-Adapter golden case (same recipe as tests/golden/make_golden_metrics.py:ip_images)."""
    import torch

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
    """The inputs of the dino_cross golden case (tests/golden/make_golden_metrics.py:dino_images)."""
    import torch

    from diffsim_b200 import synth

    g = torch.Generator().manual_seed(33)
    md = synth.SynthModel(1, 6, 257, 64, seed=78)
    based = md.new_base(g)
    return md.image(based, 1.0, torch.float16, "sd", g), md.image(based, 0.6, torch.float16, "sd", g)


def clip_images():
    """The inputs of the clip_cross golden case (tests/golden/make_golden_metrics.py): (q,k,v) of two images as
    (1,12,50,64) views of (1,50,768) fp16 memory, then the fp16 out_proj weight and bias."""
    import torch

    from diffsim_b200 import synth

    g = torch.Generator().manual_seed(32)
    H, S, D = 12, 50, 64
    mc = synth.SynthModel(1, H, S, D, seed=77)
    basec = mc.new_base(g)
    a = mc.image(basec, 1.0, torch.float16, "sd", g)
    b = mc.image(basec, 0.7, torch.float16, "sd", g)
    weight = (torch.randn(H * D, H * D, generator=g) / (H * D) ** 0.5).half()
    bias = (0.1 * torch.randn(H * D, generator=g)).half()
    return a, b, weight, bias


def diffeats_features():
    """The fp16 feature maps of the diffeats_minmax_cosine golden case (tests/golden/make_golden.py)."""
    import torch

    g = torch.Generator().manual_seed(6)
    fa = torch.randn(2, 256, 320, generator=g) * 1.3 + 0.4
    fb = 0.7 * fa + 0.5 * torch.randn(2, 256, 320, generator=g)
    return fa.half(), fb.half()


def gram_features():
    """The fp16 ReLU-like feature maps of the gram golden case (tests/golden/make_golden_metrics.py)."""
    import torch

    g = torch.Generator().manual_seed(34)
    fa = torch.randn(1, 64, 16, 24, generator=g).abs().half()
    fb = (0.6 * fa.float() + 0.4 * torch.randn(1, 64, 16, 24, generator=g).abs()).half()
    return fa, fb


def regenerate_case(case):
    """Rebuild the (q,k,v) images of a golden case from its seed."""
    import torch

    from diffsim_b200 import synth

    dtype = getattr(torch, case["dtype"].split(".")[-1])
    B, H, S, D = case["shape"]
    m = synth.SynthModel(B, H, S, D, seed=2334)
    if case["alphas"] is None:
        images, pairs = synth.make_pairs(m, case["n_pairs"], dtype, seed=case["seed"], layout=case["layout"])
        assert [tuple(p) for p in pairs] == [tuple(p) for p in case["pairs"]]
        return images
    g = torch.Generator().manual_seed(case["seed"])
    base = m.new_base(g)
    images = [m.image(base, 1.0, dtype, case["layout"], g)]
    for a in case["alphas"]:
        images.append(m.image(base, a, dtype, case["layout"], g))
    return images


def checksum(t):
    import torch

    raw = t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32).to(torch.int64).reshape(-1)
    w = (torch.arange(raw.numel(), dtype=torch.int64) % 1009) + 1
    return int((raw * w).sum().item())
