"""GPU parity of the widened rows: IP-Adapter AAS (a2), CLIP / DINO AAS and the baseline-metric reductions (a6, f3),
the batched drivers (f4) and the retrieval path (f1) -- all through the C ABI, against the reference-generated vectors
of tests/golden/metrics_golden.pt and the CPU oracle."""
import pytest
import torch

from conftest import checksum, clip_images, dino_images, gram_features, ip_images
from oracle import aas_oracle as O

pytestmark = pytest.mark.gpu

REL_16BIT = 1e-3   # north_star: scores within 1e-3 relative on 16-bit inputs


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _keep(t, dev):
    out = torch.empty_strided(t.shape, t.stride(), dtype=t.dtype, device=dev)
    out.copy_(t)
    return out


def test_ip_adapter_score_matches_the_reference_run(metrics_golden):
    dev = _cuda()
    from diffsim_b200.diffsim import aas_score_ip_adapter

    for case in metrics_golden["ip_adapter"]["cases"]:
        imgs = ip_images(case["seed"], case["ip_tokens"], case["n_adapters"], case["alpha"])
        A, B = [(_keep(q, dev), [t.to(dev) for t in ks], [t.to(dev) for t in vs]) for q, ks, vs in imgs]
        got = aas_score_ip_adapter(A, B, "cosine", match_reference_dtype=False)
        assert float(got) == pytest.approx(case["score_fp32_math"], rel=REL_16BIT)
        t1 = O.aas_ip_adapter_score(*imgs[0], *imgs[1], tier="T1")
        assert float(got) == pytest.approx(t1, rel=2e-4)
        # reference dtype / shape: torch.mean(torch.stack([...])) of fp16 (1,) tensors -> 0-d fp16
        ref_like = aas_score_ip_adapter(A, B, "cosine")
        assert ref_like.dtype == torch.float16 and ref_like.shape == ()
        assert float(ref_like) == pytest.approx(case["score_native_f16"], abs=2e-3)
        with pytest.raises(AttributeError):     # diffsim/diffsim.py:191-192 is not executable in the reference either
            aas_score_ip_adapter(A, B, "mse")


def test_diffsim_class_ip_adapter_path():
    dev = _cuda()
    from diffsim_b200.diffsim import DiffSim, SyntheticTrunk

    ds = DiffSim(torch.float16, dev, ip_adapter=True, trunk=SyntheticTrunk((2, 8, 256, 160), torch.float16, dev))
    same = ds.diffsim("cat@1.0", "cat@1.0", 512, "p", "up_blocks", [0], 600, ip_adapter=True)
    near = ds.diffsim("cat@1.0", "cat@0.9", 512, "p", "up_blocks", [0], 600, ip_adapter=True)
    far = ds.diffsim("cat@1.0", "dog@1.0", 512, "p", "up_blocks", [0], 600, ip_adapter=True)
    assert float(same) == pytest.approx(1.0, abs=1e-3) and float(same) > float(near) > float(far)


def test_dino_cross_score_matches_the_reference_run(metrics_golden):
    dev = _cuda()
    from diffsim_b200 import metrics

    c = metrics_golden["dino_cross"]
    A, B = dino_images()
    Ad, Bd = tuple(_keep(t, dev) for t in A), tuple(_keep(t, dev) for t in B)
    got = metrics.dino_cross_score(Ad, Bd, c["attention_head_size"], match_reference_dtype=False)
    assert float(got) == pytest.approx(c["score_fp32_math"], rel=REL_16BIT)
    assert metrics.dino_cross_score(Ad, Bd, c["attention_head_size"]).dtype == torch.float16


def test_clip_cross_score_matches_the_reference_run(metrics_golden):
    dev = _cuda()
    from diffsim_b200 import metrics

    c = metrics_golden["clip_cross"]
    img_a, img_b, w_host, bias_host = clip_images()
    assert [[checksum(t) for t in im] for im in (img_a, img_b, (w_host, bias_host))] == c["checksums"]
    (qa, ka, va), (qb, kb, vb) = (tuple(_keep(t, dev) for t in im) for im in (img_a, img_b))
    shape = (1, qa.shape[2], qa.shape[1] * qa.shape[3])
    w, b = w_host.to(dev), bias_host.to(dev)
    a_on_b = metrics.attention_calc(qa, kb, vb, c["scale"], shape, w, b)
    assert a_on_b.shape == shape and a_on_b.dtype == torch.float16
    ref = c["attention_calc_a_on_b_fp32"].double()
    assert (a_on_b.double().cpu() - ref).abs().max().item() < 4e-3 * max(1.0, ref.abs().max().item())
    got = metrics.clip_cross_score((qa, ka, va), (qb, kb, vb), c["scale"], shape, w, b, match_reference_dtype=False)
    assert got.shape == (1,)
    # two 16-bit roundings (attention output, projection output) sit between the kernel path and the fp32 reference
    assert float(got) == pytest.approx(c["score_fp32_math"], rel=REL_16BIT)
    t1 = O.clip_cross_score(*img_a, *img_b, c["scale"], shape, w_host, bias_host, round_to=torch.float16)
    assert float(got) == pytest.approx(t1, rel=2e-4)


def test_gram_and_flat_feature_scores(metrics_golden):
    dev = _cuda()
    from diffsim_b200 import metrics

    c = metrics_golden["gram"]
    fa_host, fb_host = gram_features()
    assert [checksum(fa_host), checksum(fb_host)] == c["checksums"]
    fa, fb = fa_host.to(dev), fb_host.to(dev)
    g = metrics.gram_matrix(fa)
    ref = c["gram_a_fp32"].double()
    assert g.shape == (64, 64) and (g.double().cpu() - ref).abs().max().item() <= 1e-3 * ref.abs().max().item()  # fp16 ulp
    got = metrics.gram_similarity(fa, fb, match_reference_dtype=False)
    assert float(got) == pytest.approx(c["score_fp32_math"], rel=REL_16BIT)
    assert float(got) == pytest.approx(O.gram_similarity(fa_host, fb_host, round_to=torch.float16), rel=1e-5)
    # flat cosine / embedding score / masked mean
    x, y = fa.reshape(1, -1), fb.reshape(1, -1)
    assert float(metrics.feature_score(x, y, False)) == pytest.approx(O.flat_cosine(x.cpu(), y.cpu()), rel=2e-5)
    s, n = metrics.embedding_score(fa.reshape(64, -1), fb.reshape(64, -1))
    want = sum(100.0 * O.flat_cosine(fa_host.reshape(64, -1)[i], fb_host.reshape(64, -1)[i]) for i in range(64))
    assert n == 64 and float(s) == pytest.approx(want, rel=2e-5)
    grid = torch.randn(2, 24, 24, 32, device=dev)
    masks = (torch.rand(2, 1, 24, 24, device=dev) > 0.5).float()
    e = metrics.ffa_embedding(grid, masks)
    assert metrics.ffa_similarity(e[0], e[1]) == pytest.approx(O.flat_cosine(e[0].cpu(), e[1].cpu()), abs=2e-5)
    # all-pairs form == pairwise form
    feats = torch.randn(12, 4, 40, device=dev).half()
    m = metrics.all_pairs(feats)
    assert float(m[3, 7]) == pytest.approx(float(metrics.feature_score(feats[3], feats[7], False)), abs=2e-5)


def test_batched_driver_equals_per_pair_reference_loop():
    """drivers.run_2afc (every image extracted once, one fused call) against the reference's loop: DiffSim.diffsim twice
    per triplet and a host-side comparison per triplet (cute_main.py:111-132,196-205)."""
    dev = _cuda()
    from diffsim_b200 import drivers
    from diffsim_b200.diffsim import DiffSim, SyntheticTrunk

    ds = DiffSim(torch.float16, dev, trunk=SyntheticTrunk((2, 8, 256, 160), torch.float16, dev))
    trips = [(f"c{i}@1.0", f"c{i}@{0.55 + 0.05 * (i % 5):.2f}", f"c{i}@{0.35 + 0.07 * (i % 7):.2f}") for i in range(12)]
    trips.append(("c0@1.0", "c1@1.0", "c0@0.9"))    # shares images with earlier triplets
    args = (512, "p", "up_blocks", [0], 600)
    for sim in ("cosine", "mse"):
        r = drivers.run_2afc(ds, trips, *args, similarity=sim, device=dev)
        correct = correct2 = 0
        for t, (a, b, c) in enumerate(trips):
            ab = ds.diffsim(a, b, *args, similarity=sim)
            ac = ds.diffsim(a, c, *args, similarity=sim)
            assert float(r.diff_ab[t]) == pytest.approx(float(ab), rel=2e-3, abs=1e-4)   # fp16 score tensors
            ok = bool(ab < ac) if sim == "mse" else bool(ab > ac)
            ok2 = bool(ab * 2 < ac) if sim == "mse" else bool(ab > 2 * ac)
            assert bool(r.flags[t]) == ok
            correct += ok
            correct2 += ok2
        assert (r.total, r.correct, r.correct_2x) == (len(trips), correct, correct2)


def test_retrieval_from_a_stored_cache(tmp_path):
    dev = _cuda()
    from diffsim_b200 import retrieval as R, scoring, synth

    m = synth.SynthModel(2, 4, 128, 64, seed=2334)
    images, labels = synth.make_styles(m, 5, 4, torch.float16, seed=3)
    names = [f"{labels[i]:03d}_{i % 4 + 1}" for i in range(len(images))]
    path = str(tmp_path / "sref.safetensors")
    R.save_qkv(path, scoring.QKVCache.from_images(images), names, "k")
    cache, names2 = R.load_qkv(path, dev, expect_key="k")
    dm = scoring.aas_matrix_local(cache, cache)
    s = scoring.symmetrize(dm)
    acc = R.retrieval_accuracy(s, labels, topk=3)
    assert acc["precision@k"] == 1.0                      # 3 other images of the same style come first
    ref = O.symmetrize(O.aas_matrix([im[0] for im in images], [im[1] for im in images], [im[2] for im in images]))
    assert ((s.double().cpu() - ref).abs() / ref.abs().clamp_min(1e-9)).max().item() < REL_16BIT
    paths = R.write_retrieval_results(s, names2, str(tmp_path / "out"), topk=4)
    first = R.read_retrieval_result(paths[0], limit=3)
    assert all(p.startswith(names[0].split("_")[0]) for p in first)
