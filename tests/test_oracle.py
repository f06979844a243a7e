"""The CPU oracle against the vectors produced by the reference's own code (tests/golden/make_golden.py),
plus the known-answer identities of the AAS formula (SURVEY.md section 4)."""
import math

import pytest
import torch

from conftest import checksum, diffeats_features, regenerate_case
from oracle import aas_oracle as O


def _cases(golden):
    return {c["name"]: c for c in golden["cases"]}


@pytest.mark.parametrize("name", ["small_f32", "small_f16", "small_bf16", "ragged_f16", "sd15_up0_f16_cute16",
                                  "sd15_up0_bf16", "sd15_up0_alpha_sweep", "dit_xl2_f16_packed", "sd15_mid_f16",
                                  "sdxl_like_f16"])
def test_oracle_matches_reference_run(golden, name):
    case = _cases(golden)[name]
    images = regenerate_case(case)
    # the regenerated inputs are the ones the reference saw
    for im, cs in zip(images, case["checksums"]):
        assert [checksum(t) for t in im] == cs
    dtype = images[0][0].dtype
    for sim in ("cosine", "mse"):
        ref32 = case["scores"][sim]["reference_fp32_math"]
        refnat = case["scores"][sim]["reference_native_dtype"]
        for (a, b), r32, rn in zip(case["pairs"], ref32, refnat):
            t0 = O.aas_pair_score(*images[a], *images[b], mode=sim, tier="T0")
            t1 = O.aas_pair_score(*images[a], *images[b], mode=sim, tier="T1")
            # fp32 run of the reference's own lines vs float64 restatement on identical inputs
            # (torch's fp32 CPU cosine over 655 360 elements differs from fp64 by ~1.3e-5 relative)
            assert t0 == pytest.approx(r32, rel=5e-5, abs=1e-7)
            # rounding the attention outputs to the storage dtype moves the score by far less than the tolerance
            tol = {torch.float32: 1e-6, torch.float16: 2e-4, torch.bfloat16: 2e-3}[dtype]
            assert t1 == pytest.approx(t0, rel=tol, abs=tol * 1e-2)
            # the reference's native-dtype score is the fp32 one quantised to fp16 / bf16 (plus its own noise)
            qtol = {torch.float32: 5e-5, torch.float16: 2e-3, torch.bfloat16: 1.6e-2}[dtype]
            assert rn == pytest.approx(t0, rel=qtol, abs=qtol * 1e-2)


def test_alpha_sweep_is_monotone(golden):
    case = _cases(golden)["sd15_up0_alpha_sweep"]
    cos = case["scores"]["cosine"]["reference_fp32_math"]
    mse = case["scores"]["mse"]["reference_fp32_math"]
    assert cos[0] == pytest.approx(1.0, abs=1e-4) and mse[0] == pytest.approx(0.0, abs=1e-6)
    assert all(cos[i] > cos[i + 1] for i in range(len(cos) - 1))
    assert all(mse[i] < mse[i + 1] for i in range(len(mse) - 2))


def _img(seed, shape=(2, 2, 64, 40), dtype=torch.float32, alpha=0.7):
    from diffsim_b200 import synth

    m = synth.SynthModel(*shape, seed=2334)
    g = torch.Generator().manual_seed(seed)
    base = m.new_base(torch.Generator().manual_seed(99))
    return m.image(base, alpha, dtype, "sd", g)


def test_identities():
    A, B = _img(1), _img(2)
    # score(A, A) = 1 / 0
    assert O.aas_pair_score(*A, *A, mode="cosine") == pytest.approx(1.0, abs=1e-12)
    assert O.aas_pair_score(*A, *A, mode="mse") == pytest.approx(0.0, abs=1e-12)
    # symmetric at the Q/K/V boundary
    assert O.aas_pair_score(*A, *B) == pytest.approx(O.aas_pair_score(*B, *A), rel=1e-12)
    s = O.aas_pair_score(*A, *B)
    qb, kb, vb = B
    # joint permutation of B's key/value rows
    perm = torch.randperm(kb.shape[2], generator=torch.Generator().manual_seed(3))
    d1 = O.aas_directional(*A, kb, vb)
    assert O.aas_directional(*A, kb[:, :, perm], vb[:, :, perm]) == pytest.approx(d1, rel=1e-10)
    # softmax shift: adding one vector to every key row changes nothing
    shift = torch.randn(1, 1, 1, kb.shape[3], generator=torch.Generator().manual_seed(4))
    assert O.aas_directional(A[0], A[1] + shift, A[2], kb + shift, vb) == pytest.approx(d1, rel=1e-6)  # fp32 add rounds
    # cosine is invariant to scaling all V, mse scales with c^2
    c = 4.0  # a power of two: the scaling itself is exact in fp32
    assert O.aas_pair_score(A[0], A[1], A[2] * c, qb, kb, vb * c) == pytest.approx(s, rel=1e-10)
    m1 = O.aas_pair_score(*A, *B, mode="mse")
    assert O.aas_pair_score(A[0], A[1], A[2] * c, qb, kb, vb * c, mode="mse") == pytest.approx(m1 * c * c, rel=1e-10)


def test_attention_matches_torch_sdpa():
    import torch.nn.functional as F

    q, k, v = _img(5)
    ours = O.attention(q, k, v)
    ref = F.scaled_dot_product_attention(q.double(), k.double(), v.double(), dropout_p=0.0, is_causal=False)
    assert (ours - ref).abs().max().item() < 1e-12
    # explicit scale (metrics/clip_i.py:121)
    ours = O.attention(q, k, v, scale=0.3)
    ref = F.scaled_dot_product_attention(q.double(), k.double(), v.double(), scale=0.3)
    assert (ours - ref).abs().max().item() < 1e-12


def test_cosine_eps_semantics():
    import torch.nn.functional as F

    x = torch.zeros(16)
    y = torch.randn(16, generator=torch.Generator().manual_seed(1))
    assert O.flat_cosine(x, y) == float(F.cosine_similarity(x.unsqueeze(0), y.unsqueeze(0)))
    x = torch.full((16,), 1e-9, dtype=torch.float64)
    assert O.flat_cosine(x, x) == pytest.approx(float(F.cosine_similarity(x.unsqueeze(0), x.unsqueeze(0))), rel=1e-9)


def test_minmax_cosine_matches_reference_helper(golden):
    ex = golden["extra"]["diffeats_minmax_cosine"]
    fa, fb = diffeats_features()
    assert [checksum(fa), checksum(fb)] == ex["checksums"]
    got = O.minmax_cosine(fa, fb)
    assert got == pytest.approx(ex["score_f16_inputs"], rel=2e-6)


def test_twoafc_rules():
    ab, ac = [0.5, 0.2, 0.3, 0.9], [0.4, 0.2, 0.1, 0.1]
    assert O.twoafc(ab, ac, "cosine") == (3, 2, [True, False, True, True])
    assert O.twoafc(ab, ac, "mse")[0] == 0  # lower is closer; ties are never correct


def test_matrix_is_the_pair_formula():
    imgs = [_img(10 + i, alpha=0.5 + 0.1 * i) for i in range(3)]
    dm = O.aas_matrix([i[0] for i in imgs], [i[1] for i in imgs], [i[2] for i in imgs])
    S = O.symmetrize(dm)
    for i in range(3):
        assert dm[i, i].item() == pytest.approx(1.0, abs=1e-12)
        for j in range(3):
            assert S[i, j].item() == pytest.approx(O.aas_pair_score(*imgs[i], *imgs[j]), rel=1e-12)


def test_projection_oracle_matches_the_reference_capture_lines():
    """oracle.project_qkv (float64) against the reference's own capture arithmetic -- attn.to_q / to_k / to_v +
    head-split views, diffsim/hacked_attn.py:61-69,74-77 -- in fp32 (1e-4 of max(|y|, 0.05)) and fp16 (1.5e-3: one fp16 ulp on top)."""
    from diffsim_b200 import synth

    m = synth.SynthModel(2, 4, 64, 40, seed=2334)
    g = torch.Generator().manual_seed(1)
    hidden = m.hidden(m.new_base(g), 0.7, g)
    for dtype, tol in ((torch.float32, 1e-4), (torch.float16, 1.5e-3)):
        w = m.linear_weights(dtype)
        C = w.shape[1]
        h = hidden.to(dtype)
        ref = O.reference_capture(h, w[:C], w[C:2 * C], w[2 * C:], heads=4)
        got = O.project_qkv(h, w)
        for r, o in zip(ref, got):
            o = o.view(2, 64, 4, 40).transpose(1, 2)
            assert r.shape == (2, 4, 64, 40) and r.stride()[-1] == 1
            err = ((r.double() - o).abs() / o.abs().clamp_min(0.05)).max().item()
            assert err < tol, (dtype, err)
