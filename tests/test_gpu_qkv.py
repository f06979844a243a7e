"""K4 on the GPU: the QKV projection of the hooked layer (diffsim/hacked_attn.py:61-69,74-77; DiT: diffsim_dit.py:21-23)
against the float64 oracle, through the C ABI, and the hook-input scoring path built on it."""
import pytest
import torch

from oracle import aas_oracle as O

pytestmark = pytest.mark.gpu


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return "cuda"


def _ulp_close(got: torch.Tensor, ref64: torch.Tensor, dtype) -> None:
    """got (16-bit) must be the float64 result rounded to dtype, give or take ONE unit in the last place (fp32
    accumulation order differs from the oracle's float64): tolerance stated here as eps * |ref| + eps * 2^-6."""
    eps = torch.finfo(dtype).eps
    err = (got.double().cpu() - ref64).abs()
    tol = eps * ref64.abs() + eps * 2.0 ** -6
    bad = (err > tol).sum().item()
    assert bad == 0, f"{bad} of {err.numel()} elements off by more than one ulp (max err {err.max().item():.3e})"
    exact = (got.cpu() == ref64.to(dtype)).float().mean().item()
    assert exact > 0.97, f"only {exact:.3f} of the elements are the correctly rounded result"


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_sd_projection_matches_oracle(dtype):
    dev = _cuda()
    from diffsim_b200 import ops, synth

    m = synth.SynthModel(2, 8, 256, 160, seed=2334)
    g = torch.Generator().manual_seed(11)
    hidden = torch.stack([m.hidden(m.new_base(g), a, g) for a in (1.0, 0.8, 0.3)]).to(dtype)   # (3,2,256,1280)
    w = m.linear_weights(dtype)                                                                 # (3840,1280)
    q, k, v = ops.qkv_project(hidden.to(dev), w.to(dev))
    rq, rk, rv = O.project_qkv(hidden, w)
    assert q.shape == (3, 2, 256, 1280)
    for got, ref in ((q, rq), (k, rk), (v, rv)):
        _ulp_close(got, ref, dtype)


def test_dit_packed_projection_with_bias_and_ragged_rows():
    dev = _cuda()
    from diffsim_b200 import ops

    g = torch.Generator().manual_seed(3)
    C, rows = 1152, 2 * 256 - 56                      # rows not a multiple of the 128-row tile
    hidden = torch.randn(rows, C, generator=g).half()
    w = (torch.randn(3 * C, C, generator=g) / C ** 0.5).half()
    b = torch.randn(3 * C, generator=g).half()
    (packed,) = ops.qkv_project(hidden.to(dev), w.to(dev), b.to(dev), n_outputs=1)
    (ref,) = O.project_qkv(hidden, w, b, n_outputs=1)
    assert packed.shape == (rows, 3 * C)
    _ulp_close(packed, ref, torch.float16)
    # the reference's views of the packed activation (diffsim_dit.py:22-23) are then consumed in place
    qkv = packed.view(1, rows, 3, 16, 72).permute(2, 0, 3, 1, 4)
    assert qkv[0].stride()[-1] == 1


@pytest.mark.parametrize("rows,c_in,n_out", [(1000, 1280, 3840), (512, 320, 960), (777, 64, 192), (4096, 1152, 3456),
                                             (5000, 640, 1920), (4096, 512, 3000)])
def test_one_cta_and_cta_pair_gemm_kernels_are_bitwise_equal(rows, c_in, n_out):
    """The 1-CTA (128 x 256) and CTA-pair (256 x 256) GEMM kernels accumulate every output over k in the same order, so
    the projection is bitwise the same whichever serves it.  The last shape's 1000 columns per output are not a multiple of 64: the pair
    kernel then writes 16-bit outputs without TMA stores."""
    dev = _cuda()
    from diffsim_b200 import _native, ops

    lib = _native.load()
    g = torch.Generator().manual_seed(rows + c_in)
    h = torch.randn(rows, c_in, generator=g).half()
    w = (torch.randn(n_out, c_in, generator=g) / c_in ** 0.5).half()
    b = torch.randn(n_out, generator=g).half()
    outs = {}
    try:
        for variant in (0, 2):
            assert lib.ds_debug_set_gemm_variant(variant) == variant
            outs[variant] = ops.qkv_project(h.to(dev), w.to(dev), b.to(dev), 3)
    finally:
        lib.ds_debug_set_gemm_variant(-1)
    for one_cta, pair in zip(outs[0], outs[2]):
        assert torch.equal(one_cta, pair)
    for got, ref in zip(outs[2], O.project_qkv(h, w, b)):
        _ulp_close(got, ref, torch.float16)


def test_projection_writes_straight_into_a_cache_and_scores_match():
    dev = _cuda()
    from diffsim_b200 import scoring, synth

    B, H, S, D = 2, 8, 256, 160
    m = synth.SynthModel(B, H, S, D, seed=2334)
    g = torch.Generator().manual_seed(5)
    base = m.new_base(g)
    hidden = torch.stack([m.hidden(base, a, g) for a in (1.0, 0.9, 0.5, 0.1)]).half()
    w = m.linear_weights(torch.float16)
    big = scoring.QKVCache.empty(6, B, H, S, D, torch.float16, dev)          # larger than needed: row strides are the cache's
    cache = scoring.project_cache(hidden.to(dev), w.to(dev), H, out=big)
    assert cache.n_images == 4 and cache.q.data_ptr() == big.q.data_ptr()
    pairs = [(0, 1), (0, 2), (0, 3), (1, 2)]
    got = scoring.score_pairs(cache, pairs, "cosine").cpu().double()
    # oracle: float64 projection rounded to fp16 (what the reference's nn.Linear returns), then the pair formula
    rq, rk, rv = O.project_qkv(hidden, w, round_to=torch.float16)
    split = lambda t: t.view(B, S, H, D).transpose(1, 2)  # noqa: E731
    imgs = [(split(rq[i]), split(rk[i]), split(rv[i])) for i in range(4)]
    ref = torch.tensor([O.aas_pair_score(*imgs[a], *imgs[b]) for a, b in pairs], dtype=torch.float64)
    rel = ((got - ref).abs() / ref.abs().clamp_min(1e-9)).max().item()
    assert rel < 1e-3, f"scores through the projection differ from the oracle by {rel:.2e} (tolerance 1e-3 relative)"
    assert got[0] > got[1] > got[2]                                           # similarity ordering survives


def test_host_hidden_scorer_equals_the_device_resident_path():
    dev = _cuda()
    from diffsim_b200 import ops, scoring, synth

    B, H, S, D = 2, 8, 256, 160
    T = 20
    hid, w = synth.device_hidden(B, H, S, D, 3 * T, torch.float16, dev, seed=7, pin_host=True)
    scorer = scoring.HostHiddenTripletScorer((B, H, S, D), w, None, torch.float16, dev, chunk_triplets=8)
    c1, c2 = scorer.score(hid, T)
    cache = scoring.project_cache(hid.to(dev), w, H)
    trips = torch.arange(3 * T, dtype=torch.int32, device=dev).view(-1, 3)
    _, _, counts, _ = ops.aas_triplets(cache.q, cache.k, cache.v, trips, "cosine")
    assert (c1, c2) == tuple(int(x) for x in counts.cpu())
    assert scorer.h2d_bytes == 3 * T * B * S * H * D * 2 and scorer.d2h_bytes == 8


def test_projection_rejects_bad_arguments_loudly():
    dev = _cuda()
    from diffsim_b200 import _native as N, ops

    h = torch.zeros(4, 100, dtype=torch.float16, device=dev)          # 100 channels: not a multiple of 8
    w = torch.zeros(24, 100, dtype=torch.float16, device=dev)
    with pytest.raises(N.DiffSimError):
        ops.qkv_project(h, w)
    h32 = torch.zeros(4, 64, dtype=torch.float32, device=dev)
    with pytest.raises(RuntimeError):
        ops.qkv_project(h32, torch.zeros(24, 64, dtype=torch.float32, device=dev))
