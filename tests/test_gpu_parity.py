"""Parity of the CUDA path (through the C ABI) with the CPU oracle and the reference-generated golden vectors.

Tolerances (north_star): scores within 1e-3 relative for 16-bit inputs (checked against the oracle's float64
arithmetic on the SAME 16-bit inputs: tier T1 rounds the attention outputs to the storage dtype like the kernel
and like the reference's SDPA outputs; tier T0 rounds nothing), 1e-5 for the fp32 reductions; decisions
(2AFC, argmax / top-k) identical wherever the oracle's margin exceeds the tolerance band.
"""
import pytest
import torch

from conftest import checksum, diffeats_features, regenerate_case
from oracle import aas_oracle as O

pytestmark = pytest.mark.gpu

REL_16BIT = 1e-3


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from diffsim_b200 import _native as N

    N.check(N.load().ds_device_ok())  # loud failure if the extension or an sm_100 device is missing
    return "cuda"


def _rel(got, ref):
    got, ref = got.double().cpu(), ref.double().cpu()
    return ((got - ref).abs() / ref.abs().clamp_min(1e-9)).max().item()


def _rand_qkv(B, H, Sq, Skv, D, dtype, seed, dev):
    g = torch.Generator().manual_seed(seed)

    def mk(S, std):
        return (torch.randn(B, S, H * D, generator=g) * std).to(dtype).to(dev).view(B, S, H, D).transpose(1, 2)

    return mk(Sq, 1.5), mk(Skv, 1.5), mk(Skv, 1.0)


# ------------------------------------------------------------------------------------------------------
# K1 as an SDPA replacement
# ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(2, 8, 256, 256, 160), (2, 8, 64, 64, 160), (2, 16, 256, 256, 72), (2, 8, 256, 256, 80),
                                   (2, 8, 256, 256, 40), (1, 4, 256, 256, 64), (1, 4, 256, 256, 128),
                                   (1, 12, 50, 50, 64), (1, 6, 257, 200, 64), (2, 3, 100, 130, 160), (1, 2, 1, 1, 64)])
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_attn_fwd_matches_oracle(shape, dtype):
    dev = _cuda()
    from diffsim_b200 import ops

    B, H, Sq, Skv, D = shape
    q, k, v = _rand_qkv(B, H, Sq, Skv, D, dtype, 0, dev)
    out = ops.attn_fwd(q, k, v)
    assert out.shape == q.shape and out.dtype == dtype
    ref = O.attention(q.cpu(), k.cpu(), v.cpu())
    tol = 2e-2 if dtype == torch.bfloat16 else 4e-3  # one ulp of the storage dtype at |o| ~ 3, plus P rounding
    assert torch.isfinite(out).all()
    assert (out.double().cpu() - ref).abs().max().item() < tol


def test_attn_fwd_explicit_scale_and_dit_layout():
    dev = _cuda()
    from diffsim_b200 import ops, synth

    m = synth.SynthModel(2, 16, 256, 72, seed=5)
    q, k, v = m.image(m.new_base(), 0.9, torch.float16, layout="dit")
    packed = torch.empty(2, 256, 3, 16, 72, dtype=torch.float16, device=dev)
    for i, t in enumerate((q, k, v)):
        packed[:, :, i] = t.permute(0, 2, 1, 3).to(dev)
    qkv = packed.permute(2, 0, 3, 1, 4)  # diffsim/diffsim_dit.py:22-23
    assert qkv[0].stride() == (256 * 3 * 16 * 72, 72, 3 * 16 * 72, 1)
    out = ops.attn_fwd(qkv[0], qkv[1], qkv[2])
    assert (out.double().cpu() - O.attention(q, k, v)).abs().max().item() < 4e-3
    out = ops.attn_fwd(qkv[0], qkv[1], qkv[2], scale=0.05)  # metrics/clip_i.py:121 passes an explicit scale
    assert (out.double().cpu() - O.attention(q, k, v, scale=0.05)).abs().max().item() < 4e-3


# kv lengths beyond one 256-row group (SDXL up_blocks 1024 / 4096 tokens, SD-1.5 up_blocks[1..2]): the online
# softmax with the lazy running maximum; "ramp" inputs make later kv rows dominate so that the rescale path runs.
@pytest.mark.parametrize("case", [(1, 2, 128, 320, 64, torch.float16, "random"), (1, 2, 200, 448, 64, torch.float16, "random"),
                                  (2, 4, 1024, 1024, 64, torch.float16, "random"), (1, 2, 1024, 1024, 80, torch.float16, "random"),
                                  (1, 2, 512, 4096, 40, torch.float16, "random"), (1, 2, 4096, 4096, 64, torch.bfloat16, "random"),
                                  (1, 1, 300, 700, 160, torch.float16, "random"), (1, 2, 256, 256, 160, torch.float16, "ramp"),
                                  (1, 2, 256, 1024, 64, torch.float16, "ramp"), (1, 2, 128, 2048, 64, torch.bfloat16, "ramp")])
def test_attn_fwd_long_kv_and_rescale_path(case):
    dev = _cuda()
    from diffsim_b200 import ops

    B, H, Sq, Skv, D, dtype, kind = case
    q, k, v = _rand_qkv(B, H, Sq, Skv, D, dtype, Skv + D, dev)
    if kind == "ramp":
        ramp = (1.0 + 9.0 * torch.arange(Skv, device=k.device).float() / Skv).view(1, 1, Skv, 1)
        k = (k.float() * ramp).to(dtype)
    out = ops.attn_fwd(q, k, v)
    ref = O.attention(q.cpu(), k.cpu(), v.cpu())
    tol = 2e-2 if dtype == torch.bfloat16 else 4e-3
    err = (out.double().cpu() - ref).abs().max().item()
    assert torch.isfinite(out).all() and err <= tol * max(1.0, ref.abs().max().item()), err


@pytest.mark.parametrize("shape,dtype", [((2, 4, 640, 64), torch.float16), ((1, 2, 1024, 64), torch.bfloat16),
                                         ((2, 10, 1024, 64), torch.float16)])
def test_aas_pairs_long_kv(shape, dtype):
    """AAS pair scores at SDXL-like token counts (diffsim/diffsim_xl.py:135-155) against the T1 oracle."""
    dev = _cuda()
    from diffsim_b200 import ops, synth

    m = synth.SynthModel(*shape, seed=2334)
    images, pairs = synth.make_pairs(m, 2, dtype, seed=9)
    q, k, v = synth.stack_cache(images, dev)
    for sim in ("cosine", "mse"):
        got = ops.aas_pairs(q, k, v, pairs, sim).cpu().double()
        ref = torch.tensor([O.aas_pair_score(*images[a], *images[b], mode=sim) for a, b in pairs], dtype=torch.float64)
        assert ((got - ref).abs() / ref.abs().clamp_min(1e-9)).max().item() < REL_16BIT


def test_unsupported_requests_fail_loudly():
    dev = _cuda()
    from diffsim_b200 import ops
    from diffsim_b200._native import DiffSimError

    q, k, v = _rand_qkv(1, 1, 64, 64, 48, torch.float16, 0, dev)
    with pytest.raises(DiffSimError, match="head dim"):
        ops.attn_fwd(q, k, v)
    q = torch.randn(1, 1, 64, 64, device=dev)  # fp32 attention is not a thing the reference runs
    with pytest.raises(DiffSimError):
        ops.attn_fwd(q, q, q)


# ------------------------------------------------------------------------------------------------------
# fused AAS scores vs the reference-generated golden vectors
# ------------------------------------------------------------------------------------------------------
GOLDEN_GPU_CASES = ["small_f16", "small_bf16", "ragged_f16", "sd15_up0_f16_cute16", "sd15_up0_bf16",
                    "sd15_up0_alpha_sweep", "dit_xl2_f16_packed", "sd15_mid_f16"]


@pytest.mark.parametrize("name", GOLDEN_GPU_CASES)
@pytest.mark.parametrize("sim", ["cosine", "mse"])
def test_aas_pairs_match_reference_run(golden, name, sim):
    dev = _cuda()
    from diffsim_b200 import ops, synth

    case = {c["name"]: c for c in golden["cases"]}[name]
    images = regenerate_case(case)
    q, k, v = synth.stack_cache(images, dev)
    got = ops.aas_pairs(q, k, v, case["pairs"], sim).cpu().double()
    ref32 = torch.tensor(case["scores"][sim]["reference_fp32_math"], dtype=torch.float64)
    t1 = torch.tensor([O.aas_pair_score(*images[a], *images[b], mode=sim) for a, b in case["pairs"]], dtype=torch.float64)
    # within 1e-3 of the reference's own lines evaluated in fp32 on the same 16-bit inputs, and of the oracle
    assert ((got - ref32).abs() / ref32.abs().clamp_min(1e-6)).max().item() < REL_16BIT
    assert ((got - t1).abs() / t1.abs().clamp_min(1e-6)).max().item() < REL_16BIT
    # the reference's native fp16/bf16 score is our score up to the quantisation of the storage dtype
    refn = torch.tensor(case["scores"][sim]["reference_native_dtype"], dtype=torch.float64)
    q_tol = 2e-3 if images[0][0].dtype == torch.float16 else 1.6e-2
    assert ((got - refn).abs() / refn.abs().clamp_min(1e-6)).max().item() < q_tol


def test_alpha_sweep_decisions(golden):
    """score(A,A) = 1 and the ranking over alpha is the reference's."""
    dev = _cuda()
    from diffsim_b200 import ops, synth

    case = {c["name"]: c for c in golden["cases"]}["sd15_up0_alpha_sweep"]
    images = regenerate_case(case)
    q, k, v = synth.stack_cache(images, dev)
    got = ops.aas_pairs(q, k, v, case["pairs"], "cosine").cpu()
    assert got[0].item() == pytest.approx(1.0, abs=1e-4)
    ref = torch.tensor(case["scores"]["cosine"]["reference_fp32_math"])
    assert torch.argsort(got, descending=True).tolist() == torch.argsort(ref, descending=True).tolist()


def test_pair_score_is_symmetric_and_deterministic():
    dev = _cuda()
    from diffsim_b200 import ops, synth

    m = synth.SynthModel(2, 8, 256, 160, seed=2334)
    images, pairs = synth.make_pairs(m, 6, torch.float16, seed=77)
    q, k, v = synth.stack_cache(images, dev)
    fwd = ops.aas_pairs(q, k, v, pairs, "cosine")
    rev = ops.aas_pairs(q, k, v, [(b, a) for a, b in pairs], "cosine")
    again = ops.aas_pairs(q, k, v, pairs, "cosine")
    assert torch.equal(fwd, rev)     # (dir(a->b) + dir(b->a)) / 2 either way: same partials, same order
    assert torch.equal(fwd, again)   # bit-reproducible
    # every image against itself
    same = ops.aas_pairs(q, k, v, [(i, i) for i in range(len(images))], "mse")
    assert same.abs().max().item() == 0.0


def test_triplets_share_the_reference_image_and_decide_like_the_oracle():
    dev = _cuda()
    from diffsim_b200 import ops, synth

    m = synth.SynthModel(2, 8, 256, 160, seed=2334)
    images, trips = synth.make_triplets(m, 24, torch.float16, seed=3, near_tie_fraction=0.25)
    q, k, v = synth.stack_cache(images, dev)
    for sim in ("cosine", "mse"):
        ab, ac, counts, flags = ops.aas_triplets(q, k, v, trips, sim)
        # identical to scoring the two pairs separately (the shared self attention changes nothing)
        pa = ops.aas_pairs(q, k, v, [(r, l) for r, l, _ in trips], sim)
        pc = ops.aas_pairs(q, k, v, [(r, rt) for r, _, rt in trips], sim)
        assert torch.equal(ab, pa) and torch.equal(ac, pc)
        o_ab = [O.aas_pair_score(*images[r], *images[l], mode=sim) for r, l, _ in trips]
        o_ac = [O.aas_pair_score(*images[r], *images[rt], mode=sim) for r, _, rt in trips]
        assert _rel(ab, torch.tensor(o_ab)) < REL_16BIT and _rel(ac, torch.tensor(o_ac)) < REL_16BIT
        # decisions: identical wherever the oracle's margin is outside the tolerance band; near-ties are counted
        _, _, o_flags = O.twoafc(o_ab, o_ac, sim)
        near = 0
        for t in range(len(trips)):
            margin = abs(o_ab[t] - o_ac[t]) / max(abs(o_ab[t]), abs(o_ac[t]), 1e-9)
            if margin > 2 * REL_16BIT:
                assert bool(flags[t].item()) == o_flags[t]
            else:
                near += 1
        assert near <= len(trips) // 2
        assert int(counts[0].item()) == int(flags.sum().item())
        # the stand-alone decision kernel agrees
        c2, f2 = ops.twoafc(ab, ac, sim)
        assert torch.equal(c2, counts) and torch.equal(f2, flags)


def test_round_scores_emulates_reference_dtype():
    dev = _cuda()
    from diffsim_b200 import ops, synth

    m = synth.SynthModel(2, 4, 64, 64, seed=2334)
    images, trips = synth.make_triplets(m, 8, torch.bfloat16, seed=9)
    q, k, v = synth.stack_cache(images, dev)
    ab, ac, _, _ = ops.aas_triplets(q, k, v, trips, "cosine", round_scores=True)
    assert torch.equal(ab, ab.to(torch.bfloat16).float())  # representable in the input dtype
    ab32, _, _, _ = ops.aas_triplets(q, k, v, trips, "cosine")
    assert (ab - ab32).abs().max().item() < 1e-2


# ------------------------------------------------------------------------------------------------------
# retrieval matrix
# ------------------------------------------------------------------------------------------------------
def test_matrix_matches_oracle_and_row_blocks_are_bitwise_identical():
    dev = _cuda()
    from diffsim_b200 import ops, scoring, synth

    m = synth.SynthModel(2, 4, 128, 64, seed=2334)
    images, labels = synth.make_styles(m, 5, 4, torch.float16, seed=4)
    q, k, v = synth.stack_cache(images, dev)
    dm = ops.aas_matrix(q, k, v, k, v, "cosine")
    ref = O.aas_matrix([i[0] for i in images], [i[1] for i in images], [i[2] for i in images])
    assert (dm.double().cpu() - ref).abs().max().item() < 1e-4
    assert dm.diagonal().sub(1).abs().max().item() < 1e-4
    # top-1 neighbour of every image is the oracle's (styles are well separated)
    S, Sref = scoring.symmetrize(dm).cpu(), O.symmetrize(ref)
    S.fill_diagonal_(-1)
    Sref.fill_diagonal_(-1)
    assert S.argmax(1).tolist() == Sref.argmax(1).tolist()
    assert all(labels[i] == labels[j] for i, j in enumerate(S.argmax(1).tolist()))
    # row-block sharding (what each rank computes) == the rows of the full matrix, bit for bit
    for r0, r1 in ((0, 7), (7, 20), (13, 14)):
        blk = ops.aas_matrix(q[r0:r1], k[r0:r1], v[r0:r1], k, v, "cosine")
        assert torch.equal(blk, dm[r0:r1])
    # pairs agree with the symmetrised matrix
    pairs = [(0, 1), (3, 17), (9, 9)]
    ps = ops.aas_pairs(q, k, v, pairs, "cosine").cpu()
    for (a, b), s in zip(pairs, ps.tolist()):
        assert s == pytest.approx(0.5 * (dm[a, b].item() + dm[b, a].item()), rel=1e-6)


@pytest.mark.parametrize("shape,dtype", [((2, 8, 256, 160), torch.float16), ((1, 3, 512, 64), torch.bfloat16),
                                         ((2, 2, 256, 72), torch.float16), ((1, 2, 1024, 40), torch.float16)])
def test_kv_multicast_over_cta_pairs_is_bitwise_neutral(shape, dtype):
    """K1 may run as clusters of two CTAs (the q tiles 2j, 2j + 1 of one (group, b, h)) that fetch every K/V tile once for both
    with TMA multicast; automatic for the N x N matrix, forced here for pair and triplet lists too.  Same arithmetic per
    CTA: every score is bitwise that of the unclustered launch."""
    dev = _cuda()
    from diffsim_b200 import _native, ops, synth

    lib = _native.load()
    m = synth.SynthModel(*shape, seed=2334)
    images, labels = synth.make_styles(m, 4, 3, dtype, seed=11)
    q, k, v = synth.stack_cache(images, dev)
    pairs = [(0, 1), (2, 7), (5, 5), (11, 3), (4, 9)]
    trips = torch.tensor([[0, 1, 2], [3, 4, 5], [6, 7, 8], [9, 10, 11], [1, 5, 9]], dtype=torch.int32, device=dev)
    out = {}
    try:
        for mc in (0, 1):
            assert lib.ds_debug_set_attn_mc(mc) == mc
            t = ops.aas_triplets(q, k, v, trips, "cosine")
            out[mc] = [ops.aas_pairs(q, k, v, pairs, "cosine"), ops.aas_pairs(q, k, v, pairs, "mse"),
                       ops.aas_matrix(q, k, v, k, v, "cosine"), ops.aas_matrix(q[:5], k[:5], v[:5], k, v, "mse")]
            out[mc] += [x for x in (t if isinstance(t, (tuple, list)) else [t]) if torch.is_tensor(x)]
    finally:
        lib.ds_debug_set_attn_mc(-1)
    assert len(out[0]) == len(out[1]) >= 5
    for a, b in zip(out[0], out[1]):
        assert torch.equal(a, b)
    assert torch.equal(ops.aas_matrix(q, k, v, k, v, "cosine"), out[0][2])     # automatic mode (multicast on for the matrix)
    ref = torch.tensor([O.aas_pair_score(*images[a], *images[b], mode="cosine") for a, b in pairs], dtype=torch.float64)
    assert ((out[1][0].cpu().double() - ref).abs() / ref.abs().clamp_min(1e-9)).max().item() < REL_16BIT


# ------------------------------------------------------------------------------------------------------
# K2 / K3
# ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float32])
@pytest.mark.parametrize("P,E", [(1, 655360), (5, 1000), (3, 8191), (16, 589824), (2, 7), (1, 1)])
def test_pair_reduce(dtype, P, E):
    dev = _cuda()
    from diffsim_b200 import ops

    g = torch.Generator().manual_seed(P * 1000 + E)
    x = torch.randn(P, E, generator=g) * 0.7 + 0.2
    y = 0.6 * x + 0.4 * torch.randn(P, E, generator=g)
    xd, yd = x.to(dtype).to(dev), y.to(dtype).to(dev)
    for mode in ("cosine", "mse", "minmax_cosine"):
        if mode == "minmax_cosine" and E == 1:
            continue  # (max - min) == 0: the reference divides by zero (NaN)
        got = ops.pair_reduce(xd, yd, mode).cpu()
        ref = torch.tensor([O.similarity(xd[p].cpu(), yd[p].cpu(), mode) for p in range(P)])
        assert _rel(got, ref) < 1e-5, mode


def test_pair_reduce_full_size_properties():
    """Size-independent properties at the benchmark size: cos(x,x)=1, mse(x,x)=0, scale invariance, linearity."""
    dev = _cuda()
    from diffsim_b200 import ops

    P, E = 64, 655360
    x = torch.randn(P, E, device=dev).half()
    y = torch.randn(P, E, device=dev).half()
    assert (ops.pair_reduce(x, x, "cosine") - 1).abs().max().item() < 1e-6
    assert ops.pair_reduce(x, x, "mse").abs().max().item() == 0.0
    c1 = ops.pair_reduce(x, y, "cosine")
    c2 = ops.pair_reduce(x * 2, y * 0.5, "cosine")  # powers of two: exact in fp16
    assert (c1 - c2).abs().max().item() < 1e-6
    m1 = ops.pair_reduce(x, y, "mse")
    m2 = ops.pair_reduce(x * 2, y * 2, "mse")
    assert ((m2 - 4 * m1).abs() / m1).max().item() < 1e-6
    assert torch.equal(c1, ops.pair_reduce(x, y, "cosine"))  # deterministic


def test_minmax_cosine_matches_reference_helper(golden):
    dev = _cuda()
    from diffsim_b200 import ops

    ex = golden["extra"]["diffeats_minmax_cosine"]
    fa, fb = diffeats_features()
    assert [checksum(fa), checksum(fb)] == ex["checksums"]
    got = ops.pair_reduce(fa.reshape(1, -1).to(dev), fb.reshape(1, -1).to(dev), "minmax_cosine")
    assert got.item() == pytest.approx(ex["score_f16_inputs"], rel=1e-5)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("nr,nc,L", [(128, 128, 64), (160, 96, 200), (300, 300, 4096), (40, 520, 10240), (1, 1, 8)])
def test_simmat(dtype, nr, nc, L):
    dev = _cuda()
    from diffsim_b200 import ops

    g = torch.Generator().manual_seed(nr + nc + L)
    a = (torch.randn(nr, L, generator=g) * 0.5 + 0.1).to(dtype).to(dev)
    b = (torch.randn(nc, L, generator=g) * 0.5 - 0.2).to(dtype).to(dev)
    for mode in ("cosine", "minmax_cosine"):
        got = ops.simmat(a, b, mode).double().cpu()
        ad, bd = a.double().cpu(), b.double().cpu()
        if mode == "minmax_cosine":
            ad = (ad - ad.amin(1, keepdim=True)) / (ad.amax(1, keepdim=True) - ad.amin(1, keepdim=True))
            bd = (bd - bd.amin(1, keepdim=True)) / (bd.amax(1, keepdim=True) - bd.amin(1, keepdim=True))
        ref = (ad @ bd.T) / (ad.norm(dim=1, keepdim=True).clamp_min(1e-8) * bd.norm(dim=1).clamp_min(1e-8))
        assert (got - ref).abs().max().item() < 1e-5
    # the matrix agrees with the per-pair reduction kernel
    pr = ops.pair_reduce(a[: min(nr, nc)], b[: min(nr, nc)], "cosine").cpu()
    assert (ops.simmat(a, b, "cosine").diagonal().cpu() - pr).abs().max().item() < 1e-5


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("nr,nc,L", [(512, 512, 4096), (777, 520, 10008), (600, 1030, 200), (2032, 2032, 1024 + 8)])
def test_simmat_k_blocked_operand_copies(dtype, nr, nc, L):
    """Large operands go through k-blocked copies written by the statistics pass (automatic above 1.5 GB per operand; forced
    here at test sizes).  Same MMAs in the same order: the result is bitwise that of the row-major path -- ragged row counts
    (tiles overhanging the copy's padded rows), L with a partly filled last k block, self and rows x other."""
    dev = _cuda()
    from diffsim_b200 import _native, ops

    lib = _native.load()
    g = torch.Generator().manual_seed(nr * 3 + nc + L)
    a = (torch.randn(nr, L, generator=g) * 0.5 + 0.1).to(dtype).to(dev)
    b = (torch.randn(nc, L, generator=g) * 0.5 - 0.2).to(dtype).to(dev)
    try:
        out = {}
        for blocked in (0, 1):
            assert lib.ds_debug_set_simmat_blocked(blocked) == blocked
            out[blocked] = [ops.simmat(a, b, "cosine"), ops.simmat(a, None, "minmax_cosine"), ops.simmat(b, None, "cosine")]
    finally:
        lib.ds_debug_set_simmat_blocked(-1)
    for x, y in zip(out[0], out[1]):
        assert torch.equal(x, y)
    ref = O.simmat(a[:48].cpu(), b.cpu(), "cosine")
    assert (out[1][0][:48].double().cpu() - ref).abs().max().item() < 2e-5
    # a view with a leading dimension larger than L
    wide = torch.zeros(nr, L + 24, dtype=dtype, device=dev)
    wide[:, :L] = a
    try:
        lib.ds_debug_set_simmat_blocked(1)
        assert torch.equal(ops.simmat(wide[:, :L], b, "cosine"), out[1][0])
    finally:
        lib.ds_debug_set_simmat_blocked(-1)


def test_simmat_self_is_symmetric_with_unit_diagonal():
    dev = _cuda()
    from diffsim_b200 import ops

    f = torch.randn(200, 5000, device=dev).half()
    C = ops.simmat(f)
    assert (C.diagonal() - 1).abs().max().item() < 1e-5
    assert (C - C.t()).abs().max().item() < 1e-6


@pytest.mark.parametrize("n,L", [(300, 4096), (1000, 2048), (130, 200), (2032, 1024)])
def test_simmat_symmetric_schedule_equals_the_full_one(n, L):
    """rows == cols takes the upper-triangle tile schedule (about half the MMAs) and one statistics pass; the result must
    agree with the general schedule and be exactly symmetric."""
    dev = _cuda()
    from diffsim_b200 import ops

    g = torch.Generator().manual_seed(n + L)
    f = (torch.randn(n, L, generator=g) * 0.8 + 0.1).half().to(dev)
    for mode in ("cosine", "minmax_cosine"):
        sym = ops.simmat(f, None, mode)
        full = ops.simmat(f, f.clone(), mode)       # a different buffer: the general schedule
        # the two schedules may cut L into different numbers of fp32 partials: equal up to that regrouping
        assert (sym - full).abs().max().item() < 2e-5
        assert torch.equal(sym, sym.t())            # mirrored, not recomputed
    ref = O.simmat(f[:64].cpu(), f.cpu(), "cosine")
    got = ops.simmat(f, None, "cosine")[:64].double().cpu()
    assert (got - ref).abs().max().item() < 2e-4
