"""Aligned Attention Score between images of different token counts on a B200.

Two captures made at different image sizes (SD-1.5 up_blocks at 512^2: S = 256, at 768^2: S = 576; two SDXL aspect
buckets) score against each other: in dir(a -> b) = sim(Attn(Q_a, K_b, V_b), Attn(Q_a, K_a, V_a)) both attentions have
image a's S_a rows, so the flat similarity is defined (diffsim/diffsim.py:177-197).  The self item walks S_self = S_a kv
rows and the cross items S_cross = S_b, in K1 and in both K5 bodies.  Checked here: the forward against the float64
oracle and against the reference's own torch lines, the bitwise contracts of the grouped, matrix and multicast forms,
the gradients against float64 autograd, the bitwise contracts of the grouped and matrix backwards, and the rejection of
k / v (k_self / v_self) pairs of different lengths.
"""
import pytest
import torch

from oracle import aas_grad_oracle as G
from oracle import aas_matrix_grad_oracle as M
from oracle import aas_oracle as O
from test_gpu_grad import TOL

pytestmark = pytest.mark.gpu

REL_16BIT = 1e-3                                               # test_gpu_parity's score tolerance against the oracle
REF_NATIVE = {torch.float16: 2e-3, torch.bfloat16: 1.6e-2}     # ... and against the reference's fp16 / bf16 score
D_ALL = (40, 64, 72, 80, 128, 160)
DTYPES = (torch.float16, torch.bfloat16)
LAYOUTS = ("sd", "dit", "contig")


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _tokens(base, S, g, noise):
    """base (3, B, S0, H, D) resampled to S tokens (nearest source token) plus noise: a capture of the same content at
    another resolution."""
    S0 = base.shape[2]
    idx = (torch.arange(S) * S0) // S
    return base[:, :, idx] + noise * torch.randn(base.shape[:2] + (S,) + base.shape[3:], generator=g)


def _layout(x, dtype, layout, dev):
    """(q, k, v) of x (N, 3, B, S, H, D) as (N,B,H,S,D) views in the given memory layout."""
    x = x.to(dtype).to(dev)
    if layout == "dit":   # packed qkv: (N, B, S, 3, H, D)
        packed = x.permute(0, 2, 3, 1, 4, 5).contiguous()
        return tuple(packed[:, :, :, i].permute(0, 1, 3, 2, 4) for i in range(3))
    if layout == "sd":    # head-split views of (N, B, S, H*D)
        return tuple(x[:, i].contiguous().permute(0, 1, 3, 2, 4) for i in range(3))
    return tuple(x[:, i].permute(0, 1, 3, 2, 4).contiguous() for i in range(3))


def _caches(lengths, B, H, D, dtype, layout, seed=0, noise=0.7, S0=None):
    """One (q, k, v) cache of N images per entry (N, S) of lengths, all of one content (correlated scores)."""
    dev = _cuda()
    g = torch.Generator().manual_seed(seed)
    base = torch.randn(3, B, S0 or max(S for _, S in lengths), H, D, generator=g)
    return [_layout(torch.stack([_tokens(base, S, g, noise) for _ in range(N)]), dtype, layout, dev) for N, S in lengths]


def _rel(got, ref):
    got, ref = got.double().cpu(), ref.double().cpu()
    return ((got - ref).abs() / ref.abs().clamp_min(1e-9)).max().item()


def _same(a, b):
    assert a.shape == b.shape
    assert torch.equal(a.view(torch.int32), b.view(torch.int32)), (a - b).abs().max().item()


# ------------------------------------------------------------------------------------------------------
# forward
# ------------------------------------------------------------------------------------------------------
def _score_case(SA, SB, D, dtype, layout, mode):
    from diffsim_b200.diffsim import aas_score

    (qa, ka, va), (qb, kb, vb) = _caches([(1, SA), (1, SB)], 2, 2, D, dtype, layout, seed=SA + SB + D)
    A, B = (qa[0], ka[0], va[0]), (qb[0], kb[0], vb[0])
    got = aas_score(A, B, mode, match_reference_dtype=False).cpu().double().reshape(())
    cpu = [t.cpu() for t in (*A, *B)]
    t1 = torch.tensor(O.aas_pair_score(*cpu, mode=mode), dtype=torch.float64)
    native = O.reference_pair_score(*cpu, mode=mode).double().reshape(())
    print(f"AAS S=({SA},{SB}) D={D} {dtype} {layout} {mode}: {float(got):.6f} oracle {float(t1):.6f} "
          f"reference {float(native):.6f}")
    assert torch.isfinite(got)
    assert _rel(got, t1) < REL_16BIT
    assert _rel(got, native) < REF_NATIVE[dtype]
    # the reference-dtype form: the two directions rounded and added like the reference's fp16 / bf16 scalars
    ref_form = aas_score(A, B, mode)
    assert ref_form.dtype == dtype and ref_form.shape == ((1,) if mode == "cosine" else ())


LENGTH_CASES = [(256, 576, 160), (576, 256, 72), (256, 64, 40), (200, 1024, 128), (4096, 1024, 64)]


@pytest.mark.parametrize("SA,SB,D", LENGTH_CASES)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("mode", ("cosine", "mse"))
def test_score_at_mixed_lengths_matches_oracle_and_reference(SA, SB, D, dtype, mode):
    _score_case(SA, SB, D, dtype, LAYOUTS[(SA + SB) % 3], mode)


@pytest.mark.parametrize("D", D_ALL)
@pytest.mark.parametrize("dtype", DTYPES)
def test_score_at_mixed_lengths_every_head_dim_and_layout(D, dtype):
    for i, layout in enumerate(LAYOUTS):
        _score_case(256 if i != 1 else 320, 576 if i != 2 else 136, D, dtype, layout, ("cosine", "mse")[(i + D) % 2])


def _groups_one_by_one(q, ks, vs, k, v, gq, go, kv, mode):
    from diffsim_b200 import ops

    one, off = [0], [0, 1]
    out = []
    for g, i in enumerate(gq):
        for t in range(go[g], go[g + 1]):
            j = kv[t]
            out.append(ops.aas_groups(q[i:i + 1], ks[i:i + 1], vs[i:i + 1], k[j:j + 1], v[j:j + 1], one, off, one, mode))
    return torch.cat(out)


@pytest.mark.parametrize("short_self", (True, False))
@pytest.mark.parametrize("dtype", DTYPES)
def test_one_stream_mixes_single_and_multi_group_items(short_self, dtype):
    """Self item of one 256-row kv group against cross items of several (1024 rows), and the reverse, in one stream;
    the long items' keys ramp up along the sequence so that the lazy softmax maximum moves in later groups."""
    from diffsim_b200 import ops

    SA, SB = (256, 1024) if short_self else (1024, 256)
    (q, ks, vs), (_, k, v) = _caches([(2, SA), (3, SB)], 1, 4, 64, dtype, "sd", seed=3)
    for t, S in ((ks, SA), (k, SB)):
        if S > 256:
            t.mul_((1.0 + 3.0 * torch.arange(S, device=t.device).float() / S).view(1, 1, 1, S, 1).to(dtype))
    gq, go, kv = [0, 1, 0], [0, 3, 4, 6], [0, 1, 2, 2, 1, 0]
    for mode in ("cosine", "mse"):
        got = ops.aas_groups(q, ks, vs, k, v, gq, go, kv, mode)
        _same(got, _groups_one_by_one(q, ks, vs, k, v, gq, go, kv, mode))
        ref = torch.tensor([O.aas_directional(q[i].cpu(), ks[i].cpu(), vs[i].cpu(), k[kv[t]].cpu(), v[kv[t]].cpu(), mode)
                            for i, t in zip([0, 0, 0, 1, 0, 0], range(6))], dtype=torch.float64)
        assert _rel(got, ref) < REL_16BIT, (got, ref)


@pytest.mark.parametrize("D,dtype,layout", [(160, torch.float16, "sd"), (64, torch.bfloat16, "dit"),
                                            (72, torch.float16, "contig")])
def test_groups_matrix_and_multicast_are_bitwise_consistent(D, dtype, layout):
    """At mixed lengths: a grouped list equals its one-entry calls, the matrix equals its row-major list as groups, and
    K/V multicast over CTA pairs (forced on, forced off, automatic) changes no bit."""
    from diffsim_b200 import _native, ops

    lib = _native.load()
    (qa, ka, va), (qb, kb, vb) = _caches([(3, 512), (4, 192)], 2, 2, D, dtype, layout, seed=D)
    gq, go, kv = [0, 2, 1, 0], [0, 2, 5, 6, 8], [1, 3, 0, 1, 2, 3, 2, 0]
    out = {}
    try:
        for mc in (0, 1):
            assert lib.ds_debug_set_attn_mc(mc) == mc
            out[mc] = [ops.aas_groups(qa, ka, va, kb, vb, gq, go, kv, "cosine"),
                       ops.aas_groups(qb, kb, vb, ka, va, [3, 0], [0, 2, 3], [2, 0, 1], "mse"),
                       ops.aas_matrix(qa, ka, va, kb, vb, "cosine"), ops.aas_matrix(qb, kb, vb, ka, va, "mse")]
    finally:
        lib.ds_debug_set_attn_mc(-1)
    for a, b in zip(out[0], out[1]):
        _same(a, b)
    _same(ops.aas_matrix(qa, ka, va, kb, vb, "cosine"), out[0][2])
    _same(out[0][0], _groups_one_by_one(qa, ka, va, kb, vb, gq, go, kv, "cosine"))
    for (q, ks, vs, k, v), dm, mode in (((qa, ka, va, kb, vb), out[0][2], "cosine"), ((qb, kb, vb, ka, va), out[0][3], "mse")):
        nr, nc = q.shape[0], k.shape[0]
        rows = ops.aas_groups(q, ks, vs, k, v, list(range(nr)), [r * nc for r in range(nr + 1)], list(range(nc)) * nr, mode)
        _same(dm, rows.view(nr, nc))


def test_scores_between_two_caches_are_the_pair_scores():
    from diffsim_b200 import scoring
    from diffsim_b200.diffsim import aas_score

    (qa, ka, va), (qb, kb, vb) = _caches([(3, 256), (2, 576)], 2, 4, 80, torch.float16, "sd", seed=5)
    a, b = scoring.QKVCache(qa, ka, va), scoring.QKVCache(qb, kb, vb)
    for mode in ("cosine", "mse"):
        S = scoring.aas_scores_between(a, b, mode)
        assert S.shape == (3, 2) and S.dtype == torch.float32
        for i in range(3):
            for j in range(2):
                s = aas_score((qa[i], ka[i], va[i]), (qb[j], kb[j], vb[j]), mode, match_reference_dtype=False)
                _same(S[i, j].reshape(1), s.reshape(1))


def test_mismatched_key_value_lengths_are_rejected():
    from diffsim_b200 import _native, ops

    (q, ks, vs), (_, k, v) = _caches([(2, 256), (2, 384)], 1, 2, 64, torch.float16, "contig")
    one, off = [0], [0, 1]
    with pytest.raises(_native.DiffSimError, match="k and v"):
        ops.aas_groups(q, ks, vs, k, v[:, :, :, :256], one, off, one)
    with pytest.raises(_native.DiffSimError, match="k_self and v_self"):
        ops.aas_groups(q, ks, vs[:, :, :, :128], k, v, one, off, one)
    with pytest.raises(_native.DiffSimError, match="k and v"):
        ops.aas_matrix(q, ks, vs, k[:, :, :, :300], v)
    d = torch.ones(1, device=q.device)
    with pytest.raises(_native.DiffSimError):
        ops.aas_groups_bwd(q, ks, vs, k, v[:, :, :, :256], one, off, one, d)
    with pytest.raises(_native.DiffSimError):
        ops.aas_matrix_bwd(q, ks[:, :, :, :128], vs, k, v, torch.ones(2, 2, device=q.device))


# ------------------------------------------------------------------------------------------------------
# gradients
# ------------------------------------------------------------------------------------------------------
def _grad_rel(x, ref):
    return float((x.double() - ref.double()).norm() / ref.double().norm())


@pytest.mark.parametrize("SA,SB,D", [(256, 576, 160), (576, 256, 64), (200, 1024, 80)])
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("mode", ("cosine", "mse"))
def test_score_grads_at_mixed_lengths_match_float64(SA, SB, D, dtype, mode):
    from diffsim_b200 import ops
    from diffsim_b200.diffsim import aas_score

    (qa, ka, va), (qb, kb, vb) = _caches([(1, SA), (1, SB)], 2, 4, D, dtype, "sd", seed=SA * SB + D, noise=0.6)
    A, B = (qa[0], ka[0], va[0]), (qb[0], kb[0], vb[0])
    g = torch.full((1,), 0.5, device=qa.device)
    got = ops.pair_dirs_bwd(*A, *B, g, g, mode)
    ref = G.pair_score_grads(*A, *B, mode)
    errs = [_grad_rel(a, b) for a, b in zip(got, ref)]
    print(f"aas_score grads S=({SA},{SB}) D={D} {dtype} {mode}: " + " ".join(f"{e:.2e}" for e in errs))
    assert max(errs) <= TOL[dtype], errs
    # autograd through aas_score is the same fp32 result, cast
    leaves = [t.clone().requires_grad_(True) for t in (*A, *B)]
    s = aas_score(tuple(leaves[:3]), tuple(leaves[3:]), mode, match_reference_dtype=False)
    (s.sum() * 1e4).backward()
    f32 = ops.pair_dirs_bwd(*A, *B, torch.full((1,), 5e3, device=qa.device), torch.full((1,), 5e3, device=qa.device), mode)
    for t, r in zip(leaves, f32):
        assert torch.equal(t.grad, r.to(dtype))


def _groups_grad_oracle(q, ks, vs, k, v, gq, go, kv, d, mode):
    rnd = q.dtype
    leaves = G._leaves(q, ks, vs, k, v)
    lq, lks, lvs, lk, lv = leaves
    total = 0
    for g, i in enumerate(gq):
        for t in range(go[g], go[g + 1]):
            total = total + float(d[t]) * G.dir_value(lq[i], lks[i], lvs[i], lk[kv[t]], lv[kv[t]], mode, None, rnd)
    return torch.autograd.grad(total, leaves)


@pytest.mark.parametrize("D,dtype,layout,mode", [(160, torch.float16, "sd", "cosine"), (64, torch.bfloat16, "dit", "mse"),
                                                 (40, torch.float16, "contig", "mse"), (128, torch.bfloat16, "sd", "cosine")])
def test_groups_grads_at_mixed_lengths(D, dtype, layout, mode):
    """aas_groups_bwd against float64 autograd and, bitwise, against one aas_dir_bwd per entry in list order."""
    from diffsim_b200 import ops

    (q, ks, vs), (_, k, v) = _caches([(3, 136), (4, 300)], 2, 2, D, dtype, layout, seed=D + 1, noise=0.6)
    gq, go, kv = [0, 2, 0, 1], [0, 3, 4, 5, 7], [1, 2, 0, 3, 3, 0, 2]
    d = torch.randn(len(kv), generator=torch.Generator().manual_seed(D)).to(q.device)
    got = ops.aas_groups_bwd(q, ks, vs, k, v, gq, go, kv, d, mode)
    want = [torch.zeros(t.shape, dtype=torch.float32, device=t.device) for t in (q, ks, vs, k, v)]
    for g, i in enumerate(gq):
        for t in range(go[g], go[g + 1]):
            j = kv[t]
            ops.aas_dir_bwd(q[i], ks[i], vs[i], k[j], v[j], d[t:t + 1], mode,
                            grads=(want[0][i], want[1][i], want[2][i], want[3][j], want[4][j]))
    for a, b in zip(got, want):
        _same(a, b)
    ref = _groups_grad_oracle(q, ks, vs, k, v, gq, go, kv, d.cpu(), mode)
    errs = [_grad_rel(a, b) for a, b in zip(got, ref)]
    print(f"groups grads D={D} {dtype} {layout} {mode}: " + " ".join(f"{e:.2e}" for e in errs))
    assert max(errs) <= TOL[dtype], errs
    # autograd through aas_groups is the same backward
    leaves = [t.clone().requires_grad_(True) for t in (q, ks, vs, k, v)]
    (ops.aas_groups(*leaves, gq, go, kv, mode) * d).sum().backward()
    for t, r in zip(leaves, got):
        assert torch.equal(t.grad, r.to(dtype))


@pytest.mark.parametrize("SR,SC,D,dtype,layout,mode", [(256, 576, 160, torch.float16, "sd", "cosine"),
                                                        (320, 136, 72, torch.bfloat16, "dit", "mse"),
                                                        (130, 700, 64, torch.float16, "contig", "mse")])
def test_matrix_grads_at_mixed_lengths(SR, SC, D, dtype, layout, mode):
    """aas_matrix_bwd against float64 autograd (M.matrix_grads); each gradient family alone is bitwise the full call."""
    from diffsim_b200 import ops

    (q, ks, vs), (_, k, v) = _caches([(2, SR), (3, SC)], 2, 2, D, dtype, layout, seed=SR + SC, noise=0.6)
    d = torch.randn(2, 3, generator=torch.Generator().manual_seed(D)).to(q.device)
    full = ops.aas_matrix_bwd(q, ks, vs, k, v, d, mode)
    rows = ops.aas_matrix_bwd(q, ks, vs, k, v, d, mode, need_cols=False)
    cols = ops.aas_matrix_bwd(q, ks, vs, k, v, d, mode, need_rows=False)
    for a, b in zip(full[:3], rows[:3]):
        _same(a, b)
    for a, b in zip(full[3:], cols[3:]):
        _same(a, b)
    assert rows[3] is None and cols[0] is None
    exact = M.matrix_grads(q, ks, vs, k, v, d.cpu(), mode, None, dtype)
    errs = [_grad_rel(a, b) for a, b in zip(full, exact)]
    print(f"matrix grads S=({SR},{SC}) D={D} {dtype} {layout} {mode}: " + " ".join(f"{e:.2e}" for e in errs))
    assert max(errs) <= TOL[dtype], errs
    leaves = [t.clone().requires_grad_(True) for t in (q, ks, vs, k, v)]
    (ops.aas_matrix(*leaves, mode) * d).sum().backward()
    for t, r in zip(leaves, full):
        assert torch.equal(t.grad, r.to(dtype))
