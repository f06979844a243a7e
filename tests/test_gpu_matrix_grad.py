"""Matrix K5 backward (ds_aas_matrix_bwd, ops.aas_matrix_bwd, autograd through ops.aas_matrix) on a B200.

Every case is checked two ways, as in test_gpu_grad_edges.py: tight, against the float64 rounding model
oracle.aas_matrix_grad_oracle.matrix_grads_rounded (per-row and Frobenius metrics); loose, against the exact float64
gradient with test_gpu_grad's TOL.  The column-cache gradients are, besides, bitwise those of ds_aas_groups_bwd on the
row-major list: they receive the same cross terms in the same order.
"""
import pytest
import torch

from oracle import aas_grad_oracle as G
from oracle import aas_matrix_grad_oracle as M
from test_gpu_grad import TOL

pytestmark = pytest.mark.gpu

# Tight tier: (per-row error, Frobenius error) against the rounding model, at most 4x the worst observed over this file on
# a B200 (power limit 1000 W): fp16 per-row 8.4e-4, Frobenius 2.7e-5; bf16 per-row 4.8e-3, Frobenius 5.6e-5.
TIGHT = {torch.float16: (3.2e-3, 1e-4), torch.bfloat16: (1.9e-2, 2.2e-4)}
# Two paths that round the self terms' dO differently -- the grouped backward (each fy_rc rounded to 16 bits), a fold per
# column block -- against one fold: the same metrics, at most 4x the worst observed over this file on that B200: fp16
# per-row 2.2e-3, Frobenius 3.2e-4; bf16 per-row 5.1e-2, Frobenius 4.2e-3.
TIGHT_PATHS = {torch.float16: (8e-3, 1.2e-3), torch.bfloat16: (2e-1, 1.6e-2)}

D_ALL = (40, 64, 72, 80, 128, 160)
DTYPES = (torch.float16, torch.bfloat16)
LAYOUTS = ("sd", "dit", "contig")
NR, NC = 3, 5


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _fro(x, ref):
    e = float((x.double() - ref.double()).norm())
    n = float(ref.double().norm())
    return e / n if n > 0 else (0.0 if e == 0 else float("inf"))


def _cache(N, B, H, S, D, dtype, layout, dev, g, base):
    """(q, k, v) caches of N images correlated through `base`, (N,B,H,S,D) views in the given memory layout."""
    x = (base[None] + 0.7 * torch.randn(N, 3, B, S, H, D, generator=g)).to(dtype).to(dev)
    if layout == "dit":   # packed qkv: (N, B, S, 3, H, D)
        packed = x.permute(0, 2, 3, 1, 4, 5).contiguous()
        return tuple(packed[:, :, :, i].permute(0, 1, 3, 2, 4) for i in range(3))
    if layout == "sd":    # head-split views of (N, B, S, H*D)
        return tuple(x[:, i].contiguous().permute(0, 1, 3, 2, 4) for i in range(3))
    return tuple(x[:, i].permute(0, 1, 3, 2, 4).contiguous() for i in range(3))


def _case(D, dtype, layout, S=136, seed=0, B=2, H=2):
    """rows (q, k_self, v_self) of NR images, columns (k, v) of NC other images, and a d_Dm."""
    dev = _cuda()
    g = torch.Generator().manual_seed(seed)
    base = torch.randn(3, B, S, H, D, generator=g)
    q, ks, vs = _cache(NR, B, H, S, D, dtype, layout, dev, g, base)
    _, k, v = _cache(NC, B, H, S, D, dtype, layout, dev, g, base)
    return q, ks, vs, k, v, torch.randn(NR, NC, generator=g).to(dev)


def _stored(q, k, v, scale=None):
    from diffsim_b200 import ops

    return ops.attn_fwd(q, k, v, scale, out=torch.empty(q.shape, dtype=q.dtype, device=q.device))


def _model(q, ks, vs, k, v, d, mode, scale=None):
    X = torch.stack([torch.stack([_stored(q[r], k[c], v[c], scale) for c in range(k.shape[0])]) for r in range(q.shape[0])])
    Y = torch.stack([_stored(q[r], ks[r], vs[r], scale) for r in range(q.shape[0])])
    return M.matrix_grads_rounded(q, ks, vs, k, v, X, Y, d, mode, scale)


def _check(name, got, model, exact, dtype):
    rows = [G.max_row_err(a, b) for a, b in zip(got, model)]
    fro = [_fro(a, b) for a, b in zip(got, model)]
    loose = [_fro(a, b) for a, b in zip(got, exact)]
    fmt = lambda es: " ".join(f"{e:.2e}" for e in es)  # noqa: E731
    print(f"{name} {str(dtype)[6:]}: vs model per-row {fmt(rows)} rel {fmt(fro)} | vs exact rel {fmt(loose)}")
    assert all(t.dtype == torch.float32 and torch.isfinite(t).all() and t.abs().sum() > 0 for t in got)
    tol_rows, tol_fro = TIGHT[dtype]
    assert max(rows) <= tol_rows, rows
    assert max(fro) <= tol_fro, fro
    assert max(loose) <= TOL[dtype], loose


def _close(name, got, ref, dtype):
    rows = [G.max_row_err(a, b) for a, b in zip(got, ref)]
    fro = [_fro(a, b) for a, b in zip(got, ref)]
    print(f"{name} {str(dtype)[6:]}: per-row {' '.join(f'{e:.2e}' for e in rows)} rel {' '.join(f'{e:.2e}' for e in fro)}")
    tol_rows, tol_fro = TIGHT_PATHS[dtype]
    assert max(rows) <= tol_rows and max(fro) <= tol_fro, (rows, fro)


def _same(a, b):
    assert a.shape == b.shape
    assert torch.equal(a.view(torch.int32), b.view(torch.int32)), (a - b).abs().max().item()


CASES = [(D, dt, LAYOUTS[i % 3], ("cosine", "mse")[(i // 3) % 2]) for i, (D, dt) in
         enumerate([(D, dt) for D in D_ALL for dt in DTYPES])]


@pytest.mark.parametrize("D,dtype,layout,mode", CASES + [(160, torch.float16, "contig", "cosine"),
                                                        (64, torch.bfloat16, "sd", "mse")])
def test_matrix_bwd_against_the_models(D, dtype, layout, mode):
    from diffsim_b200 import ops

    q, ks, vs, k, v, d = _case(D, dtype, layout, seed=D)
    got = ops.aas_matrix_bwd(q, ks, vs, k, v, d, mode)
    _check(f"matrix_bwd D={D} {layout} {mode}", got, _model(q, ks, vs, k, v, d, mode),
           M.matrix_grads(q, ks, vs, k, v, d, mode, None, dtype), dtype)


@pytest.mark.parametrize("D,dtype,mode", [(64, torch.float16, "cosine"), (160, torch.bfloat16, "mse")])
def test_matrix_bwd_ragged_length_and_scale(D, dtype, mode):
    from diffsim_b200 import ops

    q, ks, vs, k, v, d = _case(D, dtype, "sd", S=193, seed=3)
    got = ops.aas_matrix_bwd(q, ks, vs, k, v, d, mode, 0.11)
    _check(f"matrix_bwd ragged D={D} {mode}", got, _model(q, ks, vs, k, v, d, mode, 0.11),
           M.matrix_grads(q, ks, vs, k, v, d, mode, 0.11, dtype), dtype)


@pytest.mark.parametrize("mode", ("cosine", "mse"))
@pytest.mark.parametrize("D,dtype,layout", [(160, torch.float16, "sd"), (72, torch.bfloat16, "dit")])
def test_column_gradients_are_bitwise_the_grouped_backward(D, dtype, layout, mode):
    from diffsim_b200 import ops

    q, ks, vs, k, v, d = _case(D, dtype, layout, seed=11)
    got = ops.aas_matrix_bwd(q, ks, vs, k, v, d, mode)
    gq = list(range(NR))
    go = [r * NC for r in range(NR + 1)]
    kv = [c for _ in range(NR) for c in range(NC)]
    ref = ops.aas_groups_bwd(q, ks, vs, k, v, gq, go, kv, d.reshape(-1), mode)
    _same(got[3], ref[3])
    _same(got[4], ref[4])
    _close(f"vs grouped D={D} {mode}", got[:3], ref[:3], dtype)


def test_infonce_through_the_shared_cache_matches_the_pairs():
    from diffsim_b200 import ops, scoring

    q, k, v, _, _, _ = _case(64, torch.float16, "sd", seed=5)
    n = q.shape[0]

    def loss_of(S):
        return torch.nn.functional.cross_entropy(S / 0.05, torch.arange(n, device=S.device))

    leaves = [t.detach().requires_grad_() for t in (q, k, v)]
    cache = scoring.QKVCache(*leaves)
    loss_of(scoring.symmetrize(scoring.aas_matrix_local(cache, cache))).backward()
    ref = [t.detach().requires_grad_() for t in (q, k, v)]
    pairs = [[i, j] for i in range(n) for j in range(i, n)]
    s = ops.aas_pairs(*ref, pairs)
    S = torch.zeros(n, n, device=q.device)
    iu = torch.tensor(pairs, device=q.device).t()
    S = S.index_put((iu[0], iu[1]), s).index_put((iu[1], iu[0]), s)
    loss_of(S).backward()
    for a, b in zip(leaves, ref):
        assert _fro(a.grad.float(), b.grad.float()) <= TOL[torch.float16]


def test_forward_is_bitwise_with_and_without_grad():
    from diffsim_b200 import ops

    q, ks, vs, k, v, _ = _case(80, torch.bfloat16, "dit", seed=2)
    with torch.no_grad():
        n0 = ops.LAUNCHES
        plain = ops.aas_matrix(q, ks, vs, k, v)
        n_plain = ops.LAUNCHES - n0
    leaves = [t.detach().requires_grad_() for t in (q, ks, vs, k, v)]
    n0 = ops.LAUNCHES
    dm = ops.aas_matrix(*leaves)
    assert ops.LAUNCHES - n0 == n_plain
    assert dm.grad_fn is not None and torch.equal(dm.detach(), plain)
    g = torch.randn_like(dm)
    dm.backward(g)
    want = ops.aas_matrix_bwd(q, ks, vs, k, v, g)
    for leaf, w in zip(leaves, want):
        assert torch.equal(leaf.grad, w.to(leaf.dtype))


def test_out_torch_op_and_sharded_build_no_graph(tmp_path):
    import torch.distributed as dist

    import diffsim_b200.torch_ops  # noqa: F401
    from diffsim_b200 import ops, scoring

    q, k, v, _, _, _ = _case(64, torch.float16, "sd", seed=6)
    leaves = [t.detach().requires_grad_() for t in (q, k, v)]
    out = torch.empty(NR, NR, device=q.device)
    assert ops.aas_matrix(leaves[0], leaves[1], leaves[2], leaves[1], leaves[2], out=out).grad_fn is None
    t = torch.ops.diffsim_b200.aas_matrix(leaves[0], leaves[1], leaves[2], leaves[1], leaves[2])
    assert t.grad_fn is None or "AAS" not in t.grad_fn.name()
    assert torch.equal(t.detach(), out)
    dist.init_process_group("nccl", init_method=f"file://{tmp_path}/store", rank=0, world_size=1,
                            device_id=q.device)
    try:
        dm = scoring.aas_matrix_sharded(scoring.QKVCache(*leaves))
    finally:
        dist.destroy_process_group()
    assert dm.grad_fn is None and not dm.requires_grad
    assert torch.equal(dm, out)


def test_repeated_and_two_stream_calls_are_bitwise_equal():
    from diffsim_b200 import ops

    q, ks, vs, k, v, d = _case(128, torch.float16, "contig", seed=8)
    a = ops.aas_matrix_bwd(q, ks, vs, k, v, d)
    for x, y in zip(ops.aas_matrix_bwd(q, ks, vs, k, v, d), a):
        _same(x, y)
    one = ops.aas_matrix_bwd(q[:1], ks[:1], vs[:1], k, v, d[:1])
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s1):
        r1 = ops.aas_matrix_bwd(q, ks, vs, k, v, d)
    with torch.cuda.stream(s2):
        r2 = ops.aas_matrix_bwd(q[:1], ks[:1], vs[:1], k, v, d[:1])
    torch.cuda.synchronize()
    for x, y in zip(r1, a):
        _same(x, y)
    for x, y in zip(r2, one):
        _same(x, y)


def test_chunking(monkeypatch):
    from diffsim_b200 import _native as N, ops

    q, ks, vs, k, v, d = _case(72, torch.float16, "sd", seed=9)
    full = ops.aas_matrix_bwd(q, ks, vs, k, v, d)
    lib = N.load()
    ws = lambda r, c: lib.ds_aas_matrix_bwd_workspace_bytes(ops._desc(q[:r], 5), ops._desc(k[:c], 5))  # noqa: E731
    # blocks of one row: bitwise one call
    monkeypatch.setattr(ops, "GROUPS_BWD_WORKSPACE_CAP", ws(1, NC))
    assert len(ops._matrix_spans(NR, NC, ws)) == NR
    for x, y in zip(ops.aas_matrix_bwd(q, ks, vs, k, v, d), full):
        _same(x, y)
    # column blocks of two: the cross terms are unchanged, each block folds its own self term
    monkeypatch.setattr(ops, "GROUPS_BWD_WORKSPACE_CAP", ws(1, 2))
    assert len(ops._matrix_spans(NR, NC, ws)) == NR * 3
    cut = ops.aas_matrix_bwd(q, ks, vs, k, v, d)
    _same(cut[3], full[3])
    _same(cut[4], full[4])
    _close("column blocks", cut[:3], full[:3], torch.float16)
    # one shared cache (rows = columns): the blocks' self gradients go through a separate buffer
    monkeypatch.undo()
    kk, vv = k[:NR], v[:NR]
    shared = ops.aas_matrix_bwd(q, kk, vv, kk, vv, d[:, :NR])
    assert shared[1] is shared[3]
    monkeypatch.setattr(ops, "GROUPS_BWD_WORKSPACE_CAP", ws(1, NR))
    cut = ops.aas_matrix_bwd(q, kk, vv, kk, vv, d[:, :NR])
    tol_rows, tol_fro = TIGHT[torch.float16]   # the same terms, summed in another order
    for a, b in zip(cut, shared):
        assert G.max_row_err(a, b) <= tol_rows and _fro(a, b) <= tol_fro


SENTINEL = -1234.5


def test_strided_grads_accumulate_and_wide_ldd():
    from diffsim_b200 import ops

    q, ks, vs, k, v, d = _case(64, torch.bfloat16, "sd", seed=10)
    want = ops.aas_matrix_bwd(q, ks, vs, k, v, d)
    wide = torch.full((NR, NC + 3), float("nan"), device=q.device)
    wide[:, :NC] = d
    bufs, grads = [], []
    for t in (q, ks, vs, k, v):   # (N, B, S, H, D + 8) fp32 with guard bands, viewed as (N, B, H, S, D)
        buf = torch.full((t.shape[0], t.shape[1], t.shape[3], t.shape[2], t.shape[4] + 8), SENTINEL, device=q.device)
        g = buf[..., 4:4 + t.shape[4]].permute(0, 1, 3, 2, 4)
        g.zero_()
        bufs.append(buf)
        grads.append(g)
    got = ops.aas_matrix_bwd(q, ks, vs, k, v, wide[:, :NC], grads=grads)
    assert all(a is b for a, b in zip(got, grads))
    for buf, g, w in zip(bufs, grads, want):
        _same(g.contiguous(), w)
        assert (buf[..., :4] == SENTINEL).all() and (buf[..., -4:] == SENTINEL).all()
    ops.aas_matrix_bwd(q, ks, vs, k, v, wide[:, :NC], grads=grads)   # added into
    for g, w in zip(grads, want):
        assert torch.allclose(g, 2 * w, rtol=1e-5, atol=1e-6 * float(w.abs().max()))
    # a non-unit inner stride of d_Dm is made contiguous
    for x, y in zip(ops.aas_matrix_bwd(q, ks, vs, k, v, d.t().contiguous().t()), want):
        _same(x, y)
