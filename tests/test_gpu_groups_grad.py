"""Grouped K5 backward (ds_aas_groups_bwd, ds_aas_pairs_bwd, ds_aas_triplets_bwd) on a B200.

The contract: the gradient buffers end up bit for bit as after one ds_aas_dir_bwd call per entry, in list order, on the
slices of the caches (that path is tested against the float64 rounding model in test_gpu_grad_edges.py).
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

D_ALL = (40, 64, 72, 80, 128, 160)
DTYPES = (torch.float16, torch.bfloat16)
LAYOUTS = ("sd", "dit", "contig")


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _cache(N, B, H, S, D, dtype, layout, dev, g, base=None):
    """(q, k, v) caches of N correlated images, (N,B,H,S,D) views in the given memory layout."""
    if base is None:
        base = torch.randn(3, B, S, H, D, generator=g)
    x = (base[None] + 0.7 * torch.randn(N, 3, B, S, H, D, generator=g)).to(dtype).to(dev)
    if layout == "dit":   # packed qkv: (N, B, S, 3, H, D)
        packed = x.permute(0, 2, 3, 1, 4, 5).contiguous()
        return tuple(packed[:, :, :, i].permute(0, 1, 3, 2, 4) for i in range(3))
    if layout == "sd":    # head-split views of (N, B, S, H*D)
        return tuple(x[:, i].contiguous().permute(0, 1, 3, 2, 4) for i in range(3))
    return tuple(x[:, i].permute(0, 1, 3, 2, 4).contiguous() for i in range(3))


def _zeros(*ts):
    return [torch.zeros(t.shape, dtype=torch.float32, device=t.device) for t in ts]


def _loop(q, ks, vs, k, v, gq, go, kv, d_dir, mode, scale, grads):
    """The per-entry reference: ds_aas_dir_bwd once per entry, in list order, into slices of `grads`."""
    from diffsim_b200 import ops

    dq, dks, dvs, dk, dv = grads
    for g, i in enumerate(gq):
        for t in range(go[g], go[g + 1]):
            j = kv[t]
            ops.aas_dir_bwd(q[i], ks[i], vs[i], k[j], v[j], d_dir[t:t + 1], mode, scale,
                            grads=(dq[i], dks[i], dvs[i], dk[j], dv[j]))


def _same(a, b):
    assert a.shape == b.shape
    assert torch.equal(a.view(torch.int32), b.view(torch.int32)), (a - b).abs().max().item()


# query image 0 in two groups; image 0 paired with itself; image 1 repeated; image 4 only a kv image
GQ, GO, KV = [0, 3, 0, 2], [0, 3, 4, 5, 7], [1, 2, 0, 1, 4, 1, 3]


def _run_groups(D, dtype, layout, mode, aliased, Sq=160, Skv=160, scale=None, seed=0):
    from diffsim_b200 import ops

    dev = _cuda()
    g = torch.Generator().manual_seed(seed)
    B, H, N = 2, 2, 5
    q, k, v = _cache(N, B, H, Sq, D, dtype, layout, dev, g)
    if Skv != Sq:
        _, k, v = _cache(N, B, H, Skv, D, dtype, layout, dev, g)
    if aliased:
        ks, vs = k, v
    else:   # separate self caches (same images, other memory)
        ks, vs = k.clone(), v.clone()
    d_dir = torch.randn(len(KV), generator=g).to(dev)
    want = _zeros(q, ks, vs, k, v)
    if aliased:
        want[1], want[2] = want[3], want[4]
    _loop(q, ks, vs, k, v, GQ, GO, KV, d_dir, mode, scale, want)
    got = ops.aas_groups_bwd(q, ks, vs, k, v, GQ, GO, KV, d_dir, mode, scale)
    if aliased:
        assert got[1] is got[3] and got[2] is got[4]
    for a, b in zip(got, want):
        _same(a, b)
    assert all(torch.isfinite(a).all() and a.abs().sum() > 0 for a in got)


CASES = [(D, dt, LAYOUTS[i % 3], ("cosine", "mse")[(i // 3) % 2]) for i, (D, dt) in
         enumerate([(D, dt) for D in D_ALL for dt in DTYPES])]


@pytest.mark.parametrize("D,dtype,layout,mode", CASES)
def test_groups_bwd_is_bitwise_the_per_entry_loop(D, dtype, layout, mode):
    _run_groups(D, dtype, layout, mode, aliased=True)


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("mode", ("cosine", "mse"))
def test_groups_bwd_separate_self_gradients(layout, mode):
    _run_groups(64, torch.bfloat16, layout, mode, aliased=False)


@pytest.mark.parametrize("D", (64, 160))
def test_groups_bwd_ragged_and_unequal_lengths(D):
    _run_groups(D, torch.float16, "sd", "cosine", aliased=True, Sq=193, Skv=129, scale=0.11)
    _run_groups(D, torch.bfloat16, "contig", "mse", aliased=False, Sq=77, Skv=250)


def _pairs_case(D, dtype, layout, mode, seed=1):
    dev = _cuda()
    g = torch.Generator().manual_seed(seed)
    q, k, v = _cache(5, 2, 2, 144, D, dtype, layout, dev, g)
    pairs = [[0, 1], [2, 0], [1, 1], [3, 4], [0, 1]]
    return q, k, v, pairs, torch.randn(len(pairs), generator=g).to(dev)


@pytest.mark.parametrize("D,dtype,layout,mode", [(160, torch.float16, "sd", "cosine"), (72, torch.bfloat16, "dit", "mse"),
                                                 (40, torch.float16, "contig", "mse"), (128, torch.bfloat16, "sd", "cosine")])
def test_pairs_and_triplets_bwd_are_bitwise_the_loop(D, dtype, layout, mode):
    from diffsim_b200 import ops

    q, k, v, pairs, d = _pairs_case(D, dtype, layout, mode)
    want = _zeros(q, k, v)
    gq = [x for a, b in pairs for x in (a, b)]
    kv = [x for a, b in pairs for x in (b, a)]
    _loop(q, k, v, k, v, gq, list(range(len(gq) + 1)), kv, d.repeat_interleave(2) * 0.5, mode, None,
          (want[0], want[1], want[2], want[1], want[2]))
    for a, b in zip(ops.aas_pairs_bwd(q, k, v, pairs, d, mode), want):
        _same(a, b)

    trips = [[0, 1, 2], [3, 0, 0], [4, 1, 3]]
    g = torch.Generator().manual_seed(7)
    d_ab, d_ac = torch.randn(3, generator=g).to(q.device), torch.randn(3, generator=g).to(q.device)
    gq, go, kv, dd = [], [0], [], []
    for t, (r, l, rt) in enumerate(trips):
        gq += [r, l, rt]
        kv += [l, rt, r, r]
        go += [go[-1] + 2, go[-1] + 3, go[-1] + 4]
        dd += [d_ab[t] * 0.5, d_ac[t] * 0.5, d_ab[t] * 0.5, d_ac[t] * 0.5]
    want = _zeros(q, k, v)
    _loop(q, k, v, k, v, gq, go, kv, torch.stack(dd), mode, None, (want[0], want[1], want[2], want[1], want[2]))
    for a, b in zip(ops.aas_triplets_bwd(q, k, v, trips, d_ab, d_ac, mode), want):
        _same(a, b)


def test_autograd_pairs_match_the_loop_and_aas_score():
    from diffsim_b200 import diffsim, ops

    q, k, v, pairs, _ = _pairs_case(160, torch.float16, "sd", "cosine")
    with torch.no_grad():
        n0 = ops.LAUNCHES
        s0 = ops.aas_pairs(q, k, v, pairs)
        n_plain = ops.LAUNCHES - n0
    leaves = [t.detach().requires_grad_() for t in (q, k, v)]
    n0 = ops.LAUNCHES
    s = ops.aas_pairs(*leaves, pairs)
    assert ops.LAUNCHES - n0 == n_plain
    assert torch.equal(s.detach(), s0) and s.grad_fn is not None
    s.sum().backward()
    want = ops.aas_pairs_bwd(q, k, v, pairs, torch.ones(len(pairs), device=q.device))
    for leaf, w in zip(leaves, want):
        assert torch.equal(leaf.grad, w.to(leaf.dtype))
    # against one aas_score per pair (the per-pair autograd path), at K5's loose tolerance
    ref = [t.detach().requires_grad_() for t in (q, k, v)]
    total = 0
    for a, b in pairs:
        total = total + diffsim.aas_score((ref[0][a], ref[1][a], ref[2][a]), (ref[0][b], ref[1][b], ref[2][b]),
                                          match_reference_dtype=False)
    total.sum().backward()
    for leaf, r in zip(leaves, ref):
        err = (leaf.grad.double() - r.grad.double()).norm() / r.grad.double().norm()
        assert err < 2e-2, err.item()


@pytest.mark.parametrize("which", ("ab", "ac", "both"))
@pytest.mark.parametrize("round_scores", (False, True))
def test_triplet_hinge_loss_gradients(which, round_scores):
    from diffsim_b200 import ops

    q, k, v, _, _ = _pairs_case(64, torch.bfloat16, "sd", "cosine", seed=3)
    trips = [[0, 1, 2], [3, 4, 0]]
    with torch.no_grad():
        ref = ops.aas_triplets(q, k, v, trips, round_scores=round_scores)
    leaves = [t.detach().requires_grad_() for t in (q, k, v)]
    ab, ac, counts, flags = ops.aas_triplets(*leaves, trips, round_scores=round_scores)
    assert torch.equal(ab.detach(), ref[0]) and torch.equal(ac.detach(), ref[1]) and torch.equal(counts, ref[2])
    assert not counts.requires_grad and not flags.requires_grad
    loss = {"ab": -ab.sum(), "ac": ac.sum(), "both": torch.relu(0.1 - (ab - ac)).sum()}[which]
    loss.backward()
    # the gradients the loss hands to ab and ac (None for the one it does not use)
    active = ((0.1 - (ref[0] - ref[1])) > 0).float().cpu()
    gab = {"ab": -torch.ones(2), "ac": None, "both": -active}[which]
    gac = {"ab": None, "ac": torch.ones(2), "both": active}[which]
    gab, gac = [None if x is None else x.to(q.device) for x in (gab, gac)]
    want = ops.aas_triplets_bwd(q, k, v, trips, gab, gac)
    for leaf, w in zip(leaves, want):
        assert torch.equal(leaf.grad, w.to(leaf.dtype))


def test_torch_ops_build_no_graph():
    import diffsim_b200.torch_ops  # noqa: F401

    q, k, v, pairs, _ = _pairs_case(64, torch.float16, "sd", "cosine")
    leaves = [t.detach().requires_grad_() for t in (q, k, v)]
    idx = torch.tensor(pairs, dtype=torch.int32, device=q.device)
    # the dispatcher may attach its not-implemented autograd node, but the impl must not record ops' autograd Functions
    s = torch.ops.diffsim_b200.aas_pairs(*leaves, idx)
    ab, ac, _, _ = torch.ops.diffsim_b200.aas_triplets(*leaves, torch.tensor([[0, 1, 2]], device=q.device))
    for out in (s, ab, ac):
        assert out.grad_fn is None or "AAS" not in out.grad_fn.name(), out.grad_fn.name()
        assert out.grad_fn is None or all(f is None or "AAS" not in f.name() for f, _ in out.grad_fn.next_functions)


def test_repeated_chunked_and_two_stream_calls_are_bitwise_equal(monkeypatch):
    from diffsim_b200 import ops

    q, k, v, pairs, d = _pairs_case(80, torch.float16, "dit", "cosine")
    a = ops.aas_pairs_bwd(q, k, v, pairs, d)
    b = ops.aas_pairs_bwd(q, k, v, pairs, d)
    for x, y in zip(a, b):
        _same(x, y)
    g = torch.Generator().manual_seed(2)
    dd = torch.randn(len(KV), generator=g).to(q.device)
    full = ops.aas_groups_bwd(q, k, v, k, v, GQ, GO, KV, dd)
    one = ops.aas_pairs_bwd(q, k, v, pairs[:1], d[:1])
    monkeypatch.setattr(ops, "GROUPS_BWD_WORKSPACE_CAP", 1)   # one group (pair) per library call
    for x, y in zip(ops.aas_pairs_bwd(q, k, v, pairs, d), a):
        _same(x, y)
    for x, y in zip(ops.aas_groups_bwd(q, k, v, k, v, GQ, GO, KV, dd), full):
        _same(x, y)
    monkeypatch.undo()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s1):
        r1 = ops.aas_pairs_bwd(q, k, v, pairs, d)
    with torch.cuda.stream(s2):
        r2 = ops.aas_pairs_bwd(q, k, v, pairs[:1], d[:1])
    torch.cuda.synchronize()
    for x, y in zip(r1, a):
        _same(x, y)
    for x, y in zip(r2, one):
        _same(x, y)


def test_out_of_range_index_gives_nan_and_keeps_guard_bands():
    from diffsim_b200 import ops

    q, k, v, _, _ = _pairs_case(64, torch.float16, "sd", "cosine")
    dev = q.device
    guards = []
    grads = []
    for t in (q, k, v):
        buf = torch.full((t.shape[0], t.shape[1], t.shape[3], t.shape[2], t.shape[4] + 8), 7.0, device=dev)
        grads.append(buf[..., 4:4 + t.shape[4]].permute(0, 1, 3, 2, 4))
        guards.append(buf)
    ops.aas_pairs_bwd(q, k, v, [[0, 9]], torch.ones(1, device=dev), grads=grads)
    for buf, gr in zip(guards, grads):
        assert torch.isnan(gr).all()
        assert (buf[..., :4] == 7.0).all() and (buf[..., -4:] == 7.0).all()
