"""K2 backward on the GPU: ds_pair_reduce_bwd against float64 torch autograd of the reference's expressions (per-row
relative error, oracle.reduce_grad_oracle.ROW_TOL), ties, zero and constant rows, determinism, the autograd plumbing
and the unchanged no-grad path, and the metrics built on the reduction against their float64 chains."""
import pytest
import torch

from oracle import aas_grad_oracle as G
from oracle import reduce_grad_oracle as R

pytestmark = pytest.mark.gpu

MODES = ("cosine", "mse", "minmax_cosine")
DTYPES = (torch.float16, torch.bfloat16, torch.float32)
TOL = {torch.float16: 3e-3, torch.bfloat16: 2e-2}   # the loose (exact-gradient) tier of test_gpu_grad.py


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return "cuda"


def _check(x, y, g, mode, dx, dy, record_property=None, name="", reference="autograd"):
    """Worst per-row relative error of (dx, dy) against float64 autograd (or the closed form), NaN rows matched."""
    ref = (R.autograd_grads if reference == "autograd" else R.pair_reduce_grads)(x, y, g, mode)
    floors = R.cross_term_norms(x, y, g, mode)
    worst = 0.0
    for got, r, fl in zip((dx, dy), ref, floors):
        if got is None:
            continue
        nan_rows = r.reshape(r.shape[0], -1).isnan().any(1)
        assert torch.equal(got.reshape(r.shape[0], -1).isnan().any(1), nan_rows), name
        assert not got.reshape(r.shape[0], -1)[~nan_rows].isnan().any(), name
        err = R.row_errors(got, r, fl)
        worst = max(worst, float(err.nan_to_num(0).max()))
    if record_property is not None:
        record_property(f"row_err_{name}", worst)
    print(f"{name}: worst per-row rel err {worst:.2e}")
    assert worst <= R.ROW_TOL, (name, worst)
    return worst


def _pair(P, E, dtype, dev, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(P, E, generator=g) * 0.7 + 0.2
    y = 0.6 * x + 0.4 * torch.randn(P, E, generator=g)
    d = torch.randn(P, generator=g)
    return x.to(dtype).to(dev), y.to(dtype).to(dev), d.to(dev)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("P,E", [(1, 655360), (5, 1000), (3, 8191), (16, 589824), (2, 7), (1, 1)])
def test_bwd_matches_float64_autograd(dtype, P, E, record_property):
    dev = _cuda()
    from diffsim_b200 import ops

    x, y, d = _pair(P, E, dtype, dev, seed=P * 1000 + E)
    for mode in MODES:
        if mode == "minmax_cosine" and E == 1:
            continue  # a one-element row is constant: NaN (test_zero_and_constant_rows)
        dx, dy = ops.pair_reduce_bwd(x, y, d, mode)
        assert dx.dtype == dy.dtype == torch.float32 and dx.shape == x.shape and dy.shape == y.shape
        _check(x, y, d, mode, dx, dy, record_property, f"{mode}_{str(dtype)[6:]}_{P}x{E}")


@pytest.mark.parametrize("dtype", DTYPES)
def test_unaligned_and_strided_rows(dtype, record_property):
    dev = _cuda()
    from diffsim_b200 import ops

    P, E = 3, 5000
    g = torch.Generator().manual_seed(11)
    buf = (torch.randn(P * (E + 3) + 1, generator=g)).to(dtype).to(dev)
    x = buf[1:1 + P * (E + 3)].view(P, E + 3)[:, :E]            # element-aligned only: the scalar path
    y = (torch.randn(P, E + 64, generator=g)).to(dtype).to(dev)[:, :E]   # 16-byte aligned rows, stride > E
    d = torch.randn(P, generator=g).to(dev)
    for mode in MODES:
        dx, dy = ops.pair_reduce_bwd(x, y, d, mode)
        _check(x, y, d, mode, dx, dy, record_property, f"strided_{mode}_{str(dtype)[6:]}")


@pytest.mark.parametrize("dtype", DTYPES)
def test_min_and_max_tied_many_times(dtype, record_property):
    dev = _cuda()
    from diffsim_b200 import ops

    g = torch.Generator().manual_seed(12)
    P, E = 4, 200003
    x = (torch.randn(P, E, generator=g) * 2).round().clamp(-3, 3)           # thousands of elements at each end
    y = (0.5 * x + torch.randn(P, E, generator=g)).round().clamp(-2, 4)
    x, y = x.to(dtype).to(dev), y.to(dtype).to(dev)
    d = torch.randn(P, generator=g).to(dev)
    assert ((x == x.amax(1, keepdim=True)).sum(1) > 100).all()
    dx, dy = ops.pair_reduce_bwd(x, y, d, "minmax_cosine")
    _check(x, y, d, "minmax_cosine", dx, dy, record_property, f"ties_{str(dtype)[6:]}")


def test_zero_and_constant_rows(record_property):
    dev = _cuda()
    from diffsim_b200 import ops

    g = torch.Generator().manual_seed(13)
    x = torch.randn(5, 3000, generator=g)
    y = torch.randn(5, 3000, generator=g)
    x[0], y[1], x[2], y[2] = 0, 0, 0, 0      # zero x, zero y, both zero
    x[3] = 0.25                              # constant x: the min-max score is NaN
    x, y = x.half().to(dev), y.half().to(dev)
    d = torch.randn(5, generator=g).to(dev)
    for mode in MODES:
        dx, dy = ops.pair_reduce_bwd(x, y, d, mode)
        _check(x, y, d, mode, dx, dy, record_property, f"zero_constant_{mode}")
    dx, dy = ops.pair_reduce_bwd(x, y, d, "minmax_cosine")
    assert dx[3].isnan().all() and dy[3].isnan().all() and not dx[4].isnan().any()   # NaN in its row only


def test_need_flags_and_repeated_calls_are_bitwise():
    dev = _cuda()
    from diffsim_b200 import ops

    x, y, d = _pair(8, 300000, torch.float16, dev, seed=3)
    for mode in MODES:
        full = ops.pair_reduce_bwd(x, y, d, mode)
        n0 = ops.LAUNCHES
        only_x = ops.pair_reduce_bwd(x, y, d, mode, need_y=False)
        assert ops.LAUNCHES - n0 == (1 if mode == "mse" else 2)
        only_y = ops.pair_reduce_bwd(x, y, d, mode, need_x=False)
        assert only_x[1] is None and only_y[0] is None
        assert torch.equal(only_x[0], full[0]) and torch.equal(only_y[1], full[1])
        assert ops.pair_reduce_bwd(x, y, d, mode, need_x=False, need_y=False) == (None, None)
        for _ in range(2):
            again = ops.pair_reduce_bwd(x, y, d, mode)
            assert torch.equal(again[0], full[0]) and torch.equal(again[1], full[1])


def test_autograd_forward_is_bitwise_and_issues_the_same_launches():
    dev = _cuda()
    from diffsim_b200 import ops

    x, y, d = _pair(6, 70000, torch.bfloat16, dev, seed=4)
    for mode in MODES:
        n0 = ops.LAUNCHES
        plain = ops.pair_reduce(x, y, mode)
        n1 = ops.LAUNCHES
        xl, yl = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
        out = ops.pair_reduce(xl, yl, mode)
        assert ops.LAUNCHES - n1 == n1 - n0 == 1
        assert out.grad_fn is not None and torch.equal(out.detach(), plain)
        out.backward(d)
        ref = ops.pair_reduce_bwd(x, y, d, mode)
        assert xl.grad.dtype == x.dtype   # the fp32 gradient cast to the input dtype by the engine
        assert torch.equal(xl.grad, ref[0].to(x.dtype)) and torch.equal(yl.grad, ref[1].to(y.dtype))
        # a frozen operand is not computed
        yl.grad = None
        n2 = ops.LAUNCHES
        ops.pair_reduce(x, yl, mode).backward(d)
        assert torch.equal(yl.grad, ref[1].to(y.dtype)) and ops.LAUNCHES - n2 == (2 if mode == "mse" else 3)


def test_torch_op_builds_no_graph():
    dev = _cuda()
    import diffsim_b200.torch_ops  # noqa: F401

    x, y, _ = _pair(2, 4096, torch.float16, dev, seed=5)
    out = torch.ops.diffsim_b200.pair_reduce(x.requires_grad_(), y, "cosine")
    assert out.grad_fn is None or "PairReduce" not in out.grad_fn.name(), out.grad_fn.name()
    assert out.grad_fn is None or all(f is None or "PairReduce" not in f.name() for f, _ in out.grad_fn.next_functions)


def test_full_size_fp16(record_property):
    dev = _cuda()
    from diffsim_b200 import ops

    P, E = 64, 655360
    x = torch.randn(P, E, device=dev).half()
    y = (0.5 * x.float() + torch.randn(P, E, device=dev)).half()
    d = torch.randn(P, device=dev)
    for mode in MODES:
        dx, dy = ops.pair_reduce_bwd(x, y, d, mode)
        _check(x, y, d, mode, dx, dy, record_property, f"full_{mode}", reference="closed_form")
        del dx, dy


# ---- metrics end to end, against the float64 chain with every rounding passed straight through ----------------------
def _st(t, dtype):
    return G._st_round(t, dtype)


def _rel(x, ref):
    return float((x.double() - ref.double()).norm() / ref.double().norm())


def test_clip_cross_score_gradients():
    dev = _cuda()
    from conftest import clip_images
    from diffsim_b200 import metrics

    (qa, ka, va), (qb, kb, vb), w, b = clip_images()
    H, S, D = qa.shape[1], qa.shape[2], qa.shape[3]
    scale, shape = D ** -0.5, (1, S, H * D)
    leaves = [t.to(dev).clone().requires_grad_(True) for t in (qa, ka, va, qb, kb, vb, w, b)]
    loss_scale = 1024.0
    score = metrics.clip_cross_score(tuple(leaves[0:3]), tuple(leaves[3:6]), scale, shape, leaves[6], leaves[7])
    with torch.no_grad():
        plain = metrics.clip_cross_score((qa.to(dev), ka.to(dev), va.to(dev)), (qb.to(dev), kb.to(dev), vb.to(dev)),
                                         scale, shape, w.to(dev), b.to(dev))
    assert torch.equal(score.detach(), plain)
    (score.float().sum() * loss_scale).backward()

    f = G._leaves(*leaves)
    dt = torch.float16

    def calc(q, k, v):
        o = G.attention(q, k, v, scale, dt).transpose(1, 2).reshape(1, S, H * D)
        return _st(o @ f[6].t() + f[7], dt)

    x = torch.stack([calc(f[0], f[4], f[5]).reshape(-1), calc(f[3], f[1], f[2]).reshape(-1)])
    y = torch.stack([calc(f[0], f[1], f[2]).reshape(-1), calc(f[3], f[4], f[5]).reshape(-1)])
    dd = _st(torch.nn.functional.cosine_similarity(x, y, dim=1), dt)
    ref = torch.autograd.grad(_st((dd[0:1] + dd[1:2]) / 2, dt).sum() * loss_scale, f)
    errs = [_rel(l.grad, r) for l, r in zip(leaves, ref)]
    print("clip_cross grads rel err (qa ka va qb kb vb W b):", " ".join(f"{e:.1e}" for e in errs))
    assert max(errs) <= TOL[dt], errs


def test_gram_diffeats_and_embedding_gradients():
    dev = _cuda()
    from conftest import diffeats_features, gram_features
    from diffsim_b200 import metrics

    dt = torch.float16
    errs = {}
    # gram: the fp16 Gram through K4 (rounded), the cosine of the last rows through K2, rounded to fp16
    fa, fb = (t.to(dev).clone().requires_grad_(True) for t in gram_features())
    (metrics.gram_similarity(fa, fb).float().sum() * 1024.0).backward()
    a64, b64 = G._leaves(fa, fb)
    ga = _st(a64.reshape(64, -1) @ a64.reshape(64, -1).t(), dt)
    gb = _st(b64.reshape(64, -1) @ b64.reshape(64, -1).t(), dt)
    s = _st(torch.nn.functional.cosine_similarity(ga[-1:], gb[-1:]), dt)
    ra, rb = torch.autograd.grad(s.sum() * 1024.0, (a64, b64))
    errs["gram"] = (_rel(fa.grad, ra), _rel(fb.grad, rb))
    # diffeats: min-max normalised flat cosine of (2, 256, 320) maps (loss scaled: per-element gradients ~ 1/E; the
    # scale also reaches the fp16 score's gradient, so it stays below fp16's largest value)
    fa, fb = (t.to(dev).clone().requires_grad_(True) for t in diffeats_features())
    (metrics.diffeats_score(fa, fb).float().sum() * 4096.0).backward()
    a64, b64 = G._leaves(fa, fb)
    s = _st(R.reference_score(a64, b64, "minmax_cosine"), dt)
    ra, rb = torch.autograd.grad(s * 4096.0, (a64, b64))
    errs["diffeats"] = (_rel(fa.grad, ra), _rel(fb.grad, rb))
    # embedding: 100 * row-wise cosine summed over the batch
    g = torch.Generator().manual_seed(9)
    ex = torch.randn(8, 768, generator=g).half().to(dev).requires_grad_(True)
    ey = (0.5 * ex.detach().float() + torch.randn(8, 768, generator=g).to(dev)).half().requires_grad_(True)
    score, n = metrics.embedding_score(ex, ey)
    assert n == 8
    score.backward()
    x64, y64 = G._leaves(ex, ey)
    ra, rb = torch.autograd.grad(100.0 * torch.nn.functional.cosine_similarity(x64, y64, dim=1).sum(), (x64, y64))
    errs["embedding"] = (_rel(ex.grad, ra), _rel(ey.grad, rb))
    print({k: f"{v[0]:.1e} {v[1]:.1e}" for k, v in errs.items()})
    for k, v in errs.items():
        assert max(v) <= TOL[dt], (k, v)
