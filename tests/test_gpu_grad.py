"""K5 backward on the GPU: fp32 gradients of the attention and of the Aligned Attention Score against the float64
oracle (evaluated on the device), determinism, the autograd plumbing and the unchanged no-grad path."""
import pytest
import torch

from oracle import aas_grad_oracle as G

pytestmark = pytest.mark.gpu

TOL = {torch.float16: 3e-3, torch.bfloat16: 2e-2}


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return "cuda"


def _rel(x, ref):
    return float((x.double() - ref).norm() / ref.norm())


def _sd(B, H, S, D, dtype, dev, g, scale=1.0):
    # the reference's head-split view of (B, S, H*D) memory
    return (scale * torch.randn(B, S, H, D, generator=g, device=dev)).to(dtype).permute(0, 2, 1, 3)


ATTN_CASES = [
    # (B, H, Sq, Skv, D, dtype, layout)
    (2, 8, 256, 256, 160, torch.float16, "sd"),
    (2, 8, 256, 256, 160, torch.bfloat16, "sd"),
    (2, 8, 1024, 1024, 80, torch.float16, "sd"),
    (2, 20, 1024, 1024, 64, torch.float16, "sd"),
    (2, 20, 1024, 1024, 64, torch.bfloat16, "sd"),
    (2, 10, 4096, 4096, 64, torch.float16, "sd"),
    (2, 16, 256, 256, 72, torch.float16, "dit"),
    (1, 4, 256, 4, 128, torch.float16, "sd"),
    (1, 4, 256, 16, 40, torch.float16, "sd"),
    (1, 4, 200, 50, 80, torch.bfloat16, "sd"),
    (1, 4, 384, 257, 160, torch.float16, "sd"),
    (2, 3, 130, 700, 64, torch.float16, "sd"),
]


def _attn_inputs(B, H, Sq, Skv, D, dtype, layout, dev, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    if layout == "dit":
        assert Sq == Skv
        qkv = torch.randn(B, Sq, 3, H, D, generator=g, device=dev).to(dtype)   # DiT's packed qkv (in place)
        q, k, v = (qkv[:, :, i].permute(0, 2, 1, 3) for i in range(3))
    else:
        q, k, v = _sd(B, H, Sq, D, dtype, dev, g), _sd(B, H, Skv, D, dtype, dev, g), _sd(B, H, Skv, D, dtype, dev, g)
    dout = torch.randn(B, H, Sq, D, generator=g, device=dev).to(dtype)
    return q, k, v, dout


@pytest.mark.parametrize("B,H,Sq,Skv,D,dtype,layout", ATTN_CASES)
def test_attn_bwd_matches_float64_oracle(B, H, Sq, Skv, D, dtype, layout, record_property):
    dev = _cuda()
    from diffsim_b200 import ops

    q, k, v, dout = _attn_inputs(B, H, Sq, Skv, D, dtype, layout, dev)
    scale = 0.1 if D == 40 else None   # one explicit scale
    out = ops.attn_fwd(q, k, v, scale)
    got = ops.attn_bwd(q, k, v, out, dout, scale)
    ref = G.attn_grads(q, k, v, dout, scale)
    errs = [_rel(a, b) for a, b in zip(got, ref)]
    record_property("rel_err_dq_dk_dv", errs)
    print(f"attn_bwd {(B, H, Sq, Skv, D)} {dtype} {layout}: rel err dq {errs[0]:.2e} dk {errs[1]:.2e} dv {errs[2]:.2e}")
    assert all(t.dtype == torch.float32 for t in got)
    assert max(errs) <= TOL[dtype], errs


def _pair(shape, dtype, dev, alpha, seed=5):
    from diffsim_b200 import synth

    m = synth.SynthModel(*shape, seed=2334)
    g = torch.Generator().manual_seed(seed)
    base = m.new_base(g)
    return [tuple(t.to(dev) for t in m.image(base, a, dtype, "sd", g)) for a in (1.0, alpha)]


@pytest.mark.parametrize("mode", ["cosine", "mse"])
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_aas_score_grads_match_float64_oracle(mode, dtype):
    dev = _cuda()
    from diffsim_b200 import ops

    A, B = _pair((2, 8, 256, 160), dtype, dev, 0.6)
    g = torch.full((1,), 0.5, device=dev)   # score = (dir_ab + dir_ba) / 2
    got = ops.pair_dirs_bwd(*A, *B, g, g, mode)
    ref = G.pair_score_grads(*A, *B, mode)
    errs = [_rel(a, b) for a, b in zip(got, ref)]
    print(f"aas_score grads {mode} {dtype}: rel err " + " ".join(f"{e:.2e}" for e in errs))
    assert max(errs) <= TOL[dtype], errs


def test_self_pair_gradients_are_finite_and_near_zero():
    dev = _cuda()
    from diffsim_b200 import ops

    A, B = _pair((2, 8, 256, 160), torch.float16, dev, 0.6)
    g = torch.full((1,), 0.5, device=dev)
    same = ops.pair_dirs_bwd(*A, *A, g, g, "cosine")
    real = ops.pair_dirs_bwd(*A, *B, g, g, "cosine")
    for s, r in zip(same, real):
        assert torch.isfinite(s).all()
        assert float(s.norm()) <= 1e-3 * float(r.norm())


def test_ip_adapter_gradients_16_tokens():
    dev = _cuda()
    from diffsim_b200.diffsim import aas_score_ip_adapter
    from conftest import ip_images

    (qa, ka_l, va_l), (qb, kb_l, vb_l) = ip_images(11, 16, 2, 0.6)
    leaves = [t.to(dev).requires_grad_(True) for t in [qa, *ka_l, *va_l, qb, *kb_l, *vb_l]]
    qa_, ka_, va_ = leaves[0], leaves[1:3], leaves[3:5]
    qb_, kb_, vb_ = leaves[5], leaves[6:8], leaves[8:10]
    s = aas_score_ip_adapter((qa_, ka_, va_), (qb_, kb_, vb_), match_reference_dtype=False)
    (s * 1e4).backward()   # keeps the fp16 gradients in the normal range
    ref = [torch.zeros(t.shape, dtype=torch.float64, device=dev) for t in leaves]
    for i in range(2):
        gi = G.pair_score_grads(qa_, ka_[i], va_[i], qb_, kb_[i], vb_[i], "cosine", g=1e4 / 2)
        for dst, src in zip((0, 1 + i, 3 + i, 5, 6 + i, 8 + i), gi):
            ref[dst] += src
    errs = [_rel(t.grad, r) for t, r in zip(leaves, ref)]
    print("ip-adapter grads: rel err " + " ".join(f"{e:.2e}" for e in errs))
    assert max(errs) <= 5e-3, errs   # fp32 gradients cast to fp16 once more


def test_autograd_grad_is_the_fp32_result_cast_and_deterministic():
    dev = _cuda()
    from diffsim_b200 import ops
    from diffsim_b200.diffsim import aas_score

    A, B = _pair((2, 8, 256, 160), torch.float16, dev, 0.7)
    leaves = [t.clone().requires_grad_(True) for t in (*A, *B)]
    s = aas_score(tuple(leaves[:3]), tuple(leaves[3:]), match_reference_dtype=False)
    (s.sum() * 1e4).backward()
    g = torch.full((1,), 5e3, device=dev)
    f32 = ops.pair_dirs_bwd(*A, *B, g, g, "cosine")
    for t, r in zip(leaves, f32):
        assert torch.equal(t.grad, r.to(torch.float16))
    again = ops.pair_dirs_bwd(*A, *B, g, g, "cosine")
    assert all(torch.equal(a, b) for a, b in zip(f32, again))

    q, k, v, dout = _attn_inputs(2, 8, 256, 256, 160, torch.float16, "sd", dev)
    ql, kl, vl = (t.detach().requires_grad_(True) for t in (q, k, v))
    ops.attn_fwd(ql, kl, vl).backward(dout)
    out = ops.attn_fwd(q, k, v)
    r1 = ops.attn_bwd(q, k, v, out, dout)
    r2 = ops.attn_bwd(q, k, v, out, dout)
    assert all(torch.equal(a, b) for a, b in zip(r1, r2))
    for t, r in zip((ql, kl, vl), r1):
        assert torch.equal(t.grad, r.to(torch.float16))


def test_torch_ops_autograd():
    dev = _cuda()
    import diffsim_b200.torch_ops  # noqa: F401
    from diffsim_b200 import ops

    q, k, v, dout = _attn_inputs(2, 8, 256, 256, 64, torch.float16, "sd", dev)
    ql, kl, vl = (t.detach().requires_grad_(True) for t in (q, k, v))
    torch.ops.diffsim_b200.attn_fwd(ql, kl, vl).backward(dout)
    ref = ops.attn_bwd(q, k, v, ops.attn_fwd(q, k, v), dout)
    for t, r in zip((ql, kl, vl), ref):
        assert torch.equal(t.grad, r.to(torch.float16))

    A, B = _pair((2, 8, 256, 160), torch.float16, dev, 0.6)
    leaves = [t.clone().requires_grad_(True) for t in (*A, *B)]
    (torch.ops.diffsim_b200.aas_score(*leaves, "mse").sum() * 1e4).backward()
    g = torch.full((1,), 5e3, device=dev)
    f32 = ops.pair_dirs_bwd(*A, *B, g, g, "mse")
    for t, r in zip(leaves, f32):
        assert torch.equal(t.grad, r.to(torch.float16))


def test_no_grad_path_is_unchanged():
    dev = _cuda()
    from diffsim_b200 import ops
    from diffsim_b200.diffsim import aas_score

    A, B = _pair((2, 8, 256, 160), torch.float16, dev, 0.6)
    for mode in ("cosine", "mse"):
        n0 = ops.LAUNCHES
        plain = aas_score(A, B, mode)
        assert ops.LAUNCHES - n0 == 6   # two directions x (index validation + attention + finish)
        leaves = [t.clone().requires_grad_(True) for t in (*A, *B)]
        n0 = ops.LAUNCHES
        graded = aas_score(tuple(leaves[:3]), tuple(leaves[3:]), mode)
        assert ops.LAUNCHES - n0 == 6
        assert graded.requires_grad and torch.equal(plain, graded.detach())
        with torch.no_grad():
            assert not aas_score(tuple(leaves[:3]), tuple(leaves[3:]), mode).requires_grad
    q, k, v, _ = _attn_inputs(1, 2, 256, 256, 64, torch.float16, "sd", dev)
    n0 = ops.LAUNCHES
    o = ops.attn_fwd(q, k, v)
    assert ops.LAUNCHES - n0 == 2 and not o.requires_grad
    ql = q.detach().requires_grad_(True)
    o2 = ops.attn_fwd(ql, k, v)
    assert o2.requires_grad and torch.equal(o, o2.detach())
    with pytest.raises(RuntimeError, match="out="):
        ops.attn_fwd(ql, k, v, out=torch.empty_like(o))
