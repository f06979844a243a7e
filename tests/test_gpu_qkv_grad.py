"""K4 backward on the GPU: ds_qkv_project_bwd against the float64 oracle, both GEMM kernels bitwise, and the gradient
reaching the hook input and the projection weights through the capture hooks and B200AttnProcessor."""
import pytest
import torch

from oracle import qkv_grad_oracle as QG

pytestmark = pytest.mark.gpu

TOL = {torch.float16: 3e-3, torch.bfloat16: 2e-2}   # the loose (exact-gradient) tier of test_gpu_grad.py
# absolute term of the tolerance, in units of eps(dtype) x the float64 sum of |products|: the fp32 accumulation error
# (split partials added in order) measured in 16-bit ulps.  Worst seen over the cases below on a B200: 7.9e-5 (fp16, dX)
# and 8.8e-6 (bf16, dX); each constant is under 4x that.
ABS_SUM_K = {torch.float16: 3e-4, torch.bfloat16: 3.5e-5}


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return "cuda"


def _close(got, ref64, bound64, dtype, name, record_property):
    """got (16-bit) is the float64 value rounded to dtype, give or take one ulp, plus ABS_SUM_K * eps * sum |products|
    for the fp32 accumulation; fp16 results in the subnormal range are allowed one subnormal step."""
    eps = torch.finfo(dtype).eps
    sub = 2.0 ** -24 if dtype == torch.float16 else 0.0
    err = (got.double() - ref64).abs()
    over = (err - eps * ref64.abs() - sub).clamp_min(0)
    ratio = (over / (eps * bound64).clamp_min(1e-300)).max().item()
    record_property(f"abs_sum_ratio_{name}", ratio)
    assert ratio <= ABS_SUM_K[dtype], \
        f"{name}: error {ratio:.3e} x eps x sum|products| beyond one ulp (allowed {ABS_SUM_K[dtype]:.3e})"
    assert torch.isfinite(got).all()


def _inputs(rows, c_in, n_out, n_t, dtype, dev, seed, dy_scale=1.0, bias=False):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(rows, c_in, generator=g).to(dtype).to(dev)
    w = (torch.randn(n_out, c_in, generator=g) / c_in ** 0.5).to(dtype).to(dev)
    dys = [(torch.randn(rows, n_out // n_t, generator=g) * dy_scale).to(dtype).to(dev) for _ in range(n_t)]
    return x, w, dys


CASES = {
    # name: rows, c_in, n_out, n_outputs, dy scale
    "sd_c320_rows8192": (8192, 320, 960, 3, 1.0),
    "sd_c640_rows1000": (1000, 640, 1920, 3, 1.0),
    "sd_c1280_rows568": (568, 1280, 3840, 3, 1.0),
    "dit_c1152_packed_rows456": (456, 1152, 3456, 1, 1.0),
    "cols1000_rows300": (300, 1000, 3000, 3, 1.0),
    "sd_c320_dy_1e-6": (2048, 320, 960, 3, 1e-6),
}


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("case", list(CASES))
def test_bwd_matches_float64_oracle(case, dtype, record_property):
    dev = _cuda()
    from diffsim_b200 import ops

    rows, c_in, n_out, n_t, scale = CASES[case]
    x, w, dys = _inputs(rows, c_in, n_out, n_t, dtype, dev, seed=rows + c_in, dy_scale=scale)
    dx, dw, db = ops.qkv_project_bwd(x, w, dys, True, True, True)
    (rx, rw, rb), (bx, bw, bb) = QG.qkv_bwd(x, w, dys)
    assert dx.dtype == dw.dtype == db.dtype == dtype
    assert dx.shape == x.shape and dw.shape == w.shape and db.shape == (n_out,)
    _close(dx, rx, bx, dtype, "dx", record_property)
    _close(dw, rw, bw, dtype, "dw", record_property)
    _close(db, rb, bb, dtype, "db", record_property)
    if scale < 1e-3 and dtype == torch.float16:
        assert (dys[0].abs() < torch.finfo(dtype).tiny).any()   # the case does reach fp16's subnormal range


def test_unwanted_gradients_are_not_computed_and_strided_dy_is_read_in_place():
    dev = _cuda()
    from diffsim_b200 import ops

    x, w, _ = _inputs(384, 320, 960, 3, torch.float16, dev, seed=1)
    big = torch.randn(384, 3 * 320 + 64, device=dev).half()          # dy tensors with a row stride > their width
    dys = [big[:, i * 320:(i + 1) * 320] for i in range(3)]
    n0 = ops.LAUNCHES
    dx, dw, db = ops.qkv_project_bwd(x, w, dys, True, False, False)
    assert ops.LAUNCHES - n0 == 2 and dw is None and db is None
    full = ops.qkv_project_bwd(x, w, [d.contiguous() for d in dys], True, True, True)
    assert torch.equal(dx, full[0])


@pytest.mark.parametrize("case", ["sd_c320_rows8192", "sd_c1280_rows568", "dit_c1152_packed_rows456", "cols1000_rows300"])
def test_single_cta_and_pair_kernels_are_bitwise_equal_and_calls_repeat(case):
    dev = _cuda()
    from diffsim_b200 import _native as N, ops

    rows, c_in, n_out, n_t, scale = CASES[case]
    x, w, dys = _inputs(rows, c_in, n_out, n_t, torch.bfloat16, dev, seed=7, dy_scale=scale)
    lib = N.load()
    try:
        res = {}
        for variant in (0, 2, -1):
            assert lib.ds_debug_set_gemm_variant(variant) == variant
            res[variant] = [ops.qkv_project_bwd(x, w, dys, True, True, True) for _ in range(2)]
    finally:
        lib.ds_debug_set_gemm_variant(-1)
    ref = res[0][0]
    for variant, calls in res.items():
        for call in calls:
            for a, b in zip(call, ref):
                assert torch.equal(a, b), f"variant {variant}"


class _Attention(torch.nn.Module):
    """The attributes of a diffusers Attention block that the capture path reads."""

    def __init__(self, dim, heads, dtype, dev, bias=False):
        super().__init__()
        self.heads = heads
        self.to_q = torch.nn.Linear(dim, dim, bias=bias, dtype=dtype, device=dev)
        self.to_k = torch.nn.Linear(dim, dim, bias=bias, dtype=dtype, device=dev)
        self.to_v = torch.nn.Linear(dim, dim, bias=bias, dtype=dtype, device=dev)
        self.to_out = torch.nn.ModuleList([torch.nn.Linear(dim, dim, dtype=dtype, device=dev), torch.nn.Dropout(0.0)])
        self.spatial_norm = self.group_norm = None
        self.norm_cross = False
        self.residual_connection = False
        self.rescale_output_factor = 1.0
        self.processor = None

    def forward(self, hidden_states):
        return self.processor(self, hidden_states)[0] if self.processor else hidden_states


def _rel(x, ref):
    assert ref.double().norm() > 0
    return ((x.double() - ref.double()).norm() / ref.double().norm()).item()


def _grouped(grads, n_w, bias):
    # the three bias gradients are compared as one vector: the k bias has an exact gradient of zero (a shift of every key
    # by one vector moves each logit row by a constant, which the softmax ignores), so only rounding noise is left of it
    return grads[:2 + n_w] + ([torch.cat([g.reshape(-1).double() for g in grads[2 + n_w:]])] if bias else [])


def _capture_score(attn, xa, xb, fused=True, g=1024.0):
    from diffsim_b200 import hooks
    from diffsim_b200.diffsim import aas_score

    caps = []
    for x in (xa, xb):
        with hooks.capture(attn, hooks.make_sd_pre_hook(fused_qkv=fused)):
            attn(x)
        caps.append(tuple(attn.stores))
    s = aas_score(caps[0], caps[1], "cosine")
    return s, (s.float().sum() * g)


@pytest.mark.parametrize("bias", [False, True])
def test_capture_hook_gradient_reaches_hidden_and_weights(bias):
    dev = _cuda()
    from diffsim_b200 import ops

    dtype, C, heads, S = torch.float16, 320, 8, 256
    torch.manual_seed(0)
    attn = _Attention(C, heads, dtype, dev, bias=bias)
    base_a = torch.randn(1, S, C, device=dev, dtype=dtype)
    base_b = (0.6 * base_a + 0.8 * torch.randn(1, S, C, device=dev, dtype=dtype)).to(dtype)
    lins = (attn.to_q, attn.to_k, attn.to_v)
    params = [m.weight for m in lins] + ([m.bias for m in lins] if bias else [])

    def run(fused):
        xa, xb = base_a.clone().requires_grad_(True), base_b.clone().requires_grad_(True)
        for p in params:
            p.grad = None
        s, loss = _capture_score(attn, xa, xb, fused)
        loss.backward()
        return s, [xa.grad, xb.grad] + [p.grad for p in params]

    plain, _ = _capture_score(attn, base_a, base_b)
    with torch.no_grad():
        nograd, _ = _capture_score(attn, base_a, base_b)
    s, grads = run(True)
    assert all(gr is not None for gr in grads)
    assert torch.equal(s.detach(), plain.detach()) and torch.equal(s.detach(), nograd)   # bitwise, with and without grad
    ref = QG.capture_chain_grads(base_a, base_b, [m.weight for m in lins], heads, "cosine", 1024.0,
                                 [m.bias for m in lins] if bias else None)
    for got, r in zip(_grouped(grads, 3, bias), _grouped(list(ref), 3, bias)):
        assert _rel(got, r) < TOL[dtype]
    _, unfused = run(False)
    for got, r in zip(_grouped(grads, 3, bias), _grouped(unfused, 3, bias)):
        assert _rel(got, r) < TOL[dtype]
    # frozen projection weights (DiffSim as a loss on a frozen UNet): the backward runs dX only, no dW GEMM
    counts = {}
    for frozen in (False, True):
        for p in params:
            p.requires_grad_(not frozen)
        xa, xb = base_a.clone().requires_grad_(True), base_b.clone().requires_grad_(True)
        _, loss = _capture_score(attn, xa, xb)
        n0 = ops.LAUNCHES
        loss.backward()
        counts[frozen] = ops.LAUNCHES - n0
        assert xa.grad is not None
    for p in params:
        p.requires_grad_(True)
    assert counts[False] - counts[True] == 2 * (2 + (2 if bias else 0))   # per capture: dW GEMM + finish (+ dbias pair)


def test_capture_into_a_cache_slot_stays_forward_only():
    dev = _cuda()
    from diffsim_b200 import hooks, scoring

    attn = _Attention(320, 8, torch.float16, dev)
    x = torch.randn(1, 256, 320, device=dev, dtype=torch.float16, requires_grad=True)
    cache = scoring.QKVCache.empty(2, 1, 8, 256, 40, torch.float16, dev)
    with hooks.capture(attn, hooks.make_sd_pre_hook(out=[m[0] for m in cache.memory()])):
        attn(x)
    assert not attn.stores[0].requires_grad and attn.stores[0].data_ptr() == cache.q[0].data_ptr()


def test_training_step_through_the_processor_matches_the_unfused_one():
    dev = _cuda()
    from diffsim_b200 import hooks

    dtype = torch.float16
    torch.manual_seed(1)
    attn = _Attention(640, 8, dtype, dev, bias=True)
    x = torch.randn(2, 256, 640, device=dev, dtype=dtype)
    lins = (attn.to_q, attn.to_k, attn.to_v)
    grads = {}
    for fused in (True, False):
        attn.processor = hooks.B200AttnProcessor(fused_qkv=fused)
        attn.zero_grad(set_to_none=True)
        xl = x.clone().requires_grad_(True)
        out = attn(xl)
        out.float().pow(2).sum().backward()
        grads[fused] = [xl.grad] + [m.weight.grad for m in lins] + [m.bias.grad for m in lins]
        assert all(g is not None for g in grads[fused])
    for a, b in zip(grads[True][:4], grads[False][:4]):
        assert _rel(a, b) < TOL[dtype]
    assert _rel(torch.cat(grads[True][4:]), torch.cat(grads[False][4:])) < TOL[dtype]


class _DiTAttention(torch.nn.Module):
    """timm-style Attention: qkv, num_heads, head_dim, q_norm, k_norm."""

    def __init__(self, dim, heads, dtype, dev):
        super().__init__()
        self.num_heads, self.head_dim = heads, dim // heads
        self.qkv = torch.nn.Linear(dim, 3 * dim, bias=True, dtype=dtype, device=dev)
        self.q_norm = self.k_norm = torch.nn.Identity()

    def forward(self, x):
        return x


def test_dit_hook_gives_qkv_weight_and_bias_gradients():
    dev = _cuda()
    from diffsim_b200 import hooks
    from diffsim_b200.diffsim import aas_score

    dtype = torch.bfloat16
    torch.manual_seed(2)
    blk = _DiTAttention(1152, 16, dtype, dev)
    xa = torch.randn(1, 256, 1152, device=dev, dtype=dtype)
    xb = torch.randn(1, 256, 1152, device=dev, dtype=dtype)
    grads = {}
    for fused in (True, False):
        blk.zero_grad(set_to_none=True)
        caps = []
        for x in (xa, xb):
            with hooks.capture(blk, hooks.make_dit_pre_hook(fused_qkv=fused)):
                blk(x)
            caps.append(tuple(blk.stores))
        (aas_score(caps[0], caps[1], "cosine").float().sum() * 1024).backward()
        grads[fused] = (blk.qkv.weight.grad, blk.qkv.bias.grad)
        assert all(g is not None for g in grads[fused])
    for a, b in zip(grads[True], grads[False]):
        assert _rel(a, b) < TOL[dtype]
