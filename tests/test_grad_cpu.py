"""K5 backward without a GPU: the float64 gradient oracle, the autograd registration of the differentiable operators,
argument validation of the backward ABI and its loud failure without a device."""
import ctypes as C

import pytest
import torch

from diffsim_b200 import _native as N
from oracle import aas_grad_oracle as G
from oracle import aas_oracle as O


def _qkv(B, H, S, D, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(B, H, S, D, generator=g, dtype=torch.float64) for _ in range(3)]


def test_oracle_attention_gradient_passes_gradcheck():
    q, k, v = [t.requires_grad_(True) for t in _qkv(1, 2, 5, 4, 0)]
    assert torch.autograd.gradcheck(lambda a, b, c: G.attention(a, b, c, 0.7), (q, k, v))
    dout = torch.randn(1, 2, 5, 4, dtype=torch.float64)
    dq, dk, dv = G.attn_grads(q, k, v, dout, 0.7)
    o = G.attention(q, k, v, 0.7)
    ref = torch.autograd.grad((o * dout).sum(), (q, k, v))
    assert all(torch.allclose(a, b) for a, b in zip((dq, dk, dv), ref))


@pytest.mark.parametrize("mode", ["cosine", "mse"])
def test_oracle_directional_gradient_passes_gradcheck(mode):
    ts = [t.requires_grad_(True) for t in _qkv(1, 2, 6, 4, 1) + _qkv(1, 2, 6, 4, 2)[1:]]
    assert torch.autograd.gradcheck(lambda *a: G.dir_value(*a, mode=mode), ts)


def test_oracle_value_is_the_t1_score():
    a = [t.half() for t in _qkv(1, 2, 8, 16, 3)]
    b = [t.half() for t in _qkv(1, 2, 8, 16, 4)]
    for mode in ("cosine", "mse"):
        rnd = torch.float16
        v = (G.dir_value(*[t.double() for t in a], b[1].double(), b[2].double(), mode, None, rnd)
             + G.dir_value(*[t.double() for t in b], a[1].double(), a[2].double(), mode, None, rnd)) / 2
        assert float(v) == pytest.approx(O.aas_pair_score(*a, *b, mode), rel=1e-12)
    grads = G.pair_score_grads(*a, *b, "cosine")
    assert len(grads) == 6 and all(g.dtype == torch.float64 and torch.isfinite(g).all() for g in grads)


def test_straight_through_rounding_has_identity_gradient():
    x = torch.randn(10, dtype=torch.float64, requires_grad=True)
    y = G._st_round(x, torch.float16)
    assert torch.equal(y.detach(), x.detach().half().double())
    (gx,) = torch.autograd.grad(y.sum(), x)
    assert torch.equal(gx, torch.ones_like(gx))


def test_autograd_is_registered_on_the_differentiable_ops():
    from diffsim_b200 import torch_ops

    assert torch_ops.DIFFERENTIABLE == ("attn_fwd", "aas_score")
    for name in torch_ops.DIFFERENTIABLE:
        op = getattr(torch.ops.diffsim_b200, name).default
        assert torch._C._dispatch_has_kernel_for_dispatch_key(op.name(), "Autograd")
    # still no CPU kernel behind them
    x = torch.randn(1, 1, 4, 64, dtype=torch.float16, requires_grad=True)
    with pytest.raises(NotImplementedError):
        torch.ops.diffsim_b200.attn_fwd(x, x, x)


def _t4(shape, dtype, ptr=16, strides=None):
    t = N.Tensor4()
    t.ptr = ptr
    t.size[:] = list(shape)
    if strides is None:
        strides = [shape[1] * shape[2] * shape[3], shape[2] * shape[3], shape[3], 1]
    t.stride[:] = strides
    t.dtype = dtype
    return t


def test_backward_abi_validates_before_touching_the_device():
    lib = N.load()
    s = (1, 2, 128, 64)
    h, f = _t4(s, N.DS_F16), _t4(s, N.DS_F32)
    ws = (C.c_uint8 * 4096)()
    assert lib.ds_attn_bwd_workspace_bytes(h, h) >= 2 * 2 * 128 * 4
    assert lib.ds_aas_dir_bwd_workspace_bytes(h, h) >= 4 * 2 * 128 * 64 * 2

    def attn(q=h, out=h, dq=f, dk=f):
        return lib.ds_attn_bwd(q, h, h, out, h, 0.0, dq, dk, f, ws, 4096, None)

    assert attn(q=_t4(s, N.DS_F16, ptr=0)) == N.DS_ERR_INVALID and "null" in N.last_error()
    assert attn(dq=_t4(s, N.DS_F16)) == N.DS_ERR_INVALID and "float32" in N.last_error()
    assert attn(dk=_t4((1, 2, 64, 64), N.DS_F32)) == N.DS_ERR_INVALID
    assert attn(out=_t4(s, N.DS_BF16)) == N.DS_ERR_INVALID
    assert attn(q=_t4(s, N.DS_F16, ptr=24)) == N.DS_ERR_INVALID and "aligned" in N.last_error()
    assert attn(q=_t4(s, N.DS_F16, strides=[16384, 8192, 60, 1])) == N.DS_ERR_INVALID
    d96 = _t4((1, 2, 128, 96), N.DS_F16)
    assert lib.ds_attn_bwd(d96, d96, d96, d96, d96, 0.0, _t4((1, 2, 128, 96), N.DS_F32), _t4((1, 2, 128, 96), N.DS_F32),
                           _t4((1, 2, 128, 96), N.DS_F32), ws, 4096, None) == N.DS_ERR_UNSUPPORTED
    assert lib.ds_attn_bwd(h, h, h, h, h, 0.0, f, f, f, ws, 8, None) == N.DS_ERR_WORKSPACE
    g = (C.c_float * 1)()

    def dirb(mode=N.DS_SIM_COSINE, d_dir=g, dkj=f):
        return lib.ds_aas_dir_bwd(h, h, h, h, h, 0.0, mode, d_dir, f, f, f, dkj, f, ws, 4096, None)

    assert dirb(mode=N.DS_SIM_MINMAX_COSINE) == N.DS_ERR_INVALID and "mode" in N.last_error()
    assert dirb(d_dir=None) == N.DS_ERR_INVALID and "d_dir" in N.last_error()
    assert dirb(dkj=_t4(s, N.DS_BF16)) == N.DS_ERR_INVALID
    assert dirb() == N.DS_ERR_WORKSPACE


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour on a machine without a GPU")
def test_backward_without_gpu_fails_loudly():
    lib = N.load()
    s = (1, 2, 128, 64)
    x = torch.zeros(s, dtype=torch.float16)
    g32 = torch.zeros(s, dtype=torch.float32)
    h = _t4(s, N.DS_F16, ptr=x.data_ptr())
    f = _t4(s, N.DS_F32, ptr=g32.data_ptr())
    ws = torch.zeros(1 << 22, dtype=torch.uint8)
    assert lib.ds_attn_bwd(h, h, h, h, h, 0.0, f, f, f, ws.data_ptr(), ws.numel(), None) == N.DS_ERR_CUDA
    d = torch.ones(1)
    assert lib.ds_aas_dir_bwd(h, h, h, h, h, 0.0, N.DS_SIM_COSINE, d.data_ptr(), f, f, f, f, f, ws.data_ptr(),
                              ws.numel(), None) == N.DS_ERR_CUDA
    assert g32.abs().sum().item() == 0.0   # nothing was computed on the host
    from diffsim_b200 import ops

    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.attn_bwd(x, x, x, x, x)
    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.aas_dir_bwd(x, x, x, x, x, d)
    xr = x.clone().requires_grad_(True)
    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.attn_fwd(xr, x, x)
