"""Matrix K5 backward without a GPU: argument checks of ds_aas_matrix_bwd before the device is touched, the workspace
query, the loud failure without a device, and the float64 fold model against autograd."""
import ctypes as C
import math

import pytest
import torch

from diffsim_b200 import _native as N
from oracle import aas_grad_oracle as G
from oracle import aas_matrix_grad_oracle as M


def _desc(shape, dtype, ptr=256, strides=None):
    t = N.Tensor5()
    t.ptr = ptr
    t.size[:] = list(shape)
    t.stride[:] = strides if strides is not None else [math.prod(shape[i + 1:]) for i in range(5)]
    t.dtype = dtype
    return t


ROWS, COLS = (3, 1, 2, 128, 64), (5, 1, 2, 128, 64)


def test_workspace_query_grows_with_rows_and_columns():
    lib = N.load()
    img = math.prod(ROWS[1:]) * 2
    ws = lambda r, c: lib.ds_aas_matrix_bwd_workspace_bytes(_desc((r,) + ROWS[1:], N.DS_F16),  # noqa: E731
                                                             _desc((c,) + ROWS[1:], N.DS_F16))
    assert ws(1, 1) >= 6 * img   # Y, X, fx, F_r in 16 bits and fp32
    assert ws(1, 9) - ws(1, 1) >= 8 * 2 * img   # X and fx per entry
    assert ws(9, 1) - ws(1, 1) >= 8 * 6 * img   # an entry and a row per row
    assert ws(4, 4) > ws(3, 4) > ws(3, 3)
    assert ws(0, 3) == 256


def test_matrix_bwd_validates_before_touching_the_device():
    lib = N.load()
    q, kc = _desc(ROWS, N.DS_F16), _desc(COLS, N.DS_F16)
    base = 1 << 24
    gr = [_desc(ROWS, N.DS_F32, ptr=base + i * (1 << 22)) for i in range(3)]
    gc = [_desc(COLS, N.DS_F32, ptr=base + (3 + i) * (1 << 22)) for i in range(2)]
    d = (C.c_float * 16)()
    ws = (C.c_uint8 * 4096)()
    who = "ds_aas_matrix_bwd"

    def call(q=q, ks=q, k=kc, mode=N.DS_SIM_COSINE, d_Dm=d, ldd=5, grads=None):
        return lib.ds_aas_matrix_bwd(q, ks, ks, k, k, 0.0, mode, d_Dm, ldd, *(grads or gr + gc), ws, 4096, None)

    bad = [
        (dict(d_Dm=None), "null"),
        (dict(ldd=4), "ldd"),
        (dict(mode=N.DS_SIM_MINMAX_COSINE), "mode"),
        (dict(q=_desc(ROWS, N.DS_F16, ptr=0)), "null"),
        (dict(ks=_desc((2,) + ROWS[1:], N.DS_F16)), "same images"),            # row caches disagree
        (dict(k=_desc((5, 1, 2, 128, 40), N.DS_F16)), "match"),                # columns of another head dim
        (dict(grads=gr + [gc[0], _desc((5, 1, 2, 64, 64), N.DS_F32, ptr=base)]), "shape"),
        (dict(grads=[_desc(ROWS, N.DS_F16, ptr=base)] + gr[1:] + gc), "float32"),
    ]
    for kw, text in bad:
        assert call(**kw) == N.DS_ERR_INVALID, kw
        msg = N.last_error()
        assert msg.startswith(who + ": ") and text in msg, (kw, msg)
    assert call() == N.DS_ERR_WORKSPACE and N.last_error().startswith(who + ": ")
    # dk_self / dk: the same tensor (rows = columns) or disjoint; a partial overlap is refused
    sq = [_desc(ROWS, N.DS_F32, ptr=base + i * (1 << 22)) for i in range(3)]
    assert lib.ds_aas_matrix_bwd(q, q, q, q, q, 0.0, 0, d, 3, *sq, sq[1], sq[2], ws, 4096, None) == N.DS_ERR_WORKSPACE
    shifted = [_desc(ROWS, N.DS_F32, ptr=t.ptr + 4 * 64) for t in sq[1:]]
    assert lib.ds_aas_matrix_bwd(q, q, q, q, q, 0.0, 0, d, 3, *sq, *shifted, ws, 4096, None) == N.DS_ERR_INVALID
    assert N.last_error().startswith(who + ": ") and "overlap" in N.last_error()
    d96 = _desc((3, 1, 2, 128, 96), N.DS_F16)
    g96 = [_desc((3, 1, 2, 128, 96), N.DS_F32, ptr=base + i * (1 << 22)) for i in range(5)]
    assert lib.ds_aas_matrix_bwd(d96, d96, d96, d96, d96, 0.0, 0, d, 3, *g96, ws, 4096, None) == N.DS_ERR_UNSUPPORTED
    assert N.last_error().startswith(who + ": ")


def test_python_wrapper_needs_cuda():
    from diffsim_b200 import ops

    x = torch.zeros(ROWS, dtype=torch.float16)
    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.aas_matrix_bwd(x, x, x, x, x, torch.ones(3, 3))


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour on a machine without a GPU")
def test_matrix_bwd_without_gpu_fails_loudly():
    from diffsim_b200 import ops

    lib = N.load()
    x = torch.zeros(ROWS, dtype=torch.float16)
    g32 = torch.zeros((5,) + ROWS, dtype=torch.float32)
    h = _desc(ROWS, N.DS_F16, ptr=x.data_ptr())
    f = [_desc(ROWS, N.DS_F32, ptr=g32[i].data_ptr()) for i in range(5)]
    d = torch.ones(3, 3)
    ws = torch.zeros(lib.ds_aas_matrix_bwd_workspace_bytes(h, h), dtype=torch.uint8)
    assert lib.ds_aas_matrix_bwd(h, h, h, h, h, 0.0, 0, d.data_ptr(), 3, *f, ws.data_ptr(), ws.numel(),
                                 None) == N.DS_ERR_CUDA
    assert g32.abs().sum().item() == 0.0
    xr = x.clone().requires_grad_(True)
    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.aas_matrix(xr, x, x, x, x)


# ---- the float64 fold model

def _caches(nr, nc, dtype, seed=0, B=1, H=2, S=24, D=8):
    g = torch.Generator().manual_seed(seed)
    base = torch.randn(3, B, H, S, D, generator=g, dtype=torch.float64)
    rows = [(base + 0.6 * torch.randn(3, B, H, S, D, generator=g, dtype=torch.float64)).to(dtype) for _ in range(nr)]
    cols = [(base + 0.6 * torch.randn(3, B, H, S, D, generator=g, dtype=torch.float64)).to(dtype) for _ in range(nc)]
    q, ks, vs = (torch.stack([r[i] for r in rows]) for i in range(3))
    k, v = (torch.stack([c[i] for c in cols]) for i in (1, 2))
    return q, ks, vs, k, v, torch.randn(nr, nc, generator=g, dtype=torch.float64)


def _outputs(q, ks, vs, k, v, rnd):
    X = torch.stack([torch.stack([G._round(G.attention(q[r], k[c], v[c]), rnd) for c in range(k.shape[0])])
                     for r in range(q.shape[0])])
    Y = torch.stack([G._round(G.attention(q[r], ks[r], vs[r]), rnd) for r in range(q.shape[0])])
    return X, Y


@pytest.mark.parametrize("mode", ("cosine", "mse"))
def test_fold_model_is_autograd_when_nothing_is_rounded(mode):
    q, ks, vs, k, v, d = _caches(3, 5, torch.float64)
    X, Y = _outputs(q, ks, vs, k, v, None)
    model = M.matrix_grads_rounded(q, ks, vs, k, v, X, Y, d, mode)
    exact = M.matrix_grads(q, ks, vs, k, v, d, mode)
    for a, b in zip(model, exact):
        assert torch.allclose(a, b, rtol=1e-10, atol=1e-13), float((a - b).abs().max())


def test_fold_model_mutants_exceed_the_tight_tolerance(monkeypatch):
    """A fold scale off by 2^-10, or one column's self term dropped, moves the model by at least 3x the tight tolerance
    of the GPU tests (their Frobenius metric, fp16)."""
    from test_gpu_matrix_grad import TIGHT, _fro

    tol_rows, tol_fro = TIGHT[torch.float16]
    q, ks, vs, k, v, d = _caches(3, 5, torch.float16, seed=1)
    X, Y = _outputs(q, ks, vs, k, v, torch.float16)
    ref = M.matrix_grads_rounded(q, ks, vs, k, v, X, Y, d)
    fold = M.fold_factor
    monkeypatch.setattr(M, "fold_factor", lambda F, rnd: (fold(F, rnd)[0], fold(F, rnd)[1] * (1 + 2.0 ** -10)))
    scaled = M.matrix_grads_rounded(q, ks, vs, k, v, X, Y, d)
    monkeypatch.undo()
    d_drop = d.clone()
    X_drop = X.clone()
    calls = []

    def drop_first(F, rnd):   # remove column 0's self term from each row's fold
        r = len(calls)
        calls.append(r)
        x, y = X_drop[r, 0].double(), Y[r].double()
        cf, _, k_y = M._coefs(x, y, float(d_drop[r, 0]), "cosine")
        return fold(F - cf * (x - k_y * y), rnd)

    monkeypatch.setattr(M, "fold_factor", drop_first)
    dropped = M.matrix_grads_rounded(q, ks, vs, k, v, X, Y, d)
    for mutant in (scaled, dropped):
        assert max(_fro(a, b) for a, b in zip(mutant, ref)) >= 3 * tol_fro
    assert max(G.max_row_err(a, b) for a, b in zip(dropped, ref)) >= 3 * tol_rows
