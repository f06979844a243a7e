"""ds_qkv_project_bwd without a GPU: argument checks come before the device and name the entry point, the workspace
query needs no device, the call fails loudly rather than computing on the host, and the float64 oracle is the
gradient torch autograd gives."""
import ctypes as C

import pytest
import torch

from diffsim_b200 import _native as N
from oracle import qkv_grad_oracle as QG

ROWS, C_IN, N_OUT, COLS = 64, 64, 192, 64


def _bufs():
    keep = [torch.zeros(ROWS * C_IN + 64, dtype=torch.float16) for _ in range(6)]
    al = [t.data_ptr() + (-t.data_ptr()) % 16 for t in keep]   # 16-byte aligned bases
    return keep, al


def _call(lib, al, **kw):
    a = dict(hidden=al[0], n_rows=ROWS, ld_hidden=C_IN, c_in=C_IN, weight=al[1], ld_weight=C_IN, n_out=N_OUT,
             cols_per_out=COLS, dy=[al[2]] * 3, ld_dy=[COLS] * 3, dhidden=al[3], ld_dhidden=C_IN, dweight=al[4],
             ld_dweight=C_IN, dbias=al[5], dtype=N.DS_F16)
    a.update(kw)
    dy = None if a["dy"] is None else (C.c_void_p * len(a["dy"]))(*a["dy"])
    ld = (C.c_int64 * len(a["ld_dy"]))(*a["ld_dy"])
    return lib.ds_qkv_project_bwd(a["hidden"], a["n_rows"], a["ld_hidden"], a["c_in"], a["weight"], a["ld_weight"],
                                  a["n_out"], a["cols_per_out"], dy, ld, a["dhidden"], a["ld_dhidden"], a["dweight"],
                                  a["ld_dweight"], a["dbias"], a["dtype"], None, 0, None)


@pytest.mark.parametrize("bad, code", [
    (dict(dy=None), N.DS_ERR_INVALID),                                  # null dy array
    (dict(dy=[0, 0, 0]), N.DS_ERR_INVALID),                             # null dy tensors
    (dict(weight=None), N.DS_ERR_INVALID),                              # dhidden wanted without the weight
    (dict(hidden=None), N.DS_ERR_INVALID),                              # dweight wanted without the input
    (dict(hidden="+2"), N.DS_ERR_INVALID),                              # misaligned base
    (dict(dbias="+8"), N.DS_ERR_INVALID),
    (dict(ld_dy=[COLS + 4] * 3), N.DS_ERR_INVALID),                     # row stride not a multiple of 8
    (dict(ld_dweight=C_IN + 4), N.DS_ERR_INVALID),
    (dict(cols_per_out=60, n_out=180), N.DS_ERR_INVALID),              # columns per output not a multiple of 8
    (dict(c_in=60, ld_hidden=64, ld_weight=64), N.DS_ERR_INVALID),
    (dict(n_out=4 * COLS), N.DS_ERR_INVALID),                           # four gradient tensors
    (dict(n_rows=0), N.DS_ERR_INVALID),
    (dict(dtype=N.DS_F32), N.DS_ERR_UNSUPPORTED),
])
def test_arguments_are_checked_before_the_device(bad, code):
    lib = N.load()
    keep, al = _bufs()
    names = ["hidden", "weight", "dy", "dhidden", "dweight", "dbias"]
    for k, v in list(bad.items()):
        if isinstance(v, str):
            bad[k] = al[names.index(k)] + int(v)
    assert _call(lib, al, **bad) == code
    assert N.last_error().startswith("ds_qkv_project_bwd:")


def test_workspace_query_needs_no_device():
    lib = N.load()
    # SD-1.5 up0 at 96 images: the weight gradient's 768 k blocks need at least three fp32 partials of 3840 x 1280
    assert lib.ds_qkv_project_bwd_workspace_bytes(96 * 2 * 256, 1280, 3840, 1280) >= 3 * 3840 * 1280 * 4
    assert lib.ds_qkv_project_bwd_workspace_bytes(300, 1000, 3000, 1000) >= 300 * 1000 * 4
    assert lib.ds_qkv_project_bwd_workspace_bytes(0, 1280, 3840, 1280) > 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour on a machine without a GPU")
def test_no_gpu_means_loud_failure():
    lib = N.load()
    keep, al = _bufs()
    assert _call(lib, al) == N.DS_ERR_CUDA
    assert all((t == 0).all() for t in keep)   # nothing was computed on the host
    from diffsim_b200 import ops

    x = torch.randn(8, 64).half()
    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.qkv_project_bwd(x, torch.randn(192, 64).half(), [torch.randn(8, 64).half()] * 3)


def test_oracle_is_the_autograd_gradient_of_a_linear_layer():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(5, 7, 16, generator=g, dtype=torch.float64, requires_grad=True)
    w = torch.randn(24, 16, generator=g, dtype=torch.float64, requires_grad=True)
    b = torch.randn(24, generator=g, dtype=torch.float64, requires_grad=True)
    dys = [torch.randn(5, 7, 8, generator=g, dtype=torch.float64) for _ in range(3)]
    y = torch.nn.functional.linear(x, w, b)
    gx, gw, gb = torch.autograd.grad(y, (x, w, b), torch.cat(dys, dim=-1))
    (dx, dw, db), (bx, bw, bb) = QG.qkv_bwd(x.detach(), w.detach(), dys)
    assert torch.allclose(dx, gx.reshape(dx.shape)) and torch.allclose(dw, gw) and torch.allclose(db, gb)
    assert (bx >= dx.abs()).all() and (bw >= dw.abs()).all() and (bb >= db.abs()).all()
