"""The matrix backward by gradient family, without a GPU: the null-family rules of ds_aas_matrix_bwd, checked before the
device is touched; the loud failure without a device; and the differentiable row block of aas_matrix_sharded on gloo
ranks, with the per-rank block and backward replaced by the float64 oracle.  What the gloo test checks is the sharded
backward's plumbing (the gathers of dL/dDm and of Q, K, V, the row and column passes' slices, the sum of the self and
column gradients): the sharded gradients must equal single-process float64 autograd of the whole matrix."""
import ctypes as C
import math
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from diffsim_b200 import _native as N

ROWS, COLS = (3, 1, 2, 128, 64), (5, 1, 2, 128, 64)
WHO = "ds_aas_matrix_bwd"


def _desc(shape, dtype, ptr=256):
    t = N.Tensor5()
    t.ptr = ptr
    t.size[:] = list(shape)
    t.stride[:] = [math.prod(shape[i + 1:]) for i in range(5)]
    t.dtype = dtype
    return t


def test_gradient_families_are_checked_before_the_device():
    lib = N.load()
    q, kc = _desc(ROWS, N.DS_F16), _desc(COLS, N.DS_F16)
    base = 1 << 24
    gr = [_desc(ROWS, N.DS_F32, ptr=base + i * (1 << 22)) for i in range(3)]
    gc = [_desc(COLS, N.DS_F32, ptr=base + (3 + i) * (1 << 22)) for i in range(2)]
    null = N.Tensor5()
    d = (C.c_float * 16)()
    ws = (C.c_uint8 * 4096)()

    def call(grads, rows=q, cols=kc, ldd=5):
        return lib.ds_aas_matrix_bwd(rows, rows, rows, cols, cols, 0.0, N.DS_SIM_COSINE, d, ldd, *grads, ws, 4096, None)

    bad = [
        ([null] + gr[1:] + gc, "all given or all null"),            # a partial row family
        (gr[:2] + [null] + gc, "all given or all null"),
        (gr + [gc[0], null], "both given or both null"),             # a partial column family
        ([null] * 5, "all five gradients are null"),
    ]
    for grads, text in bad:
        assert call(grads) == N.DS_ERR_INVALID, text
        msg = N.last_error()
        assert msg.startswith(WHO + ": ") and text in msg, msg
    # dk_self / dk one tensor (rows = columns) needs both families
    sq = [_desc(ROWS, N.DS_F32, ptr=base + i * (1 << 22)) for i in range(3)]
    for grads in ([null, sq[1], sq[2], sq[1], sq[2]], [sq[0], sq[1], sq[2], null, sq[2]]):
        assert call(grads, cols=q, ldd=3) == N.DS_ERR_INVALID
        msg = N.last_error()
        assert msg.startswith(WHO + ": ") and "only when all five" in msg, msg
    # one whole family is a valid call: it gets as far as the (too small) workspace
    for grads in (gr + [null, null], [null] * 3 + gc):
        assert call(grads) == N.DS_ERR_WORKSPACE, N.last_error()
        assert N.last_error().startswith(WHO + ": ")
    # the given family's tensors are still checked
    assert call(gr[:2] + [_desc(ROWS, N.DS_F16, ptr=base)] + [null, null]) == N.DS_ERR_INVALID
    assert "float32" in N.last_error()
    assert call([null] * 3 + [gc[0], _desc((5, 1, 2, 64, 64), N.DS_F32, ptr=base)]) == N.DS_ERR_INVALID
    assert "shape" in N.last_error()


def test_workspace_query_is_the_full_calls():
    lib = N.load()
    q, kc = _desc(ROWS, N.DS_F16), _desc(COLS, N.DS_F16)
    assert lib.ds_aas_matrix_bwd_workspace_bytes(q, kc) > 256


def test_python_wrapper_families():
    from diffsim_b200 import ops

    x = torch.zeros(ROWS, dtype=torch.float16)
    with pytest.raises(RuntimeError, match="need_rows or need_cols"):
        ops.aas_matrix_bwd(x, x, x, x, x, torch.ones(3, 3), need_rows=False, need_cols=False)
    for kw in (dict(need_rows=False), dict(need_cols=False)):
        with pytest.raises(RuntimeError, match="no CPU path"):
            ops.aas_matrix_bwd(x, x, x, x, x, torch.ones(3, 3), **kw)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour on a machine without a GPU")
def test_one_family_without_gpu_fails_loudly():
    lib = N.load()
    x = torch.zeros(ROWS, dtype=torch.float16)
    g32 = torch.zeros((5,) + ROWS, dtype=torch.float32)
    h = N.Tensor5()
    h.ptr, h.dtype = x.data_ptr(), N.DS_F16
    h.size[:] = list(ROWS)
    h.stride[:] = [math.prod(ROWS[i + 1:]) for i in range(5)]
    f = []
    for i in range(5):
        t = N.Tensor5()
        t.ptr, t.dtype = g32[i].data_ptr(), N.DS_F32
        t.size[:], t.stride[:] = list(ROWS), list(h.stride)
        f.append(t)
    null = N.Tensor5()
    d = torch.ones(3, 3)
    ws = torch.zeros(lib.ds_aas_matrix_bwd_workspace_bytes(h, h), dtype=torch.uint8)
    for grads in (f[:3] + [null, null], [null] * 3 + f[3:]):
        assert lib.ds_aas_matrix_bwd(h, h, h, h, h, 0.0, 0, d.data_ptr(), 3, *grads, ws.data_ptr(), ws.numel(),
                                     None) == N.DS_ERR_CUDA
    assert g32.abs().sum().item() == 0.0


# ---- the sharded backward on gloo ranks

B, H, S, D = 1, 2, 16, 8


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _images(n):
    g = torch.Generator().manual_seed(41)
    base = torch.randn(3, B, S, H * D, generator=g, dtype=torch.float64)
    mem = [base[i] + 0.7 * torch.randn(n, B, S, H * D, generator=g, dtype=torch.float64) for i in range(3)]
    return [m.view(n, B, S, H, D).permute(0, 1, 3, 2, 4) for m in mem]


def _loss(block, r0, n):
    """A row-local loss: InfoNCE of each row against its own image, summed, plus a weighted sum."""
    g = torch.Generator().manual_seed(5)
    w = torch.randn(n, n, generator=g, dtype=torch.float64)[r0: r0 + block.shape[0]]
    tgt = torch.arange(r0, r0 + block.shape[0])
    return torch.nn.functional.cross_entropy(block / 0.3, tgt, reduction="sum") + (w * block).sum()


def _worker(rank, world, port, n_images, similarity, ret):
    import sys

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from diffsim_b200 import scoring
    from oracle import aas_matrix_grad_oracle as M

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        def oracle_block(local, k_all, v_all, sim, scale):
            return M.matrix_value(local.q, local.k, local.v, k_all, v_all, sim, scale)

        def oracle_grads(q_all, k_all, v_all, r0, r1, d_full, sim, scale):
            own = slice(r0, r1)
            with torch.enable_grad():   # a Function's backward runs without grad mode
                dq, dks, dvs, _, _ = M.matrix_grads(q_all[own], k_all[own], v_all[own], k_all, v_all, d_full[own], sim,
                                                    scale)
                _, _, _, dk, dv = M.matrix_grads(q_all, k_all, v_all, k_all[own], v_all[own], d_full[:, own], sim, scale)
            return dq, dks, dvs, dk, dv

        scoring._matrix_block = oracle_block
        scoring._matrix_grad_block = oracle_grads
        q, k, v = _images(n_images)
        r0, r1 = scoring.row_block(n_images, rank, world)
        leaves = [t[r0:r1].detach().requires_grad_() for t in (q, k, v)]
        block = scoring.aas_matrix_sharded(scoring.QKVCache(*leaves), similarity, gather_to_all=False)
        assert block.grad_fn is not None and block.shape == (r1 - r0, n_images)
        _loss(block, r0, n_images).backward()
        # single process: float64 autograd of the whole matrix, one leaf per cache (a cache's rows and columns add up)
        ref_leaves = [t.detach().requires_grad_() for t in (q, k, v)]
        full = M.matrix_value(ref_leaves[0], ref_leaves[1], ref_leaves[2], ref_leaves[1], ref_leaves[2], similarity)
        _loss(full, 0, n_images).backward()
        errs = [float((full.detach()[r0:r1] - block.detach()).abs().max()) if r1 > r0 else 0.0]
        for a, b in zip(leaves, ref_leaves):
            assert a.grad is not None and a.grad.shape == a.shape and a.grad.stride() == a.stride()
            if r1 > r0:
                errs.append(float((a.grad - b.grad[r0:r1]).abs().max() / b.grad.abs().max()))
        ret[rank] = errs
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,n_images,similarity", [(2, 5, "cosine"), (3, 7, "mse"), (3, 2, "cosine")])
def test_sharded_gradients_equal_single_process_autograd(world, n_images, similarity):
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), n_images, similarity, ret), nprocs=world, join=True)
    assert sorted(ret.keys()) == list(range(world))
    for rank in range(world):
        assert max(ret[rank]) <= 1e-12, (rank, ret[rank])
