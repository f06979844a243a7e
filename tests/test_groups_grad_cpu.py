"""Grouped K5 backward without a GPU: argument checks of ds_aas_groups_bwd / _pairs_bwd / _triplets_bwd before the
device is touched, the workspace queries, the loud failure without a device, and a model of the contribution lists."""
import ctypes as C
import math

import pytest
import torch

from diffsim_b200 import _native as N


def _desc(shape, dtype, ptr=256, strides=None):
    t = N.Tensor5()
    t.ptr = ptr
    t.size[:] = list(shape)
    t.stride[:] = strides if strides is not None else [math.prod(shape[i + 1:]) for i in range(5)]
    t.dtype = dtype
    return t


S = (3, 1, 2, 128, 64)
NUMEL = math.prod(S)


def _f32(ptr):
    return _desc(S, N.DS_F32, ptr=ptr)


def test_workspace_queries_grow_with_the_list():
    lib = N.load()
    h = _desc(S, N.DS_F16)
    one = lib.ds_aas_groups_bwd_workspace_bytes(h, h, 1, 1)
    img = math.prod(S[1:]) * 2
    assert one >= 4 * img   # X, Y, fx, fy
    assert lib.ds_aas_groups_bwd_workspace_bytes(h, h, 1, 9) - one >= 8 * 3 * img   # X, fx, fy per entry
    assert lib.ds_aas_groups_bwd_workspace_bytes(h, h, 0, 0) == 256
    assert lib.ds_aas_pairs_bwd_workspace_bytes(h, 4) >= lib.ds_aas_groups_bwd_workspace_bytes(h, h, 8, 8)
    assert lib.ds_aas_triplets_bwd_workspace_bytes(h, 4) >= lib.ds_aas_groups_bwd_workspace_bytes(h, h, 12, 16)


def test_groups_bwd_validates_before_touching_the_device():
    lib = N.load()
    h = _desc(S, N.DS_F16)
    base = 1 << 20
    f = [_f32(base + i * 4 * NUMEL) for i in range(5)]
    idx = (C.c_int32 * 4)(0, 1, 2, 3)
    d = (C.c_float * 4)()
    ws = (C.c_uint8 * 4096)()

    def call(who="ds_aas_groups_bwd", q=h, mode=N.DS_SIM_COSINE, d_dir=d, grads=None, gq=idx, ws_bytes=4096):
        g = grads or [f[0], f[1], f[2], f[1], f[2]]
        if who == "ds_aas_groups_bwd":
            return lib.ds_aas_groups_bwd(q, h, h, h, h, gq, idx, 1, idx, 2, 0.0, mode, d_dir, *g, ws, ws_bytes, None)
        if who == "ds_aas_pairs_bwd":
            return lib.ds_aas_pairs_bwd(q, h, h, gq, 2, 0.0, mode, d_dir, *g[:3], ws, ws_bytes, None)
        return lib.ds_aas_triplets_bwd(q, h, h, gq, 1, 0.0, mode, d_dir, d, *g[:3], ws, ws_bytes, None)

    for who in ("ds_aas_groups_bwd", "ds_aas_pairs_bwd", "ds_aas_triplets_bwd"):
        bad = [
            (dict(gq=None), "null"),
            (dict(q=_desc(S, N.DS_F16, ptr=0)), "null"),
            (dict(q=_desc(S, N.DS_F16, ptr=24)), "aligned"),
            (dict(mode=N.DS_SIM_MINMAX_COSINE), "mode"),
            (dict(d_dir=None), "null"),
            (dict(grads=[_desc(S, N.DS_F16, ptr=base)] + f[1:]), "float32"),
            (dict(grads=[_desc((3, 1, 2, 64, 64), N.DS_F32, ptr=base)] + f[1:]), "shape"),
        ]
        for kw, text in bad:
            assert call(who, **kw) == N.DS_ERR_INVALID, (who, kw)
            msg = N.last_error()
            assert msg.startswith(who + ": ") and text in msg, msg
        assert call(who) == N.DS_ERR_WORKSPACE and N.last_error().startswith(who + ": ")
    # dk_self / dk: the same tensor or disjoint; partial overlap and mixed aliasing are refused
    shifted = _f32(f[3].ptr + 4 * 64)
    assert call(grads=[f[0], f[1], f[2], _f32(f[1].ptr + 4 * 64), f[4]]) == N.DS_ERR_INVALID
    assert "overlap" in N.last_error()
    assert call(grads=[f[0], f[1], f[2], f[1], shifted]) == N.DS_ERR_INVALID
    assert call(grads=[f[0], f[1], f[2], f[3], f[4]]) == N.DS_ERR_WORKSPACE   # disjoint: accepted
    d96 = _desc((3, 1, 2, 128, 96), N.DS_F16)
    g96 = [_desc((3, 1, 2, 128, 96), N.DS_F32, ptr=base + i * (1 << 22)) for i in range(5)]
    assert lib.ds_aas_groups_bwd(d96, d96, d96, d96, d96, idx, idx, 1, idx, 2, 0.0, 0, d, *g96, ws, 4096,
                                 None) == N.DS_ERR_UNSUPPORTED
    assert lib.ds_aas_groups_bwd(h, h, h, h, h, idx, idx, -1, idx, 2, 0.0, 0, d, *f, ws, 4096, None) == N.DS_ERR_INVALID
    assert lib.ds_aas_groups_bwd(h, h, h, h, h, idx, idx, 0, idx, 0, 0.0, 0, d, *f, ws, 4096, None) == N.DS_OK


def test_python_wrapper_checks_the_list_lengths():
    from diffsim_b200 import ops

    x = torch.zeros(S, dtype=torch.float16)
    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.aas_groups_bwd(x, x, x, x, x, [0], [0, 1], [1], torch.ones(1))


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour on a machine without a GPU")
def test_groups_bwd_without_gpu_fails_loudly():
    lib = N.load()
    x = torch.zeros(S, dtype=torch.float16)
    g32 = torch.zeros((5,) + S, dtype=torch.float32)
    h = _desc(S, N.DS_F16, ptr=x.data_ptr())
    f = [_f32(g32[i].data_ptr()) for i in range(5)]
    idx = torch.tensor([0, 1, 2], dtype=torch.int32)
    d = torch.ones(2)
    ws = torch.zeros(lib.ds_aas_groups_bwd_workspace_bytes(h, h, 1, 2), dtype=torch.uint8)
    assert lib.ds_aas_groups_bwd(h, h, h, h, h, idx.data_ptr(), idx.data_ptr(), 1, idx.data_ptr(), 2, 0.0, 0,
                                 d.data_ptr(), *f, ws.data_ptr(), ws.numel(), None) == N.DS_ERR_CUDA
    assert g32.abs().sum().item() == 0.0
    from diffsim_b200 import ops

    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.aas_pairs_bwd(x, x, x, [[0, 1]], torch.ones(1))
    xr = x.clone().requires_grad_(True)
    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.aas_pairs(xr, x, x, [[0, 1]])


# ---- the contribution lists (build_lists_kernel), modelled in Python

def contribution_lists(group_q, group_off, kv_idx, aliased, n_k):
    """{(family, key): [tau, ...]}: family "q" keyed by the query image, family "kv" by the kv image of a cross term and
    the query image of a self term (offset by n_k when dk_self is a separate buffer); tau = 2t (cross), 2t + 1 (self)."""
    lists = {}
    for g, i in enumerate(group_q):
        for t in range(group_off[g], group_off[g + 1]):
            for tau, kv_key in ((2 * t, kv_idx[t]), (2 * t + 1, i if aliased else n_k + i)):
                lists.setdefault(("q", i), []).append(tau)
                lists.setdefault(("kv", kv_key), []).append(tau)
    return {key: sorted(v) for key, v in sorted(lists.items())}


def per_entry_order(group_q, group_off, kv_idx, aliased, n_k):
    """The order in which one ds_aas_dir_bwd call per entry adds into each gradient row: cross launch, then self."""
    writes = {}
    for g, i in enumerate(group_q):
        for t in range(group_off[g], group_off[g + 1]):
            writes.setdefault(("q", i), []).append(2 * t)
            writes.setdefault(("kv", kv_idx[t]), []).append(2 * t)
            writes.setdefault(("q", i), []).append(2 * t + 1)
            writes.setdefault(("kv", i if aliased else n_k + i), []).append(2 * t + 1)
    return writes


@pytest.mark.parametrize("aliased", (True, False))
def test_contribution_lists_follow_the_per_entry_order(aliased):
    # query image 0 in two groups, image 0 paired with itself, image 1 repeated, image 4 only a kv image
    gq, go, kv = [0, 3, 0, 2], [0, 3, 4, 5, 7], [1, 2, 0, 1, 4, 1, 3]
    lists = contribution_lists(gq, go, kv, aliased, 5)
    assert lists == per_entry_order(gq, go, kv, aliased, 5)
    assert lists[("q", 0)] == [0, 1, 2, 3, 4, 5, 8, 9]
    assert ("q", 4) not in lists and lists[("kv", 4)] == [8]
    if aliased:
        assert lists[("kv", 0)] == [1, 3, 4, 5, 9]   # self terms of image 0 and its self pairing (cross 4, self 5)
    else:
        assert lists[("kv", 0)] == [4] and lists[("kv", 5)] == [1, 3, 5, 9]
    # every term sits in exactly one list of each family
    for fam in ("q", "kv"):
        terms = sorted(t for (f, _), v in lists.items() if f == fam for t in v)
        assert terms == list(range(2 * len(kv)))
