"""The matrix K5 backward by gradient family on a B200: ops.aas_matrix_bwd with need_rows / need_cols.

The row terms alone (dq, dk_self, dv_self) and the column terms alone (dk, dv) are bitwise what the full call gives
them when the self gradients are separate buffers: every per-term quantity depends only on its entry and its row, and
every gradient row receives its terms in the full call's order.  So the sharded backward -- own rows against all
columns, all rows against own columns -- is bitwise one device's, which is checked here on one GPU with the sharding
emulated, and through aas_matrix_sharded on a one-rank process group.
"""
import pytest
import torch

from test_gpu_matrix_grad import D_ALL, DTYPES, LAYOUTS, NC, NR, _case, _same

pytestmark = pytest.mark.gpu


def _parts(q, ks, vs, k, v, d, mode="cosine", scale=None):
    from diffsim_b200 import ops

    full = ops.aas_matrix_bwd(q, ks, vs, k, v, d, mode, scale)
    rows = ops.aas_matrix_bwd(q, ks, vs, k, v, d, mode, scale, need_cols=False)
    cols = ops.aas_matrix_bwd(q, ks, vs, k, v, d, mode, scale, need_rows=False)
    return full, rows, cols


def _check_parts(full, rows, cols):
    assert rows[3] is None and rows[4] is None
    assert cols[0] is None and cols[1] is None and cols[2] is None
    for i in range(3):
        _same(rows[i], full[i])
    for i in (3, 4):
        _same(cols[i], full[i])
    assert all(t.abs().sum() > 0 for t in full)


@pytest.mark.parametrize("mode", ("cosine", "mse"))
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("D", D_ALL)
def test_each_family_is_bitwise_the_full_call(D, dtype, layout, mode):
    q, ks, vs, k, v, d = _case(D, dtype, layout, seed=D + 1)
    _check_parts(*_parts(q, ks, vs, k, v, d, mode))


@pytest.mark.parametrize("D,dtype,mode", [(64, torch.float16, "cosine"), (160, torch.bfloat16, "mse"),
                                          (40, torch.bfloat16, "cosine")])
def test_each_family_ragged_length_and_scale(D, dtype, mode):
    q, ks, vs, k, v, d = _case(D, dtype, "sd", S=193, seed=4)
    _check_parts(*_parts(q, ks, vs, k, v, d, mode, 0.11))


def test_each_family_under_row_and_column_chunking(monkeypatch):
    from diffsim_b200 import _native as N, ops

    q, ks, vs, k, v, d = _case(72, torch.float16, "sd", seed=9)
    lib = N.load()
    ws = lambda r, c: lib.ds_aas_matrix_bwd_workspace_bytes(ops._desc(q[:r], 5), ops._desc(k[:c], 5))  # noqa: E731
    whole = _parts(q, ks, vs, k, v, d)
    # blocks of one row: the full call is bitwise one call, and so is each family
    monkeypatch.setattr(ops, "GROUPS_BWD_WORKSPACE_CAP", ws(1, NC))
    assert len(ops._matrix_spans(NR, NC, ws)) == NR
    full, rows, cols = _parts(q, ks, vs, k, v, d)
    _check_parts(full, rows, cols)
    for a, b in zip(full, whole[0]):
        _same(a, b)
    # column blocks of two: each block folds its own self term, in the full call and in the row family alike
    monkeypatch.setattr(ops, "GROUPS_BWD_WORKSPACE_CAP", ws(1, 2))
    assert len(ops._matrix_spans(NR, NC, ws)) == NR * 3
    _check_parts(*_parts(q, ks, vs, k, v, d))
    # the column pass of a sharded backward: all rows against a block of columns, cut into row blocks
    monkeypatch.setattr(ops, "GROUPS_BWD_WORKSPACE_CAP", ws(1, 2))
    cut = ops.aas_matrix_bwd(q, ks, vs, k[1:3], v[1:3], d[:, 1:3], need_rows=False)
    _same(cut[3], whole[0][3][1:3])
    _same(cut[4], whole[0][4][1:3])


def _shared(N_img, dtype=torch.float16, layout="sd", seed=12, D=64):
    """one cache of N_img images (rows = columns) and a d_Dm"""
    from test_gpu_matrix_grad import _cache

    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(seed)
    base = torch.randn(3, 2, 136, 2, D, generator=g)
    q, k, v = _cache(N_img, 2, 2, 136, D, dtype, layout, dev, g, base)
    return q, k, v, torch.randn(N_img, N_img, generator=g).to(dev)


def _reference(q, k, v, d, mode="cosine"):
    """one device's aas_matrix_bwd with separate self buffers"""
    from diffsim_b200 import ops

    grads = [torch.zeros(t.shape, dtype=torch.float32, device=t.device) for t in (q, k, v, k, v)]
    return ops.aas_matrix_bwd(q, k, v, k, v, d, mode, grads=grads)


@pytest.mark.parametrize("world,mode,layout", [(2, "cosine", "sd"), (3, "mse", "dit"), (3, "cosine", "contig")])
def test_emulated_shards_are_bitwise_one_device(world, mode, layout):
    from diffsim_b200 import scoring

    n = 7
    q, k, v, d = _shared(n, torch.bfloat16 if mode == "mse" else torch.float16, layout)
    ref = _reference(q, k, v, d, mode)
    for rank in range(world):
        r0, r1 = scoring.row_block(n, rank, world)
        dq, dks, dvs, dk, dv = scoring._matrix_grad_block(q, k, v, r0, r1, d, mode, None)
        for got, want in zip((dq, dks, dvs, dk, dv), ref):
            _same(got, want[r0:r1])
        _same(dks + dk, ref[1][r0:r1] + ref[3][r0:r1])
        _same(dvs + dv, ref[2][r0:r1] + ref[4][r0:r1])


def test_sharded_block_backward_on_one_rank(tmp_path):
    import torch.distributed as dist

    from diffsim_b200 import ops, scoring

    n = 5
    q, k, v, _ = _shared(n, seed=13)
    leaves = [t.detach().requires_grad_() for t in (q, k, v)]
    dist.init_process_group("nccl", init_method=f"file://{tmp_path}/store", rank=0, world_size=1, device_id=q.device)
    try:
        block = scoring.aas_matrix_sharded(scoring.QKVCache(*leaves), gather_to_all=False)
        block.retain_grad()
        torch.nn.functional.cross_entropy(block / 0.05, torch.arange(n, device=q.device), reduction="sum").backward()
    finally:
        dist.destroy_process_group()
    with torch.no_grad():
        _same(block.detach(), ops.aas_matrix(q, k, v, k, v))
    ref = _reference(q, k, v, block.grad)
    for leaf, want in zip(leaves, (ref[0], ref[1] + ref[3], ref[2] + ref[4])):
        assert leaf.grad is not None and leaf.grad.dtype == leaf.dtype
        assert torch.equal(leaf.grad, want.to(leaf.dtype))


def test_launch_counts_of_the_three_forms():
    from diffsim_b200 import ops

    q, ks, vs, k, v, d = _case(64, torch.float16, "sd", seed=14)
    counts = []
    for kw in (dict(), dict(need_cols=False), dict(need_rows=False)):
        n0 = ops.LAUNCHES
        ops.aas_matrix_bwd(q, ks, vs, k, v, d, **kw)
        counts.append(ops.LAUNCHES - n0)
    assert counts == [9, 9, 8]


def test_each_family_repeats_bitwise():
    from diffsim_b200 import ops

    q, ks, vs, k, v, d = _case(128, torch.bfloat16, "contig", seed=15)
    for kw in (dict(need_cols=False), dict(need_rows=False)):
        a = ops.aas_matrix_bwd(q, ks, vs, k, v, d, **kw)
        b = ops.aas_matrix_bwd(q, ks, vs, k, v, d, **kw)
        for x, y in zip(a, b):
            assert (x is None) == (y is None)
            if x is not None:
                _same(x, y)
