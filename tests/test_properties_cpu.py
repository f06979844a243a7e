"""Property tests (hypothesis) of the host logic and of the oracle's invariants -- the same invariants the GPU tests check at
full size without an oracle (tests/test_gpu_edges.py)."""
import os

import pytest
import torch
from hypothesis import given, settings, strategies as st

from oracle import aas_oracle as O


@settings(max_examples=60, deadline=None)
@given(n=st.integers(0, 500), world=st.integers(1, 9))
def test_row_blocks_partition_any_size(n, world):
    from diffsim_b200 import scoring

    blocks = [scoring.row_block(n, r, world) for r in range(world)]
    assert blocks[0][0] == 0 and blocks[-1][1] == n
    assert all(a1 == b0 for (_, a1), (b0, _) in zip(blocks, blocks[1:]))          # contiguous, no gaps or overlaps
    sizes = [b - a for a, b in blocks]
    assert min(sizes) >= 0 and max(sizes) - min(sizes) <= 1                       # balanced


@settings(max_examples=40, deadline=None)
@given(n=st.integers(2, 24), k=st.integers(1, 30), larger=st.booleans(), seed=st.integers(0, 10**6))
def test_ranked_indices_are_sorted_stable_and_skip_the_query(n, k, larger, seed):
    from diffsim_b200 import retrieval as R

    g = torch.Generator().manual_seed(seed)
    s = torch.randint(0, 5, (n, n), generator=g).float()      # many ties: the order must still be deterministic
    order, vals = R.ranked_indices(s, k, larger_is_closer=larger)
    assert order.shape == (n, min(k, n - 1))
    for i in range(n):
        row = order[i].tolist()
        assert i not in row and len(set(row)) == len(row)
        v = vals[i]
        assert bool(((v[:-1] >= v[1:]) if larger else (v[:-1] <= v[1:])).all())
        for a, b in zip(row, row[1:]):                          # ties keep index order (stable)
            if s[i, a] == s[i, b]:
                assert a < b


@settings(max_examples=15, deadline=None)
@given(seed=st.integers(0, 10**6), S=st.sampled_from([8, 17, 32]), D=st.sampled_from([8, 16]), c=st.floats(0.25, 4.0))
def test_oracle_invariants(seed, S, D, c):
    g = torch.Generator().manual_seed(seed)
    mk = lambda: torch.randn(1, 2, S, D, generator=g, dtype=torch.float64)  # noqa: E731
    qa, ka, va, qb, kb, vb = (mk() for _ in range(6))
    for mode in ("cosine", "mse"):
        ab = O.aas_pair_score(qa, ka, va, qb, kb, vb, mode=mode, tier="T0")
        ba = O.aas_pair_score(qb, kb, vb, qa, ka, va, mode=mode, tier="T0")
        assert ab == pytest.approx(ba, rel=1e-12, abs=1e-15)                          # diffsim(A,B) == diffsim(B,A)
    assert O.aas_pair_score(qa, ka, va, qa, ka, va, mode="cosine", tier="T0") == pytest.approx(1.0, abs=1e-12)
    assert O.aas_pair_score(qa, ka, va, qa, ka, va, mode="mse", tier="T0") == pytest.approx(0.0, abs=1e-24)
    # the cosine score does not see a common positive scale of the values; MSE scales with its square
    cos = O.aas_pair_score(qa, ka, va, qb, kb, vb, mode="cosine", tier="T0")
    assert O.aas_pair_score(qa, ka, c * va, qb, kb, c * vb, mode="cosine", tier="T0") == pytest.approx(cos, rel=1e-9)
    mse = O.aas_pair_score(qa, ka, va, qb, kb, vb, mode="mse", tier="T0")
    assert O.aas_pair_score(qa, ka, c * va, qb, kb, c * vb, mode="mse", tier="T0") == pytest.approx(c * c * mse, rel=1e-9)
    # attention rows are convex combinations of the value rows
    o = O.attention(qa, kb, vb)
    assert bool((o.amax(dim=-2) <= vb.amax(dim=-2) + 1e-12).all()) and bool((o.amin(dim=-2) >= vb.amin(dim=-2) - 1e-12).all())
    # an explicit scale equal to the default changes nothing
    assert torch.allclose(O.attention(qa, kb, vb), O.attention(qa, kb, vb, scale=D ** -0.5), rtol=1e-12, atol=1e-14)


def test_kernel_choice_hooks_validate_their_argument_and_report_the_value_in_force():
    """The test hooks of include/diffsim_b200.h only store a validated value (no device work): out-of-range arguments are
    ignored and every call returns what is in force -- which is how the GPU tests restore the defaults."""
    from diffsim_b200 import _native

    if not os.path.exists(_native.LIB_PATH):
        pytest.skip("library not built")
    lib = _native.load()
    try:
        assert lib.ds_debug_set_attn_mc(-1) == -1                 # default: multicast for the N x N matrix only
        assert lib.ds_debug_set_attn_mc(1) == 1 and lib.ds_debug_set_attn_mc(7) == 1 and lib.ds_debug_set_attn_mc(0) == 0
        assert lib.ds_debug_set_simmat_blocked(-1) == -1
        assert lib.ds_debug_set_simmat_blocked(1) == 1 and lib.ds_debug_set_simmat_blocked(5) == 1
        assert lib.ds_debug_set_gemm_variant(-1) == -1           # default: pairs when the 256 x 256 tiles fill the clusters
        assert lib.ds_debug_set_gemm_variant(2) == 2 and lib.ds_debug_set_gemm_variant(1) == 2
        assert lib.ds_debug_set_gemm_variant(18) == 2 and lib.ds_debug_set_gemm_variant(-17) == 2
        assert lib.ds_debug_set_gemm_variant(0) == 0
    finally:
        lib.ds_debug_set_attn_mc(-1)
        lib.ds_debug_set_simmat_blocked(-1)
        lib.ds_debug_set_gemm_variant(-1)
