"""Scores between images of different token counts, on the CPU: the float64 oracles the GPU tests use agree with the
reference's own torch lines (diffsim/diffsim.py:177-197) when the two images' S differ, and the library's argument
validation accepts such calls (independent self and cross kv lengths) while it still rejects a k / v or k_self / v_self
pair of different lengths.
"""
import pytest
import torch
import torch.nn.functional as F

from oracle import aas_grad_oracle as G
from oracle import aas_matrix_grad_oracle as M
from oracle import aas_oracle as O

LENGTHS = [(256, 576), (576, 256), (256, 64), (200, 1024)]


def _image(S, D=40, B=2, H=2, seed=0, dtype=torch.float64):
    g = torch.Generator().manual_seed(seed)
    return tuple(torch.randn(B, S, H, D, generator=g).to(dtype).permute(0, 2, 1, 3) for _ in range(3))


def _reference_dir(q_i, k_i, v_i, k_j, v_j, mode):
    """One direction of the reference's lines: sdpa cross vs sdpa self, flat cosine or mse."""
    sdpa = lambda q, k, v: F.scaled_dot_product_attention(q, k, v, dropout_p=0.0, is_causal=False)  # noqa: E731
    cross, self_ = sdpa(q_i, k_j, v_j), sdpa(q_i, k_i, v_i)
    if mode == "cosine":
        return F.cosine_similarity(cross.reshape(-1).unsqueeze(0), self_.reshape(-1).unsqueeze(0))[0]
    return F.mse_loss(cross, self_)


@pytest.mark.parametrize("SA,SB", LENGTHS)
@pytest.mark.parametrize("mode", ("cosine", "mse"))
def test_oracle_scores_are_the_reference_lines_at_mixed_lengths(SA, SB, mode):
    A, B = _image(SA, seed=SA), _image(SB, seed=SB + 1)
    ref = O.reference_pair_score(*A, *B, mode=mode)                     # float64 inputs: the reference in float64
    assert abs(O.aas_pair_score(*A, *B, mode=mode, tier="T0") - float(ref)) < 1e-12
    # 16-bit inputs: the oracle's T1 tier against the reference's lines evaluated in float32 on the same values
    A16, B16 = (tuple(t.half() for t in X) for X in (A, B))
    ref32 = O.reference_pair_score(*(t.float() for t in A16), *(t.float() for t in B16), mode=mode)
    assert abs(O.aas_pair_score(*A16, *B16, mode=mode) - float(ref32)) <= 1e-3 * abs(float(ref32))


@pytest.mark.parametrize("SA,SB", LENGTHS[:3])
@pytest.mark.parametrize("mode", ("cosine", "mse"))
def test_grad_oracles_are_autograd_of_the_reference_lines(SA, SB, mode):
    A, B = _image(SA, D=16, seed=SA), _image(SB, D=16, seed=SB + 1)
    got = G.pair_score_grads(*A, *B, mode)
    leaves = [t.detach().clone().requires_grad_(True) for t in (*A, *B)]
    s = (_reference_dir(*leaves[:3], *leaves[4:6], mode) + _reference_dir(*leaves[3:], *leaves[1:3], mode)) / 2
    ref = torch.autograd.grad(s, leaves)
    for a, b in zip(got, ref):
        assert torch.allclose(a, b, rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("mode", ("cosine", "mse"))
def test_matrix_oracle_at_mixed_lengths(mode):
    rows = [_image(136, D=16, B=1, seed=i) for i in range(2)]
    cols = [_image(300, D=16, B=1, seed=10 + i) for i in range(3)]
    q, ks, vs = (torch.stack([r[i] for r in rows]) for i in range(3))
    _, k, v = (torch.stack([c[i] for c in cols]) for i in range(3))
    dm = M.matrix_value(q, ks, vs, k, v, mode)
    for r in range(2):
        for c in range(3):
            assert abs(float(dm[r, c]) - float(_reference_dir(q[r], ks[r], vs[r], k[c], v[c], mode))) < 1e-12
    d = torch.randn(2, 3, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    got = M.matrix_grads(q, ks, vs, k, v, d, mode)
    leaves = [t.detach().clone().requires_grad_(True) for t in (q, ks, vs, k, v)]
    lq, lks, lvs, lk, lv = leaves
    total = sum(d[r, c] * _reference_dir(lq[r], lks[r], lvs[r], lk[c], lv[c], mode) for r in range(2) for c in range(3))
    for a, b in zip(got, torch.autograd.grad(total, leaves)):
        assert torch.allclose(a, b, rtol=1e-9, atol=1e-12)


# ------------------------------------------------------------------------------------------------------
# argument validation (runs before any device work, so it needs no GPU)
# ------------------------------------------------------------------------------------------------------
def _lib():
    from diffsim_b200 import _native as N

    try:
        return N, N.load()
    except RuntimeError as e:
        pytest.skip(str(e))


def _t5(N, shape, buf, dtype=torch.float16):
    d = N.Tensor5()
    d.ptr = buf.data_ptr()
    d.size[:] = list(shape)
    strides, s = [], 1
    for n in reversed(shape):
        strides.insert(0, s)
        s *= n
    d.stride[:] = strides
    d.dtype = N.DS_F16 if dtype == torch.float16 else N.DS_F32
    return d


def test_validation_accepts_independent_self_and_cross_lengths():
    """A call with S_q != S_self != S_cross passes validation and reaches the device check (DS_ERR_CUDA without a GPU);
    k / v or k_self / v_self of different lengths stop at validation (DS_ERR_INVALID)."""
    N, lib = _lib()
    if lib.ds_device_ok() == N.DS_OK:
        pytest.skip("a device is present: the calls below would run")
    buf = torch.empty(1 << 16, dtype=torch.int64)   # never dereferenced: the calls stop before device work
    ws = torch.empty(1 << 22, dtype=torch.uint8)
    gi = torch.zeros(4, dtype=torch.int32)
    q = _t5(N, (2, 1, 2, 200, 64), buf)

    def groups(ks, vs, k, v):
        return lib.ds_aas_groups(q, ks, vs, k, v, gi.data_ptr(), gi.data_ptr(), 1, gi.data_ptr(), 1, 0.0,
                                 N.DS_SIM_COSINE, buf.data_ptr(), ws.data_ptr(), ws.numel(), None)

    def matrix(ks, vs, k, v):
        return lib.ds_aas_matrix(q, ks, vs, k, v, 0.0, N.DS_SIM_COSINE, buf.data_ptr(), 8, ws.data_ptr(), ws.numel(),
                                 None)

    s256, s576 = _t5(N, (2, 1, 2, 256, 64), buf), _t5(N, (3, 1, 2, 576, 64), buf)
    s128, s300 = _t5(N, (2, 1, 2, 128, 64), buf), _t5(N, (3, 1, 2, 300, 64), buf)
    for call in (groups, matrix):
        assert call(s256, s256, s576, s576) == N.DS_ERR_CUDA
        assert call(s256, s256, s576, s300) == N.DS_ERR_INVALID
        assert "k and v" in N.last_error()
        assert call(s256, s128, s576, s576) == N.DS_ERR_INVALID
        assert "k_self and v_self" in N.last_error()
    f32 = torch.empty(1 << 20, dtype=torch.float32)
    grads = [_t5(N, tuple(t.size), f32, torch.float32) for t in (q, s256, s256, s576, s576)]
    rc = lib.ds_aas_groups_bwd(q, s256, s256, s576, s576, gi.data_ptr(), gi.data_ptr(), 1, gi.data_ptr(), 1, 0.0,
                               N.DS_SIM_COSINE, f32.data_ptr(), *grads[:3], *[_t5(N, tuple(t.size), buf, torch.float32)
                                                                             for t in (s576, s576)],
                               ws.data_ptr(), ws.numel(), None)
    assert rc in (N.DS_ERR_CUDA, N.DS_ERR_WORKSPACE), N.last_error()
    rc = lib.ds_aas_groups_bwd(q, s256, s128, s576, s576, gi.data_ptr(), gi.data_ptr(), 1, gi.data_ptr(), 1, 0.0,
                               N.DS_SIM_COSINE, f32.data_ptr(), *grads, ws.data_ptr(), ws.numel(), None)
    assert rc == N.DS_ERR_INVALID
