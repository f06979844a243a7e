"""K1 forward at every head dim, dtype, layout, tile edge and softmax regime, and its fused scores.

Every case is compared twice (both references are evaluated on the device):
- tight tier: against the rounding model (attn_fwd_oracle.attention_model / dir_model), which rounds exactly where K1
  rounds, with attn_fwd_oracle's metrics: the largest error in 16-bit ulps, the fraction of elements that differ from
  the model's rounded output and the relative Frobenius error (outputs), the error relative to 1 - cos or to the MSE
  (scores);
- loose tier: test_gpu_parity's tolerances, against exact float64 attention (outputs) or the T1 oracle (scores).
The exact attention differs from what K1 computes by the 16-bit roundings of P; the model does not, so the tight tier
sees errors (a 2^-10 scale, one wrong row, a dropped ragged q row or kv column) that the loose tier cannot.  Two checks
need no model: a known answer (V constant along the sequence) that must come out bitwise, and the MSE score against the
MSE of K1's own stored outputs.
"""
import math

import pytest
import torch

from oracle import aas_oracle as O
from oracle import attn_fwd_oracle as F
from test_gpu_grad_edges import _inputs
from test_gpu_parity import REL_16BIT

pytestmark = pytest.mark.gpu

F16, BF16 = torch.float16, torch.bfloat16
HEAD_DIMS = (40, 64, 72, 80, 128, 160)

# Tight tier: each tolerance is about 4x the worst value observed over this file on a B200 (power limit 1000 W).
#   outputs (attn_fwd_oracle.OUTPUT_METRICS)   max ulps   mismatch   Frobenius   per-row
#     fp16                                       13.8       6.9e-2     8.1e-5      5.7e-4
#     bf16                                        5.2       6.5e-3     1.9e-4      2.4e-3
#   scores (vs 1 - cos / relative MSE)         cosine     MSE
#     fp16                                       3.8e-5     4.4e-6
#     bf16                                       7.7e-5     6.7e-6
# The largest ulp errors and mismatch fractions are flips (attn_fwd_oracle.ulp_error) at small elements of rows with a
# dominant P (D = 160 tile edges, 315 streams) and in single-row outputs of 128 or 320 elements (Sq = 1); the Frobenius
# and per-row errors against the rounded model carry no rounding of their own and catch small global and one-row
# mistakes.  The worst cosine errors are the matrix diagonals, dir(i -> i) ~ 1, measured against the floor
# attn_fwd_oracle.COS_FLOOR of 1 - cos; off the diagonal they are below 1e-5 of 1 - cos.
TIGHT_OUT = {F16: (55.0, 0.28, 3.2e-4, 2.3e-3), BF16: (21.0, 2.6e-2, 7.5e-4, 1e-2)}
TIGHT_SCORE = {(F16, "cosine"): 1.5e-4, (F16, "mse"): 1.8e-5, (BF16, "cosine"): 3e-4, (BF16, "mse"): 2.7e-5}
# Loose tier: test_gpu_parity's absolute output tolerance against exact float64 attention (scaled by the largest |o|
# above 1, as its long-kv test does) and its relative score tolerance against the T1 oracle.
LOOSE_OUT = {F16: 4e-3, BF16: 2e-2}


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return "cuda"


def _ops():
    from diffsim_b200 import ops

    return ops


# ----------------------------------------------------------------------------------------------------------------------
# outputs of ops.attn_fwd
# ----------------------------------------------------------------------------------------------------------------------
def _check_out(name, got, o, out, exact):
    dtype = got.dtype
    errs = F.output_errors(got, o, out, dtype)
    loose = float((got.double() - exact).abs().max())
    loose_tol = LOOSE_OUT[dtype] * max(1.0, float(exact.abs().max()))
    print(f"OUT {name} {str(dtype)[6:]}: vs model " + " ".join(f"{n} {e:.2e}" for n, e in zip(F.OUTPUT_METRICS, errs))
          + f" | vs exact abs {loose:.2e}")
    assert got.dtype == dtype and got.shape == o.shape and torch.isfinite(got).all()
    assert all(e <= t for e, t in zip(errs, TIGHT_OUT[dtype])), errs
    assert loose <= loose_tol, loose


def _out_case(name, q, k, v, scale=None):
    """K1's output against the model and exact attention; returns the model's rescale counts."""
    got = _ops().attn_fwd(q, k, v, scale)
    o, out, rescales = F.attention_model(q, k, v, scale)
    _check_out(name, got, o, out, O.attention(q, k, v, scale))
    return rescales


def _qkv(B, H, Sq, Skv, D, dtype, layout, dev, seed=0):
    q, k, v, _ = _inputs(B, H, Sq, Skv, D, dtype, layout, dev, seed)
    return q, k, v


def _matrix():
    cases = []
    for i, D in enumerate(HEAD_DIMS):
        # one explicit scale per head dim, on alternating dtypes
        scaled, scale = ((F16, 0.05), (BF16, 0.3))[i % 2]
        for dtype in (F16, BF16):
            cases.append((D, dtype, "sd", scale if dtype is scaled else None))
    return cases + [(72, F16, "dit", None), (72, BF16, "dit", 0.3), (128, F16, "bhsd", None), (40, BF16, "bhsd", 0.2)]


@pytest.mark.parametrize("D,dtype,layout,scale", _matrix())
def test_attn_fwd_head_dims_dtypes_layouts(D, dtype, layout, scale):
    dev = _cuda()
    Sq, Skv = (264, 264) if layout == "dit" else (200, 264)   # ragged, more than one tile in both lengths
    q, k, v = _qkv(2, 4, Sq, Skv, D, dtype, layout, dev, seed=D)
    _out_case(f"D={D} {layout} scale={scale}", q, k, v, scale)


# QK's N is the half's kv rows rounded up to 16 (15, 16, 17); a softmax thread owns 32 columns of a half (31, 32, 33);
# a half is 128 rows, a group 256, and 385 leaves a one-row tail after a full group and a full half
KV_EDGES = [1, 15, 16, 17, 31, 32, 33, 127, 128, 129, 255, 256, 257, 385]


@pytest.mark.parametrize("Skv", KV_EDGES)
@pytest.mark.parametrize("Sq", [1, 127, 128, 129, 257])
@pytest.mark.parametrize("D", [64, 160])
def test_attn_fwd_tile_edges(D, Sq, Skv):
    dev = _cuda()
    q, k, v = _qkv(1, 2, Sq, Skv, D, F16, "sd", dev, seed=Sq * 1000 + Skv)
    _out_case(f"D={D} Sq={Sq} Skv={Skv}", q, k, v)


@pytest.mark.parametrize("dtype", [F16, BF16])
@pytest.mark.parametrize("Sq,Skv", [(129, 17), (127, 129), (257, 385)])
def test_attn_fwd_tile_edges_padded_head_dim(Sq, Skv, dtype):
    """D = 72 runs as D_PAD = 80: the padded columns of Q, K and V must not reach the output."""
    dev = _cuda()
    q, k, v = _qkv(1, 2, Sq, Skv, 72, dtype, "sd", dev, seed=Sq + Skv)
    _out_case(f"D=72 Sq={Sq} Skv={Skv}", q, k, v)


def test_attn_fwd_more_streams_than_two_waves():
    """3 x 7 x 15 = 315 (b, h, q tile) streams, more than two per CTA on 148 SMs and not a multiple of the grid; the
    last q tile of every (b, h) has 8 rows."""
    dev = _cuda()
    q, k, v = _qkv(3, 7, 1800, 300, 64, F16, "sd", dev, seed=3)
    _out_case("streams=315", q, k, v)


def _regime(kind, dtype, dev, B=1, H=4, Sq=200, Skv=700, D=64, seed=7):
    q, k, v = _qkv(B, H, Sq, Skv, D, dtype, "sd", dev, seed=seed)
    if kind == "peaky":
        q = (q.float() * 10.0).to(dtype)
    elif kind == "ramp":   # keys growing 1x..10x along the sequence: later halves exceed the first by more than tau
        ramp = (1.0 + 9.0 * torch.arange(Skv, device=dev).float() / Skv).view(1, 1, Skv, 1)
        k = (k.float() * ramp).to(dtype)
    elif kind == "uniform":
        q = torch.zeros_like(q)
    return q, k, v


@pytest.mark.parametrize("dtype", [F16, BF16])
@pytest.mark.parametrize("kind", ["random", "peaky", "ramp", "uniform"])
def test_attn_fwd_softmax_regimes(kind, dtype):
    dev = _cuda()
    q, k, v = _regime(kind, dtype, dev)
    rescales = _out_case(f"{kind}", q, k, v)
    if kind == "ramp":
        assert int(rescales.sum()) > 0   # the case takes the rescale path
    if kind in ("random", "uniform"):
        assert int(rescales.sum()) == 0


def test_attn_fwd_long_kv_bf16():
    dev = _cuda()
    q, k, v = _qkv(1, 4, 256, 4096, 128, BF16, "sd", dev, seed=11)
    _out_case("Skv=4096", q, k, v)


def _near_tau(dtype, dev, D=64, Sq=200, Skv=300):
    """Rows 0 and 1 (one warp) see s = 0 at most in their first kv half and a later maximum 0.5 log2 units below tau
    (row 0: no rescale, P up to 2^(tau - 0.5)) or above it (row 1: one rescale).  Only q[.., 0] of the two rows is
    nonzero, so their logits are q[r, 0] k[j, 0] scale exactly up to the 16-bit rounding of q."""
    q, k, v = _qkv(1, 2, Sq, Skv, D, dtype, "sd", dev, seed=17)
    tau, sl2 = F.TAU[dtype], F.kernel_scale(D) / math.log(2.0)
    g = torch.Generator(device=dev).manual_seed(18)
    kap = torch.empty(1, 2, Skv, device=dev)
    kap[..., :128] = -torch.rand(1, 2, 128, generator=g, device=dev)
    kap[..., 0] = 0.0
    kap[..., 128:] = torch.rand(1, 2, Skv - 128, generator=g, device=dev)
    kap[..., 200] = 1.0
    q, k = q.clone(), k.clone()
    k[..., 0] = kap.to(dtype)
    for r, target in ((0, tau - 0.5), (1, tau + 0.5)):
        q[:, :, r] = 0
        q[:, :, r, 0] = target / sl2
    return q, k, v


@pytest.mark.parametrize("dtype", [F16, BF16])
def test_attn_fwd_near_the_rescale_threshold(dtype):
    dev = _cuda()
    q, k, v = _near_tau(dtype, dev)
    rescales = _out_case("near tau", q, k, v)
    assert rescales[:, :, 0].eq(0).all() and rescales[:, :, 1].eq(1).all()


def _powers_of_two(D, dtype, dev):
    """c_d = +-2^e_d with the sign and exponent varying with d."""
    d = torch.arange(D, device=dev)
    return (torch.where(d % 3 == 1, -1.0, 1.0) * torch.exp2((d % 7 - 3).float())).to(dtype)


@pytest.mark.parametrize("dtype", [F16, BF16])
@pytest.mark.parametrize("D", HEAD_DIMS)
def test_attn_fwd_known_answer(D, dtype):
    """V[j, d] = c_d for every kv row j: l = sum P (the ones-tile MMA) and O_d = c_d sum P (the PV MMA) accumulate the
    same 16-bit P in the same order, so O_d * fp32(1/l) = c_d (1 + O(2^-24)) rounds to c_d exactly, whatever q and k
    are, with a ragged kv tail and on the rescale path.  It also checks that the store epilogue puts every column in
    its place."""
    dev = _cuda()
    ops = _ops()
    c = _powers_of_two(D, dtype, dev)
    for Sq, Skv, kind in ((200, 700, "ramp"), (129, 17, "random"), (1, 129, "peaky"), (257, 1, "random")):
        q, k, _ = _regime(kind, dtype, dev, B=2, H=3, Sq=Sq, Skv=Skv, D=D, seed=D + Skv)
        v = c.expand(2, 3, Skv, D).contiguous()
        got = ops.attn_fwd(q, k, v)
        assert torch.equal(got, c.expand(2, 3, Sq, D)), (Sq, Skv, kind)
        if kind == "ramp":
            assert int(F.attention_model(q, k, v)[2].sum()) > 0


SENTINEL = -1234.5


@pytest.mark.parametrize("D,dtype", [(72, F16), (72, BF16), (64, F16), (160, BF16)])
def test_attn_fwd_out_writes_only_its_view(D, dtype):
    """out= a head-split view of (B, S + 5, H, D + 8) memory: the spare rows and columns (at D = 72 the columns the
    kernel pads D to) keep their sentinel, and the view equals the default output bitwise."""
    dev = _cuda()
    ops = _ops()
    B, H, Sq, Skv = 2, 4, 200, 264
    q, k, v = _qkv(B, H, Sq, Skv, D, dtype, "sd", dev, seed=D)
    ref = ops.attn_fwd(q, k, v)
    store = torch.full((B, Sq + 5, H, D + 8), SENTINEL, dtype=dtype, device=dev)
    view = lambda t: t[:, :Sq, :, :D].permute(0, 2, 1, 3)  # noqa: E731
    outside = torch.ones(store.shape, dtype=torch.bool, device=dev)
    view(outside).fill_(False)
    got = ops.attn_fwd(q, k, v, out=view(store))
    assert got.data_ptr() == store.data_ptr()
    assert torch.equal(view(store), ref)
    assert bool((store[outside] == SENTINEL).all())


# ----------------------------------------------------------------------------------------------------------------------
# scores of ops.aas_pairs, aas_groups and aas_matrix
# ----------------------------------------------------------------------------------------------------------------------
def _images(shape, dtype, dev, alphas=(1.0, 0.6), layout="sd", kv_tokens=None, seed=5):
    from diffsim_b200 import synth

    m = synth.SynthModel(*shape, seed=2334, device=dev)
    g = torch.Generator().manual_seed(seed)
    base = m.new_base(g)
    imgs = []
    for a in alphas:
        q, k, v = m.image(base, a, dtype, layout, g)
        if kv_tokens is not None:   # IP-Adapter: the query attends to a few image tokens
            k, v = k[:, :, :kv_tokens], v[:, :, :kv_tokens]
        imgs.append((q, k, v))
    return imgs


def _stack(images, layout):
    """Three (N,B,H,S,D) caches of the images in their own memory layout: (N,B,S,H*D) for "sd", DiT's packed
    (N,B,S,3,H,D) qkv for "dit"."""
    if layout == "dit":
        packed = torch.stack([torch.stack([t.permute(0, 2, 1, 3) for t in im], dim=2) for im in images])
        return tuple(packed[:, :, :, i].permute(0, 1, 3, 2, 4) for i in range(3))
    return tuple(torch.stack([im[i].permute(0, 2, 1, 3) for im in images]).permute(0, 1, 3, 2, 4) for i in range(3))


class _Model:
    """The model's attention outputs of a set of images, computed once: self outputs and every cross output needed."""

    def __init__(self, images, scale=None):
        self.images, self.scale, self.cache = images, scale, {}

    def att(self, i, j):
        if (i, j) not in self.cache:
            q = self.images[i][0]
            self.cache[(i, j)] = F.attention_model(q, *self.images[j][1:], self.scale)[:2]
        return self.cache[(i, j)]

    def dir(self, i, j, mode):
        xc, xc16 = self.att(i, j)
        ys, ys16 = self.att(i, i)
        return F.scores_from_outputs(xc, xc16, ys, ys16, mode)


def _check_scores(name, dtype, mode, got, model, t1):
    got = [float(x) for x in got]
    tight = max(F.score_error(g, m, mode) for g, m in zip(got, model))
    loose = max(abs(g - t) / max(abs(t), 1e-9) for g, t in zip(got, t1))
    print(f"SCORE {name} {str(dtype)[6:]} {mode}: vs model {tight:.2e} | vs T1 rel {loose:.2e} "
          f"(scores {' '.join(f'{m:.6f}' for m in model)})")
    assert all(math.isfinite(g) for g in got)
    assert tight <= TIGHT_SCORE[(dtype, mode)], tight
    assert loose <= REL_16BIT, loose


def _t1_dir(images, i, j, mode, scale=None):
    return O.aas_directional(*images[i], *images[j][1:], mode=mode, scale=scale)


def _score_case(name, images, layout, mode, scale=None):
    """Both directions of the first two images through aas_groups, their pair score through aas_pairs, and the full
    directional matrix (diagonal included) through aas_matrix."""
    ops = _ops()
    dtype = images[0][0].dtype
    n = len(images)
    q, k, v = _stack(images, layout)
    model = _Model(images, scale)
    dirs = ops.aas_groups(q, k, v, k, v, [0, 1], [0, 1, 2], [1, 0], mode, scale)
    _check_scores(f"{name} groups", dtype, mode, dirs, [model.dir(0, 1, mode), model.dir(1, 0, mode)],
                  [_t1_dir(images, 0, 1, mode, scale), _t1_dir(images, 1, 0, mode, scale)])
    pair = ops.aas_pairs(q, k, v, [[0, 1]], mode, scale)
    _check_scores(f"{name} pairs", dtype, mode, pair, [(model.dir(0, 1, mode) + model.dir(1, 0, mode)) / 2],
                  [(_t1_dir(images, 0, 1, mode, scale) + _t1_dir(images, 1, 0, mode, scale)) / 2])
    mat = ops.aas_matrix(q, k, v, k, v, mode, scale).reshape(-1)
    _check_scores(f"{name} matrix", dtype, mode, mat, [model.dir(i, j, mode) for i in range(n) for j in range(n)],
                  [_t1_dir(images, i, j, mode, scale) for i in range(n) for j in range(n)])


SCORE_SHAPES = {
    # name: (SynthModel shape, layout, kv tokens)
    "sd15_up0": ((2, 8, 256, 160), "sd", None),
    "dit": ((2, 16, 256, 72), "dit", None),
    "clip": ((1, 12, 50, 64), "sd", None),
    "dino": ((1, 6, 257, 64), "sd", None),
    "sdxl": ((2, 10, 1024, 64), "sd", None),
    "ip_adapter": ((2, 8, 256, 160), "sd", 4),
}


@pytest.mark.parametrize("mode", ["cosine", "mse"])
@pytest.mark.parametrize("dtype", [F16, BF16])
@pytest.mark.parametrize("shape", list(SCORE_SHAPES))
def test_scores_shapes(shape, dtype, mode):
    dev = _cuda()
    dims, layout, kv_tokens = SCORE_SHAPES[shape]
    images = _images(dims, dtype, dev, alphas=(1.0, 0.6, 0.98), layout=layout, kv_tokens=kv_tokens)
    _score_case(shape, images, layout, mode, scale=0.1 if shape == "clip" else None)


@pytest.mark.parametrize("mode", ["cosine", "mse"])
@pytest.mark.parametrize("dtype", [F16, BF16])
@pytest.mark.parametrize("alpha", [0.6, 0.98, 0.995])
def test_scores_similarity_regimes(alpha, dtype, mode):
    """SD-1.5 up_blocks[0]; at alpha -> 1 the cosine approaches 1 and its error is measured against 1 - cos."""
    dev = _cuda()
    images = _images((2, 8, 256, 160), dtype, dev, alphas=(1.0, alpha))
    _score_case(f"alpha={alpha}", images, "sd", mode)


def _resampled(images, S):
    """The images at S tokens (nearest source token): captures of the same content at another resolution."""
    S0 = images[0][0].shape[2]
    idx = (torch.arange(S, device=images[0][0].device) * S0) // S
    return [tuple(t[:, :, idx].contiguous() for t in im) for im in images]


@pytest.mark.parametrize("mode", ["cosine", "mse"])
@pytest.mark.parametrize("dtype", [F16, BF16])
def test_scores_mixed_lengths(dtype, mode):
    """256 <-> 576 tokens through pair_dirs and aas_matrix; then one group with a 129-row query and self item against
    256-row cross items, and the reverse."""
    dev = _cuda()
    ops = _ops()
    imgs = _images((2, 8, 576, 64), dtype, dev, alphas=(1.0, 0.9, 0.7))
    big, small = imgs, _resampled(imgs, 256)
    model = _Model([small[0], big[1]])
    got = ops.pair_dirs(*small[0], *big[1], mode)
    _check_scores("256<->576 pair_dirs", dtype, mode, [got[0], got[1]], [model.dir(0, 1, mode), model.dir(1, 0, mode)],
                  [_t1_dir(model.images, 0, 1, mode), _t1_dir(model.images, 1, 0, mode)])
    q, ks, vs = _stack(small, "sd")
    _, k, v = _stack(big, "sd")
    mat = ops.aas_matrix(q, ks, vs, k, v, mode).reshape(-1)
    m2 = _Model(small + big)
    n = len(small)
    _check_scores("256x576 matrix", dtype, mode, mat, [m2.dir(i, n + j, mode) for i in range(n) for j in range(n)],
                  [_t1_dir(m2.images, i, n + j, mode) for i in range(n) for j in range(n)])

    for rows, cols in ((129, 256), (256, 129)):
        a, b = _resampled(imgs, rows), _resampled(imgs, cols)
        q, ks, vs = _stack(a, "sd")
        _, k, v = _stack(b, "sd")
        dirs = ops.aas_groups(q, ks, vs, k, v, [1], [0, 3], [0, 1, 2], mode)
        m3 = _Model(a + b)
        _check_scores(f"group self={rows} cross={cols}", dtype, mode, dirs, [m3.dir(1, 3 + j, mode) for j in range(3)],
                      [_t1_dir(m3.images, 1, 3 + j, mode) for j in range(3)])


def _sum_bound(q, D):
    """Relative bound of K1's fp32 sum of squares: a row's D_PAD / 4 FMAs per thread lane, the pair of lanes, the warp
    shuffle tree, the eight epilogue warps, the q tiles one after another, and the final rounding."""
    B, H, Sq = q.shape[:3]
    depth = (-(-D // 16) + 1) // 2 * 8 + 1 + 5 + 3 + B * H * -(-Sq // 128) + 2
    return depth * 2.0 ** -24


@pytest.mark.parametrize("dtype", [F16, BF16])
@pytest.mark.parametrize("case", ["dino", "sd15_up0", "ip_adapter", "mixed"])
def test_mse_score_is_the_mse_of_the_stored_outputs(case, dtype):
    """The MSE epilogue rounds the cross and self outputs exactly as the store form does, so dir(i -> j) must be the
    float64 MSE of attn_fwd(q_i, k_j, v_j) against attn_fwd(q_i, k_i, v_i) up to the fp32 summation; no model
    involved."""
    dev = _cuda()
    ops = _ops()
    if case == "mixed":
        imgs = _images((2, 8, 576, 64), dtype, dev, alphas=(1.0, 0.9))
        A, B = _resampled(imgs, 129)[0], imgs[1]
    else:
        dims, layout, kv_tokens = SCORE_SHAPES[case]
        A, B = _images(dims, dtype, dev, layout=layout, kv_tokens=kv_tokens)
    for (qi, ki, vi), (_, kj, vj) in ((A, B), (B, A)):
        x, y = ops.attn_fwd(qi, kj, vj).double(), ops.attn_fwd(qi, ki, vi).double()
        ref = float((x - y).square().mean())
        got = float(ops.aas_groups(qi[None], ki[None], vi[None], kj[None], vj[None], [0], [0, 1], [0], "mse")[0])
        bound = _sum_bound(qi, qi.shape[-1])
        print(f"MSEFREE {case} {str(dtype)[6:]}: rel {abs(got - ref) / ref:.2e} bound {bound:.2e}")
        assert abs(got - ref) <= bound * ref
