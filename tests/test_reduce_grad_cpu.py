"""ds_pair_reduce_bwd without a GPU: argument checks come before the device and name the entry point, the workspace
query needs no device, the call fails loudly rather than computing on the host, and the float64 closed form of
oracle.reduce_grad_oracle is the gradient float64 torch autograd gives, while wrong forms of it are caught."""
import pytest
import torch

from diffsim_b200 import _native as N
from oracle import reduce_grad_oracle as R

P, E = 2, 64


def _call(lib, buf, **kw):
    a = dict(x=buf[0], y=buf[1], n_pairs=P, E=E, x_stride=E, y_stride=E, dtype=N.DS_F16, mode=N.DS_SIM_COSINE,
             d_out=buf[2], dx=buf[3], dx_stride=E, dy=buf[4], dy_stride=E, ws=buf[5], ws_bytes=1 << 16)
    a.update(kw)
    return lib.ds_pair_reduce_bwd(a["x"], a["y"], a["n_pairs"], a["E"], a["x_stride"], a["y_stride"], a["dtype"],
                                  a["mode"], a["d_out"], a["dx"], a["dx_stride"], a["dy"], a["dy_stride"], a["ws"],
                                  a["ws_bytes"], None)


def _bufs():
    keep = [torch.zeros(P * E * 2 + 64, dtype=torch.float32) for _ in range(5)] + [torch.zeros(1 << 14)]
    return keep, [t.data_ptr() + (-t.data_ptr()) % 16 for t in keep]   # 16-byte aligned bases


@pytest.mark.parametrize("bad", [
    dict(x=None), dict(y=None), dict(d_out=None),
    dict(E=0), dict(n_pairs=-1),
    dict(dtype=9), dict(mode=7),
    dict(x="+1"),                      # not element-aligned
    dict(dx="+2"),                     # fp32 gradient not 4-byte aligned
    dict(x_stride=E - 8),              # input row stride below E
    dict(dy_stride=E - 1),             # gradient row stride below E
    dict(ws=None, ws_bytes=0),         # no workspace for the statistics pass
])
def test_arguments_are_checked_before_the_device(bad):
    lib = N.load()
    keep, al = _bufs()
    names = ["x", "y", "d_out", "dx", "dy"]
    for k, v in list(bad.items()):
        if isinstance(v, str):
            bad[k] = al[names.index(k)] + int(v)
    code = N.DS_ERR_WORKSPACE if "ws" in bad else N.DS_ERR_INVALID
    assert _call(lib, al, **bad) == code
    assert N.last_error().startswith("ds_pair_reduce_bwd:")


def test_nothing_asked_is_ok_without_a_device():
    lib = N.load()
    keep, al = _bufs()
    assert _call(lib, al, dx=None, dy=None) == N.DS_OK
    assert _call(lib, al, n_pairs=0) == N.DS_OK


def test_workspace_query_needs_no_device():
    lib = N.load()
    # up to 64 chunk records of 16 floats per row, and a counter per row
    assert lib.ds_pair_reduce_bwd_workspace_bytes(256, 655360) >= 256 * 64 * 16 * 4 + 256 * 4
    assert lib.ds_pair_reduce_bwd_workspace_bytes(0, 655360) > 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour on a machine without a GPU")
def test_no_gpu_means_loud_failure():
    lib = N.load()
    keep, al = _bufs()
    for mode in (N.DS_SIM_COSINE, N.DS_SIM_MSE, N.DS_SIM_MINMAX_COSINE):
        assert _call(lib, al, mode=mode) == N.DS_ERR_CUDA
    assert all((t == 0).all() for t in keep)   # nothing was computed on the host
    from diffsim_b200 import ops

    x = torch.randn(2, 8).half()
    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.pair_reduce_bwd(x, x, torch.ones(2))
    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.pair_reduce(x.requires_grad_(), x)


def _cases():
    """(name, x, y): ties, zero rows, near-zero rows, constant rows and ragged E, as 16-bit and float64 rows."""
    g = torch.Generator().manual_seed(5)
    out = []
    for E_ in (1, 7, 37, 1000):
        out.append((f"random_E{E_}", torch.randn(3, E_, generator=g).half(), torch.randn(3, E_, generator=g).half()))
    q = (torch.randn(4, 300, generator=g) * 2).round().clamp(-3, 3).half()   # min and max tied many times
    out.append(("ties", q, (torch.randn(4, 300, generator=g) * 2).round().clamp(-2, 4).half()))
    zx, zy = torch.randn(3, 50, generator=g).half(), torch.randn(3, 50, generator=g).half()
    zx[0], zy[1] = 0, 0
    zy[0] = 0
    out.append(("zero_rows", zx, zy))
    nz = torch.randn(2, 40, generator=g, dtype=torch.float64)   # |x| ~ 5e-9, below the 1e-8 clamp
    out.append(("near_zero_rows", nz * 8e-10, 0.8 * nz + 0.6 * torch.randn(2, 40, generator=g, dtype=torch.float64)))
    c = torch.randn(3, 20, generator=g).half()
    c[1] = 0.5
    out.append(("constant_row", c, torch.randn(3, 20, generator=g).half()))
    return out


@pytest.mark.parametrize("mode", ["cosine", "mse", "minmax_cosine"])
def test_closed_form_is_float64_autograd(mode):
    for name, x, y in _cases():
        g = torch.linspace(-1.5, 2.0, x.shape[0])
        floors = R.cross_term_norms(x, y, g, mode)
        for got, ref, fl in zip(R.pair_reduce_grads(x, y, g, mode), R.autograd_grads(x, y, g, mode), floors):
            assert torch.equal(got.isnan(), ref.isnan()), name   # NaN exactly in the rows torch gives NaN
            err = R.row_errors(got, ref, fl)
            ok = err[~err.isnan()]
            assert (ok < 1e-12).all(), (name, mode, err)
            if mode == "minmax_cosine" and name == "constant_row":
                assert got[1].isnan().all() and not got[0].isnan().any() and not got[2].isnan().any()


def _mutant_error(mode, x, y, **mutation):
    g = torch.tensor([1.0, -0.7, 0.4, 2.0])[: x.shape[0]]
    ref = R.autograd_grads(x, y, g, mode)
    got = R._grads(x, y, g, mode, **mutation)
    floors = R.cross_term_norms(x, y, g, mode)
    return max(float(R.row_errors(a, b, f).nan_to_num(0).max()) for a, b, f in zip(got, ref, floors))


def test_mutants_exceed_the_gpu_tolerance():
    cases = {name: (x, y) for name, x, y in _cases()}
    errs = {
        "ties not split": _mutant_error("minmax_cosine", *cases["ties"], split_ties=False),
        "min/max path dropped": _mutant_error("minmax_cosine", *cases["random_E1000"], minmax_terms=False),
        "clamped norm for |x|": _mutant_error("cosine", *cases["near_zero_rows"], unclamped=False),
    }
    print({k: f"{v:.2e}" for k, v in errs.items()})
    for name, err in errs.items():
        assert err > 10 * R.ROW_TOL, name
