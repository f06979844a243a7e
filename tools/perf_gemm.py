#!/usr/bin/env python
"""A/B of the GEMM kernels behind K3 / K4 (ds_debug_set_gemm_variant: 0 = 1-CTA 128x256, 2 = CTA pairs 256x256):
how far apart their similarity matrices are, then throughput on the QKV-projection and similarity-matrix shapes.
tests/test_gpu_qkv.py checks that both give bitwise the same projections."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from diffsim_b200 import ops, synth, _native as N

lib = N.load()


def timeit(fn, iters=10, warmup=3):
    for _ in range(warmup): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


# ---- similarity matrix: pair kernel vs 1-CTA kernel
g = torch.Generator(device="cuda").manual_seed(1)
for n, L in ((600, 4096), (1000, 2048), (2032, 1024)):
    f = (torch.randn(n, L, generator=g, device="cuda") * 0.8 + 0.1).half()
    f2 = f.clone()
    res = {}
    for var in (0, 2):
        lib.ds_debug_set_gemm_variant(var)
        res[var] = (ops.simmat(f, None, "cosine"), ops.simmat(f, f2, "cosine"))
    d_self = (res[0][0] - res[2][0]).abs().max().item()
    d_full = (res[0][1] - res[2][1]).abs().max().item()
    d_sf = (res[2][0] - res[2][1]).abs().max().item()
    print(f"[check simmat N={n} L={L}] |1cta-pair| self {d_self:.1e} full {d_full:.1e}; pair |self-full| {d_sf:.1e}; "
          f"symmetric={torch.equal(res[2][0], res[2][0].t())} diag {float((res[2][0].diagonal() - 1).abs().max()):.1e}", flush=True)

# ---- throughput
for n_img in (96, 768):
    hid, w = synth.device_hidden(2, 8, 256, 160, n_img, torch.float16, "cuda")
    outs = [torch.empty(n_img, 2, 256, 1280, dtype=torch.float16, device="cuda") for _ in range(3)]
    fl = 2 * n_img * 512 * 1280 * 3840
    line = f"[K4 {n_img} images]"
    for var in (0, 2, 0, 2):
        lib.ds_debug_set_gemm_variant(var)
        ms = timeit(lambda: ops.qkv_project(hid, w, None, 3, out=outs))
        line += f" variant {var}: {ms:.3f} ms {fl / ms / 1e9:.0f} TFLOP/s |"
    h2 = hid.view(-1, 1280)
    ms = timeit(lambda: h2 @ w.t())
    print(line + f" torch {ms:.3f} ms {fl / ms / 1e9:.0f} TFLOP/s", flush=True)
    del hid, outs, h2
for n, L in ((2032, 65536), (2032, 655360)):
    f = torch.empty(n, L, dtype=torch.float16, device="cuda")
    for i in range(0, n, 127):
        f[i:i + 127] = torch.randn(min(127, n - i), L, device="cuda").half()
    line = f"[K3 N={n} L={L} self]"
    for var in (0, 2, 0, 2):
        lib.ds_debug_set_gemm_variant(var)
        ms = timeit(lambda: ops.simmat(f, None, "cosine"), iters=5, warmup=2)
        line += f" variant {var}: {ms:.3f} ms |"
    print(line, flush=True)
    del f
lib.ds_debug_set_gemm_variant(-1)
