#!/usr/bin/env python
"""Throughput of the QKV-projection backward (K4, ds_qkv_project_bwd): dX = dY W and dW = dY^T X timed apart with CUDA
events, against torch's cuBLAS backward of F.linear (dY W, dY^T X on the same tensors, dY packed) in the same process.
TFLOP/s from 2 * rows * C_in * n_out per product.  Prints one line per shape and product, and the whole as JSON last.
Run it as `nvidia-smi --query-gpu=name,power.limit --format=csv; python tools/perf_qkv_bwd.py` so that the card and its
power limit are recorded with the numbers."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from diffsim_b200 import ops

SHAPES = [
    # name, rows, C_in, outputs (3: q / k / v of C_in columns each; 1: DiT's packed 3C), bias
    ("sd15_up0_96img", 96 * 2 * 256, 1280, 3, False),
    ("train_2img_c320_4096tok", 2 * 4096, 320, 3, False),
    ("train_2img_c1280_256tok", 2 * 256, 1280, 3, False),
    ("ditxl2_96img_packed_bias", 96 * 256, 1152, 1, True),
]


def timeit(fn, iters=20, warmup=5):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    if not torch.cuda.is_available():
        raise SystemExit("perf_qkv_bwd.py needs a CUDA device")
    dev, dt = "cuda", torch.float16
    g = torch.Generator(device=dev).manual_seed(0)
    results = []
    for name, rows, c_in, n_t, bias in SHAPES:
        n_out = 3 * c_in
        x = torch.randn(rows, c_in, generator=g, device=dev).to(dt)
        w = (torch.randn(n_out, c_in, generator=g, device=dev) / c_in ** 0.5).to(dt)
        dys = [torch.randn(rows, n_out // n_t, generator=g, device=dev).to(dt) for _ in range(n_t)]
        dy = torch.cat(dys, dim=1)
        flops = 2 * rows * c_in * n_out
        rec = {"shape": name, "rows": rows, "c_in": c_in, "n_out": n_out}
        for prod, k4, ref in (("dX", lambda: ops.qkv_project_bwd(x, w, dys, True, False, bias), lambda: dy @ w),
                              ("dW", lambda: ops.qkv_project_bwd(x, w, dys, False, True, False), lambda: dy.t() @ x)):
            ms_k4, ms_ref = timeit(k4), timeit(ref)
            rec[prod] = {"k4_ms": round(ms_k4, 4), "k4_tflops": round(flops / ms_k4 / 1e9, 1),
                         "cublas_ms": round(ms_ref, 4), "cublas_tflops": round(flops / ms_ref / 1e9, 1)}
            print(f"[{name} {prod}{' + db' if prod == 'dX' and bias else ''}] K4 {ms_k4:.3f} ms "
                  f"{rec[prod]['k4_tflops']:.0f} TFLOP/s | cuBLAS {ms_ref:.3f} ms {rec[prod]['cublas_tflops']:.0f} TFLOP/s",
                  flush=True)
        results.append(rec)
        del x, w, dys, dy
    print(json.dumps({"device": torch.cuda.get_device_name(), "results": results}))


if __name__ == "__main__":
    main()
