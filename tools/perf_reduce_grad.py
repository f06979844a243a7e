#!/usr/bin/env python
"""Timing of the K2 backward (ops.pair_reduce_bwd) against torch's own autograd of the same expressions on the same
tensors, alternating in one process after warm-up, and against a device copy measured in the same process.

256 row pairs of 655 360 fp16 elements (a batch of SD-1.5 up-block feature maps), all three modes.  Executed bytes per
row pair: the statistics pass reads x and y (4 E), the gradient pass reads them again and writes fp32 dx and dy (12 E):
16 E = 10.5 MB for cosine and min-max; mse has no statistics pass: 12 E = 7.9 MB.  The working set (2.7 GB) is far
larger than the 126 MB L2.  Torch's path is torch.autograd.grad of F.cosine_similarity / the row mean of (x - y)^2 /
min-max normalisation + cosine over dim 1 (fp16 gradients, the graph built once and retained).  The copy rate is
dst.copy_(src) of 1 GiB, counted as read + write.  Times are CUDA events around --iters back-to-back calls, one
synchronise per window; the median over --rounds alternating rounds is reported.
usage: python tools/perf_reduce_grad.py [--iters 10] [--rounds 5] [--out profiles/reduce_grad_b200.txt]"""
import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

P, E = 256, 655360


def _timed(fn, iters):
    import torch

    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def _torch_score(x, y, mode):
    import torch.nn.functional as F

    if mode == "cosine":
        return F.cosine_similarity(x, y, dim=1)
    if mode == "mse":
        return ((x - y) ** 2).mean(1)

    def mm(t):
        lo, hi = t.amin(1, keepdim=True), t.amax(1, keepdim=True)
        return (t - lo) / (hi - lo)

    return F.cosine_similarity(mm(x), mm(y), dim=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("perf_reduce_grad.py needs a CUDA device")
    from diffsim_b200 import ops

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    lines = [f"# tools/perf_reduce_grad.py: K2 backward vs torch autograd of the same expressions, {P} x {E} fp16, "
             f"{a.rounds} alternating rounds x {a.iters} calls, median, CUDA events",
             "gpu, power limit, SM clock, max SM clock: " + (smi[0] if smi else torch.cuda.get_device_name())]
    lines.append("# rel diff: our fp32 gradients against torch's fp16 ones, whose per-element values (~1e-6 on rows of "
                 "655 360) fall in fp16's subnormal range; tests/test_gpu_reduce_grad.py checks ours against float64")
    print("\n".join(lines[-2:]), flush=True)

    src = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    copy = lambda: dst.copy_(src)  # noqa: E731
    copy()
    copy_ms = statistics.median(_timed(copy, a.iters) for _ in range(a.rounds))
    copy_gbs = 2 * src.numel() / copy_ms / 1e6
    lines.append(f"device copy 1 GiB: {copy_ms:.3f} ms, {copy_gbs:.0f} GB/s (read + write)")
    print(lines[-1], flush=True)
    del src, dst

    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(P, E, device="cuda", generator=g).half()
    y = (0.6 * x.float() + 0.8 * torch.randn(P, E, device="cuda", generator=g)).half()
    d = torch.randn(P, device="cuda", generator=g)
    for mode in ("cosine", "mse", "minmax_cosine"):
        nbytes = P * E * (12 if mode == "mse" else 16)
        ours = lambda: ops.pair_reduce_bwd(x, y, d, mode)  # noqa: E731
        xl, yl = x.detach().requires_grad_(True), y.detach().requires_grad_(True)
        out = _torch_score(xl, yl, mode)
        ref = lambda: torch.autograd.grad(out, (xl, yl), d, retain_graph=True)  # noqa: E731
        got, want = ours(), ref()   # warm-up, and the outputs compared
        diff = [float((u.double() - w.double()).norm() / w.double().norm()) for u, w in zip(got, want)]
        del got, want
        t_ours, t_ref = [], []
        for _ in range(a.rounds):
            t_ours.append(_timed(ours, a.iters))
            t_ref.append(_timed(ref, a.iters))
        mo, mr = statistics.median(t_ours), statistics.median(t_ref)
        gbs = nbytes / mo / 1e6
        lines.append(f"{mode:14s} K2 bwd {mo:8.3f} ms  {gbs:6.0f} GB/s = {100 * gbs / copy_gbs:5.1f}% of copy "
                     f"({nbytes / P / 1e6:.1f} MB per row pair) | torch autograd {mr:8.3f} ms | {mr / mo:5.2f}x | "
                     f"rel diff dx dy vs torch fp16 {diff[0]:.1e} {diff[1]:.1e}")
        print(lines[-1], flush=True)
        del out, xl, yl
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
