#!/usr/bin/env python
"""Throughput of the Aligned Attention Score between images of different token counts, beside the equal-length case of
the same run: the grouped forward (ops.aas_groups, every query image against every gallery image), the all-pairs matrix
(ops.aas_matrix) and its backward (ops.aas_matrix_bwd, both gradient families).

Directions per shape: a->b (query images of S_a tokens, gallery of S_b), b->a, and a->a (equal lengths, the reference
point).  Work is counted per item with its own kv length: a directional attention of Sq query rows over Skv kv rows is
4 B H Sq Skv D flops (ds_attn.cu), an attention backward 10 B H Sq Skv D (ds_attn_bwd.cu).  Forward: one cross item per
entry (Skv = the gallery's S) and one self item per query image (Skv = its own S).  Backward: the recompute forward
(every cross output and every row's self output) plus one attention backward per cross term and per row's folded self
term.  Times are CUDA events around --iters back-to-back calls after one warm-up call, one synchronise per window; the
card's name and power limit are read in the same run.
usage: python tools/perf_mixed_length.py [--iters 10] [--json out.json]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# name: (B, H, D, S_a, S_b): SD-1.5 up_blocks[0] at 512^2 vs 768^2; SDXL up_blocks at 1024^2 (1024 / 4096 tokens)
SHAPES = {"sd15_up0": (2, 8, 160, 256, 576), "sdxl_d64": (2, 10, 64, 1024, 4096)}
N_QUERY, N_GALLERY = 8, 16


def _timed(fn, iters):
    import torch

    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def _cache(n, B, H, S, D, g):
    import torch

    x = torch.randn(n, 3, B, S, H, D, generator=g).half().cuda()
    return tuple(x[:, i].contiguous().permute(0, 1, 3, 2, 4) for i in range(3))   # head-split views of (n, B, S, H*D)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("perf_mixed_length.py needs a CUDA device")
    from diffsim_b200 import ops

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else torch.cuda.get_device_name(), "iters": a.iters, "rows": []}
    print("gpu, power limit, SM clock, max SM clock:", res["gpu"], flush=True)
    for name, (B, H, D, Sa, Sb) in SHAPES.items():
        g = torch.Generator().manual_seed(3)
        caches = {Sa: _cache(max(N_QUERY, N_GALLERY), B, H, Sa, D, g), Sb: _cache(max(N_QUERY, N_GALLERY), B, H, Sb, D, g)}
        for Sq, Sk in ((Sa, Sb), (Sb, Sa), (Sa, Sa)):
            q, ks, vs = (t[:N_QUERY] for t in caches[Sq])
            _, k, v = (t[:N_GALLERY] for t in caches[Sk])
            nr, nc = N_QUERY, N_GALLERY
            gq, go = list(range(nr)), [r * nc for r in range(nr + 1)]
            kv = list(range(nc)) * nr
            attn = lambda skv: 4.0 * B * H * Sq * skv * D   # noqa: E731
            fwd_flops = nr * nc * attn(Sk) + nr * attn(Sq)
            bwd_flops = fwd_flops + 2.5 * fwd_flops          # recompute + one backward (10/4 of its forward) per term
            d = torch.randn(nr, nc, generator=g).cuda()
            grads = [torch.zeros(t.shape, dtype=torch.float32, device="cuda") for t in (q, ks, vs, k, v)]
            runs = {
                "groups": (lambda: ops.aas_groups(q, ks, vs, k, v, gq, go, kv, "cosine"), fwd_flops),
                "matrix": (lambda: ops.aas_matrix(q, ks, vs, k, v, "cosine"), fwd_flops),
                "matrix_bwd": (lambda: ops.aas_matrix_bwd(q, ks, vs, k, v, d, "cosine", grads=grads), bwd_flops),
            }
            for op, (fn, flops) in runs.items():
                ms = _timed(fn, a.iters)
                row = {"shape": name, "bhd": [B, H, D], "S_q": Sq, "S_self": Sq, "S_cross": Sk, "op": op,
                       "rows": nr, "cols": nc, "ms": ms, "tflops": flops / ms / 1e9,
                       "kind": "equal" if Sq == Sk else "mixed"}
                res["rows"].append(row)
                print(f"{name:9s} S_q=S_self={Sq:5d} S_cross={Sk:5d} {row['kind']:5s} {op:10s} {nr}x{nc}: "
                      f"{ms:9.3f} ms {row['tflops']:7.1f} TFLOP/s", flush=True)
            del runs, grads
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
