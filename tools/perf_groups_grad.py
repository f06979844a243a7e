#!/usr/bin/env python
"""Timing of the grouped K5 backward (ops.aas_pairs_bwd / aas_triplets_bwd: one ds_aas_*_bwd call per list) against the
per-entry loop it is bitwise equal to (ops.aas_dir_bwd once per entry, list order), in the same process after warm-up.

Shapes are those of tools/perf_grad.py; lists are P pairs and T triplets drawn from a cache of 16 images (3 x 16 images
exceed the L2 at every shape but DiT, so K/V are not all L2-resident).  Work per entry: two attention backwards,
20 B H Sq Skv D algorithmic flops.  Times are CUDA events around --iters back-to-back calls into preallocated fp32
gradients, one synchronise per timed window.
usage: python tools/perf_groups_grad.py [--iters 5] [--json out.json]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.perf_grad import SHAPES  # noqa: E402

N_IMAGES = 16
LISTS = (("pairs", 1), ("pairs", 8), ("pairs", 64), ("triplets", 8), ("triplets", 64))


def _entries(kind, idx):
    """(query image, kv image, index of the score) of every entry, in list order (ds_aas_pairs / triplets work lists)."""
    if kind == "pairs":
        return [e for p, (a, b) in enumerate(idx) for e in ((a, b, p), (b, a, p))]
    return [e for t, (r, l, rt) in enumerate(idx) for e in ((r, l, (0, t)), (r, rt, (1, t)), (l, r, (0, t)), (rt, r, (1, t)))]


def _timed(fn, iters):
    import torch

    from diffsim_b200 import ops

    fn()
    torch.cuda.synchronize()
    n0 = ops.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, (ops.LAUNCHES - n0) // iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("perf_groups_grad.py needs a CUDA device")
    from diffsim_b200 import ops, synth

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else torch.cuda.get_device_name(), "iters": a.iters, "rows": []}
    print("gpu, power limit, SM clock, max SM clock:", res["gpu"], flush=True)
    for name, (B, H, S, D, layout) in SHAPES.items():
        m = synth.SynthModel(B, H, S, D, seed=2334)
        g = torch.Generator().manual_seed(7)
        base = m.new_base(g)
        imgs = [m.image(base, 1.0 - 0.03 * i, torch.float16, layout, g) for i in range(N_IMAGES)]
        q, k, v = synth.stack_cache(imgs, "cuda")
        grads = [torch.zeros(t.shape, dtype=torch.float32, device="cuda") for t in (q, k, v)]
        for kind, n in LISTS:
            r = torch.Generator().manual_seed(n)
            idx = [torch.randperm(N_IMAGES, generator=r)[: 2 if kind == "pairs" else 3].tolist() for _ in range(n)]
            d = [torch.randn(n, generator=r).cuda() for _ in range(2)]
            if kind == "pairs":
                grouped = lambda: ops.aas_pairs_bwd(q, k, v, idx, d[0], grads=grads)  # noqa: E731
                d_dir = [(d[0][p] * 0.5).reshape(1) for _, _, p in _entries(kind, idx)]
            else:
                grouped = lambda: ops.aas_triplets_bwd(q, k, v, idx, d[0], d[1], grads=grads)  # noqa: E731
                d_dir = [(d[w][t] * 0.5).reshape(1) for _, _, (w, t) in _entries(kind, idx)]
            ents = [(i, j, dd) for (i, j, _), dd in zip(_entries(kind, idx), d_dir)]
            dq, dk, dv = grads

            def loop():
                for i, j, dd in ents:
                    ops.aas_dir_bwd(q[i], k[i], v[i], k[j], v[j], dd, grads=(dq[i], dk[i], dv[i], dk[j], dv[j]))

            g_ms, g_l = _timed(grouped, a.iters)
            l_ms, l_l = _timed(loop, a.iters)
            flops = 20.0 * B * H * S * S * D * len(ents)
            row = {"shape": name, "bhsd": [B, H, S, D], "list": f"{kind}={n}", "entries": len(ents),
                   "grouped_ms": g_ms, "grouped_launches": g_l, "grouped_tflops": flops / g_ms / 1e9,
                   "loop_ms": l_ms, "loop_launches": l_l, "loop_tflops": flops / l_ms / 1e9, "speedup": l_ms / g_ms}
            res["rows"].append(row)
            print(f"{name:9s} {kind}={n:<3d} entries {len(ents):4d} | grouped {g_ms:8.3f} ms {g_l:4d} launches "
                  f"{row['grouped_tflops']:6.1f} TFLOP/s | loop {l_ms:8.3f} ms {l_l:5d} launches {row['loop_tflops']:6.1f} "
                  f"TFLOP/s | {row['speedup']:.2f}x", flush=True)
            del grouped
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
