#!/usr/bin/env python
"""Timing of the matrix K5 backward (ops.aas_matrix_bwd: each row's self terms folded into one attention backward)
against the grouped backward of the same row-major list (ops.aas_groups_bwd: one self term per entry), alternating in
one process after warm-up, with the outputs compared.

One shared cache of N images is both the rows and the columns (a retrieval / contrastive loss over a batch), so dk_self
is dk.  Work: the grouped list runs 2 N^2 attention backwards, the fold N^2 + N; the recompute, partials and
coefficients are the same.  Times are CUDA events around --iters back-to-back calls into preallocated fp32 gradients, one
synchronise per timed window; the median over --rounds alternating rounds is reported.  Both paths cut their work into
calls under ops.GROUPS_BWD_WORKSPACE_CAP (1 GiB) as a user's call would.
usage: python tools/perf_matrix_grad.py [--iters 3] [--rounds 3] [--json out.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# name: (B, H, S, D, layout, N)
CASES = (("sd15_up0", (2, 8, 256, 160, "sd", 16)), ("sd15_up0", (2, 8, 256, 160, "sd", 64)),
         ("sdxl", (2, 20, 1024, 64, "sd", 16)), ("dit", (2, 16, 256, 72, "dit", 64)))


def _timed(fn, iters):
    import torch

    from diffsim_b200 import ops

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
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("perf_matrix_grad.py needs a CUDA device")
    from diffsim_b200 import ops, synth

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else torch.cuda.get_device_name(), "iters": a.iters, "rounds": a.rounds, "rows": []}
    print("gpu, power limit, SM clock, max SM clock:", res["gpu"], flush=True)
    for name, (B, H, S, D, layout, n) in CASES:
        m = synth.SynthModel(B, H, S, D, seed=2334)
        g = torch.Generator().manual_seed(7)
        base = m.new_base(g)
        imgs = [m.image(base, 1.0 - 0.01 * i, torch.float16, layout, g) for i in range(n)]
        q, k, v = synth.stack_cache(imgs, "cuda")
        d = torch.randn(n, n, generator=g).cuda()
        gq, go, kv = list(range(n)), [r * n for r in range(n + 1)], [c for _ in range(n) for c in range(n)]
        gm = [torch.zeros(t.shape, dtype=torch.float32, device="cuda") for t in (q, k, v)]
        gg = [torch.zeros_like(t) for t in gm]
        matrix = lambda: ops.aas_matrix_bwd(q, k, v, k, v, d, grads=(gm[0], gm[1], gm[2], gm[1], gm[2]))  # noqa: E731
        grouped = lambda: ops.aas_groups_bwd(q, k, v, k, v, gq, go, kv, d.reshape(-1),  # noqa: E731
                                             grads=(gg[0], gg[1], gg[2], gg[1], gg[2]))
        for t in gm + gg:
            t.zero_()
        matrix()
        grouped()   # warm-up, and one call of each into zeroed buffers for the comparison
        diff = [float((x - y).norm() / y.norm()) for x, y in zip(gm, gg)]
        tm, tg = [], []
        for _ in range(a.rounds):
            ms, lm = _timed(matrix, a.iters)
            tm.append(ms)
            ms, lg = _timed(grouped, a.iters)
            tg.append(ms)
        m_ms, g_ms = statistics.median(tm), statistics.median(tg)
        row = {"shape": name, "bhsd": [B, H, S, D], "layout": layout, "n": n, "entries": n * n,
               "matrix_ms": m_ms, "matrix_launches": lm, "grouped_ms": g_ms, "grouped_launches": lg,
               "speedup": g_ms / m_ms, "rel_diff_dq_dk_dv": diff, "matrix_ms_all": tm, "grouped_ms_all": tg}
        res["rows"].append(row)
        print(f"{name:9s} N={n:3d} entries {n * n:5d} | fold {m_ms:9.2f} ms {lm:5d} launches | grouped {g_ms:9.2f} ms "
              f"{lg:5d} launches | {row['speedup']:.2f}x | rel diff dq dk dv {' '.join(f'{x:.1e}' for x in diff)}",
              flush=True)
        del q, k, v, gm, gg, imgs
        torch.cuda.empty_cache()
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
