#!/usr/bin/env python
"""Timing of the K5 backward: forward + backward of diffsim.aas_score over a batch of image pairs, against torch autograd
of the reference's own fp16 torch calls (oracle.reference_pair_score: SDPA + F.cosine_similarity) on the same GPU.

Per pair the backward covers four attentions (cross and self, both directions); algorithmic work 10 B H S^2 D flops
each.  Times are CUDA events around the backward calls (after warm-up), one synchronise per timed pass.
usage: python tools/perf_grad.py [--pairs 8] [--iters 10] [--json out.json]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {  # (B, H, S, D, layout): the hooked layers of the three scorers
    "sd15_up0": (2, 8, 256, 160, "sd"),
    "sdxl": (2, 20, 1024, 64, "sd"),
    "dit": (2, 16, 256, 72, "dit"),
}


def _time(fwd, iters, warmup=3):
    """(forward ms, backward ms) per pass: fwd() builds the graph and returns the loss."""
    import torch

    for _ in range(warmup):
        fwd().backward()
    torch.cuda.synchronize()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    f_ms = b_ms = 0.0
    for _ in range(iters):
        e[0].record()
        loss = fwd()
        e[1].record()
        loss.backward()
        e[2].record()
        torch.cuda.synchronize()
        f_ms += e[0].elapsed_time(e[1])
        b_ms += e[1].elapsed_time(e[2])
    return f_ms / iters, b_ms / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=8)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("perf_grad.py needs a CUDA device")
    from diffsim_b200 import synth
    from diffsim_b200.diffsim import aas_score
    from oracle.aas_oracle import reference_pair_score

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": gpu[0] if gpu else torch.cuda.get_device_name(), "pairs": a.pairs, "shapes": {}}
    for name, (B, H, S, D, layout) in SHAPES.items():
        m = synth.SynthModel(B, H, S, D, seed=2334)
        g = torch.Generator().manual_seed(7)
        base = m.new_base(g)
        imgs = [[t.cuda().requires_grad_(True) for t in m.image(base, 1.0 - 0.05 * i, torch.float16, layout, g)]
                for i in range(a.pairs + 1)]
        pairs = [(imgs[0], imgs[i + 1]) for i in range(a.pairs)]
        ours = _time(lambda: sum(aas_score(tuple(x), tuple(y), match_reference_dtype=False).sum() for x, y in pairs), a.iters)
        ref = _time(lambda: sum(reference_pair_score(*x, *y).float().sum() for x, y in pairs), a.iters)
        flops = 4 * 10 * B * H * S * S * D * a.pairs
        r = {"shape": [B, H, S, D], "layout": layout,
             "k5": {"fwd_ms": ours[0], "bwd_ms": ours[1], "bwd_tflops": flops / ours[1] / 1e9},
             "torch_autograd_fp16": {"fwd_ms": ref[0], "bwd_ms": ref[1], "bwd_tflops": flops / ref[1] / 1e9},
             "bwd_speedup_vs_torch": ref[1] / ours[1]}
        res["shapes"][name] = r
        print(f"{name} {(B, H, S, D)}: K5 fwd {ours[0]:.3f} ms bwd {ours[1]:.3f} ms ({r['k5']['bwd_tflops']:.1f} TFLOP/s) | "
              f"torch fwd {ref[0]:.3f} ms bwd {ref[1]:.3f} ms ({r['torch_autograd_fp16']['bwd_tflops']:.1f} TFLOP/s) | "
              f"bwd speed-up {r['bwd_speedup_vs_torch']:.2f}x", flush=True)
    print(json.dumps(res))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
