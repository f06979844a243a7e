#!/usr/bin/env python
"""Timing of the sharded all-pairs matrix backward (scoring.aas_matrix_sharded(..., gather_to_all=False)).

Default mode, one GPU: the cost of the decomposition.  For W emulated shards of one shared cache of N images, rank w's
backward is two calls of the matrix backward (scoring._matrix_grad_block): its rows against all N columns
(need_cols=False) and all N rows against its columns (need_rows=False).  The column pass recomputes X for N n_w entries
and Y for all N rows and runs a statistics-only dQ pass on its cross terms, work that one full call does once.  Reported
against one full ops.aas_matrix_bwd (separate self buffers) of the same matrix:
  - sum over the W ranks of both passes / full: the total work of the decomposition;
  - the slowest rank / (full / W): what W GPUs take against a perfect split.
Times are CUDA events around back-to-back calls, one synchronise per window, the median over --rounds alternating
rounds.  The gradients are checked bitwise against the full call.

--world W (W processes, one GPU each, NCCL): the backward wall time per rank at N images (default 256, SD-1.5 up0),
a row-local InfoNCE loss on each rank's row block; CUDA events around loss.backward() after a barrier.  Run it once with
--world 1 on the same box for the strong-scaling baseline.
usage: python tools/perf_matrix_grad_sharded.py [--rounds 3] [--json out.json]
       python tools/perf_matrix_grad_sharded.py --world 2 [--n 256] [--iters 2] [--json out.json]"""
import argparse
import json
import os
import socket
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# name: (B, H, S, D, layout, N)
CASES = (("sd15_up0", (2, 8, 256, 160, "sd", 64)), ("sdxl", (2, 20, 1024, 64, "sd", 16)),
         ("dit", (2, 16, 256, 72, "dit", 64)))
WORLDS = (2, 4, 8)


def _gpu():
    import torch

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return smi[0] if smi else torch.cuda.get_device_name()


def _cache(B, H, S, D, layout, n, dev="cuda"):
    import torch

    from diffsim_b200 import synth

    m = synth.SynthModel(B, H, S, D, seed=2334)
    g = torch.Generator().manual_seed(7)
    base = m.new_base(g)
    imgs = [m.image(base, 1.0 - 0.01 * i, torch.float16, layout, g) for i in range(n)]
    return synth.stack_cache(imgs, dev)


def _timed(fn, iters=1):
    import torch

    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def decomposition(a):
    import torch

    from diffsim_b200 import ops, scoring

    res = {"gpu": _gpu(), "rounds": a.rounds, "rows": []}
    print("gpu, power limit, SM clock, max SM clock:", res["gpu"], flush=True)
    for name, (B, H, S, D, layout, n) in CASES:
        q, k, v = _cache(B, H, S, D, layout, n)
        d = torch.randn(n, n, generator=torch.Generator().manual_seed(3)).cuda()

        def full():
            grads = [torch.zeros(t.shape, dtype=torch.float32, device="cuda") for t in (q, k, v, k, v)]
            return ops.aas_matrix_bwd(q, k, v, k, v, d, grads=grads)

        def rank_pass(world, rank):
            r0, r1 = scoring.row_block(n, rank, world)
            return lambda: scoring._matrix_grad_block(q, k, v, r0, r1, d, "cosine", None)

        ref = full()   # warm-up, and the bitwise check of every rank's gradients
        same = True
        for world in WORLDS:
            for rank in range(world):
                r0, r1 = scoring.row_block(n, rank, world)
                got = rank_pass(world, rank)()
                same &= all(torch.equal(x, y[r0:r1]) for x, y in zip(got, ref))
        del ref, got
        t_full, t_rank = [], {w: [[] for _ in range(w)] for w in WORLDS}
        for _ in range(a.rounds):
            t_full.append(_timed(full))
            for world in WORLDS:
                for rank in range(world):
                    t_rank[world][rank].append(_timed(rank_pass(world, rank)))
        f_ms = statistics.median(t_full)
        print(f"{name:9s} N={n:3d} | full backward {f_ms:8.2f} ms | bitwise per rank: {same}", flush=True)
        row = {"shape": name, "bhsd": [B, H, S, D], "layout": layout, "n": n, "full_ms": f_ms, "full_ms_all": t_full,
               "bitwise": same, "worlds": []}
        for world in WORLDS:
            per = [statistics.median(t) for t in t_rank[world]]
            total, slowest = sum(per), max(per)
            row["worlds"].append({"world": world, "rank_ms": per, "sum_over_full": total / f_ms,
                                  "slowest_over_ideal": slowest / (f_ms / world)})
            print(f"    W={world}: per rank {' '.join(f'{x:.2f}' for x in per)} ms | sum / full {total / f_ms:.3f} | "
                  f"slowest / (full / W) {slowest / (f_ms / world):.3f}", flush=True)
        res["rows"].append(row)
        del q, k, v
        torch.cuda.empty_cache()
    return res


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def loss_of(block, r0, dev):
    """a row-local InfoNCE loss: each row against its own image"""
    import torch

    tgt = torch.arange(r0, r0 + block.shape[0], device=dev)
    return torch.nn.functional.cross_entropy(block / 0.05, tgt, reduction="sum")


def _rank(rank, world, port, n, iters, ret):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist

    from diffsim_b200 import scoring

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        B, H, S, D, layout, _ = CASES[0][1]
        q, k, v = _cache(B, H, S, D, layout, n, dev)
        r0, r1 = scoring.row_block(n, rank, world)
        leaves = [t[r0:r1].detach().clone().requires_grad_() for t in (q, k, v)]
        del q, k, v
        times = []
        for _ in range(iters + 1):   # the first is warm-up
            for t in leaves:
                t.grad = None
            block = scoring.aas_matrix_sharded(scoring.QKVCache(*leaves), gather_to_all=False)
            loss = loss_of(block, r0, dev)
            dist.barrier()
            times.append(_timed(loss.backward))
        ret[rank] = times[1:]
        if world == 1:   # the strong-scaling baseline: one full matrix backward of the same d_Dm on this device
            from diffsim_b200 import ops

            d = torch.autograd.grad(loss_of(block, r0, dev), block)[0]
            full = lambda: ops.aas_matrix_bwd(*leaves, leaves[1], leaves[2], d, grads=[  # noqa: E731
                torch.zeros(t.shape, dtype=torch.float32, device=dev) for t in leaves + leaves[1:]])
            full()
            ret["full"] = [_timed(full) for _ in range(iters)]
    finally:
        dist.barrier()
        dist.destroy_process_group()


def sharded(a):
    import torch
    import torch.multiprocessing as mp

    if torch.cuda.device_count() < a.world:
        sys.exit(f"--world {a.world} needs {a.world} CUDA devices, found {torch.cuda.device_count()}")
    ret = mp.Manager().dict()
    mp.spawn(_rank, args=(a.world, _free_port(), a.n, a.iters, ret), nprocs=a.world, join=True)
    per = [statistics.median(ret[r]) for r in range(a.world)]
    res = {"gpu": _gpu(), "world": a.world, "n": a.n, "shape": CASES[0][0], "iters": a.iters, "rank_backward_ms": per,
           "rank_backward_ms_all": [list(ret[r]) for r in range(a.world)]}
    if "full" in ret:
        res["full_backward_ms"] = statistics.median(ret["full"])
        print(f"one full ops.aas_matrix_bwd of the same matrix: {res['full_backward_ms']:.1f} ms")
    print("gpu, power limit, SM clock, max SM clock:", res["gpu"])
    print(f"{CASES[0][0]} N={a.n} world={a.world}: backward per rank {' '.join(f'{x:.1f}' for x in per)} ms, "
          f"slowest {max(per):.1f} ms", flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--world", type=int, default=0)
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--iters", type=int, default=2)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("perf_matrix_grad_sharded.py needs a CUDA device")
    res = sharded(a) if a.world > 0 else decomposition(a)
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
