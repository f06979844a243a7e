#!/usr/bin/env python
"""Benchmark of the DiffSim AAS scoring hot path on B200 (contract: see the round prompt / DESIGN.md section 6).

    python bench.py --gpus 1 --steps 40 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps 3 --warmup 1        # the reference's CPU path on the host cores
    python bench.py --steps 40 --dump-outputs OUT    # also write the last timed step's results as OUT/<name>.npy

Workload (BASELINE.json configs[1]): NIGHTS-shaped 2AFC triplets (reference, left, right), SD-1.5 512^2,
up_blocks layer 0 => Q/K/V of shape (2,8,256,160) fp16 per image, AAS + cosine.  One step scores T triplets
(2T pairs) from a Q/K/V cache of 3T images that is resident in HBM (24 GB at T=2048: larger than the 126 MB L2,
so every step streams its inputs from HBM).  metric = scored pairs / second, whole job.

The JSON line also carries
  roofline      the fused attention kernel: executed flops (7 directional attentions per triplet x
                4*B*H*S*S*D) / device time of that kernel (CUDA events recorded by the library around the launch,
                on the launching stream) vs the measured BURST bf16 tensor peak of MEASURED_PEAKS.json (frac), with the
                fraction of the sustained peak beside it (frac_sustained)
  torch_cuda_reference   the reference's own lines (4 x F.scaled_dot_product_attention + 2 x F.cosine_similarity,
                diffsim/diffsim.py:177-197) on the SAME GPU: per pair as the reference executes them, batched, and
                with flash_attn 2.8 -- the GPU number the kernels have to beat
  roofline_cfg4 / roofline_cfg5   K1 on the SDXL / DiT-XL/2 shapes of BASELINE.json configs[3], [4]
  retrieval     BASELINE.json configs[2]: the Sref-shaped 2032 x 2032 all-pairs AAS matrix, row-block sharded over the
                ranks (strong scaling; the one path with a collective: NCCL all-gather of K / V)
  cpu_baseline  the reference's own torch lines (4 SDPA + 2 cosine per pair, diffsim/diffsim.py:177-197) on the
                host cores, bounded sample
  e2e           the same metric through the hook-input boundary (HostHiddenTripletScorer): pinned host hidden states
                of the hooked layer -> H2D copies inside the timed region -> QKV projection (K4) -> fused AAS kernels
                (K1) -> decision counts read back.  e2e_qkv_boundary: the same with host Q/K/V (3x the bytes).
The CPU legs (cpu_baseline, --impl reference) time what the reference executes per pair at that boundary: the capture
projections of both images (6 x F.linear, diffsim/hacked_attn.py:61-69) + 4 SDPA + 2 cosine (diffsim/diffsim.py:177-197).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (it may be read-only)

SHAPE = (2, 8, 256, 160)  # SD-1.5 512^2 up_blocks layer 0 (SURVEY.md section 8)
# dram__bytes_read.sum + dram__bytes_write.sum of K1 per triplet, from the ncu --set full capture named in TRAFFIC_SOURCE
DRAM_BYTES_PER_TRIPLET = (6.052258e9 + 8.091136e6) / 512
TRAFFIC_SOURCE = ("profiles/r2final_attn_ncu_summary.txt (ncu --set full of this bench at 512 triplets per launch, the round-2 kernel "
                  "as the bench runs it)")
WORKLOAD = "nights_2afc_triplets_sd15_512_up0_cosine"
METRIC = "scored_pairs_per_sec"


def attn_flops(shape):
    B, H, S, D = shape
    return 4.0 * B * H * S * S * D


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"bf16_tflops": p.get("bf16_tflops", 1590.0), "bf16_tflops_sustained": p.get("bf16_tflops_sustained", 1400.0),
                "hbm_gbs": p.get("hbm_gbs", 6650.0), "source": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0,
            "source": "fallback (B200_PROFILING.md)"}


class ClockSampler(threading.Thread):
    """Samples SM clock, power and throttle reasons of one GPU while the timed region runs (NVML; nvidia-smi as a
    fallback).  A short timed region still gets tens of samples."""

    def __init__(self, index: int, period_s: float = 0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period_s
        self.samples, self.stop_flag = [], threading.Event()
        self.nvml = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
        pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        names = []
        for bit, name in ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"),
                          (0x4, "sw_power_cap")):
            if r & bit:
                names.append(name)
        return sm, self.max_sm, pw, names

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout
        p = [x.strip() for x in out.strip().split(",")]
        names = [nm for nm, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], p[3:7])
                 if v.lower().startswith("active")]
        return float(p[0]), float(p[1]), float(p[2]), names

    def run(self):
        while not self.stop_flag.is_set():
            try:
                self.samples.append(self._sample_nvml() if self.nvml else self._sample_smi())
            except Exception:
                pass
            self.stop_flag.wait(self.period)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = [s[0] for s in self.samples]
        reasons = sorted({r for s in self.samples for r in s[3]})
        return {"sm_mhz": statistics.median(sm), "sm_min_mhz": min(sm), "sm_max_mhz": max(s[1] for s in self.samples),
                "reasons": reasons, "samples": len(self.samples), "power_w_max": max(s[2] for s in self.samples),
                "source": "nvml" if self.nvml else "nvidia-smi"}


def dump_outputs(out_dir: str, outputs: dict) -> None:
    """Write each result tensor as out_dir/<name>.npy: floating results as float32, integer results as float64 (exact
    for int32), so that the outputs of two builds can be compared array by array."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        a = t.cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32 if a.dtype.kind == "f" else np.float64))


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# ------------------------------------------------------------------------------------------------------
# CPU baseline: the reference's arithmetic on the host cores
# ------------------------------------------------------------------------------------------------------
def cpu_reference_pairs_per_sec(n_pairs: int, threads: int, dtype_name: str = "float16", repeats: int = 1):
    """The reference's work per scored pair at the hook-input boundary, on the host cores: for each of the two images
    attn.to_q / to_k / to_v on the hook input + head-split views (diffsim/hacked_attn.py:61-69,74-77 -- the reference
    re-runs the capture for every diffsim(A,B) call), then 4 SDPA + 2 cosine (diffsim/diffsim.py:177-197)."""
    import torch
    from diffsim_b200 import synth
    from oracle import aas_oracle as O

    torch.set_num_threads(threads)
    dtype = getattr(torch, dtype_name)
    B, H, S, D = SHAPE
    C = H * D
    m = synth.SynthModel(B, H, S, D, seed=2334)
    n_img = 8  # a small pool of distinct images, cycled: the cost per pair does not depend on the values
    g = torch.Generator().manual_seed(7)
    base = m.new_base(g)
    hid = [m.hidden(base, 0.5 + 0.06 * i, g).to(dtype) for i in range(n_img)]
    w = m.linear_weights(dtype)
    wq, wk, wv = w[:C], w[C:2 * C], w[2 * C:]

    def pair(a, b):
        qa, ka, va = O.reference_capture(hid[a], wq, wk, wv, H)
        qb, kb, vb = O.reference_capture(hid[b], wq, wk, wv, H)
        return O.reference_pair_score(qa, ka, va, qb, kb, vb)

    for i in range(2):  # warm-up
        pair(0, 1)
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        acc = 0.0
        for p in range(n_pairs):
            acc += float(pair(p % n_img, (p + 1 + p // n_img) % n_img))
        best = min(best, time.perf_counter() - t0)
    return n_pairs / best, best


def run_reference_arm(args):
    """--impl reference: the reference's CPU implementation of the path (its torch calls), all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import torch

    threads = os.cpu_count() or 1
    sample = args.cpu_pairs
    for _ in range(max(0, args.warmup)):
        cpu_reference_pairs_per_sec(max(8, sample // 8), threads)
    times, vals = [], []
    for _ in range(max(1, args.steps)):
        v, t = cpu_reference_pairs_per_sec(sample, threads)
        vals.append(v)
        times.append(t)
    value = sum(sample for _ in vals) / sum(times)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": {"workload": WORKLOAD, "shape_BHSD": list(SHAPE), "similarity": "cosine",
                   "boundary": "hook input (hidden states of the target attn1 layer) -> pair score",
                   "note": "reference arithmetic per pair (6x F.linear capture projections, hacked_attn.py:61-69; 4x "
                           "F.scaled_dot_product_attention + 2x F.cosine_similarity, diffsim/diffsim.py:177-197) in torch %s "
                           "on the host cores; VAE / UNet trunk not included" % torch.__version__},
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} pairs per step, fp16, torch.set_num_threads({threads})"},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0



# ------------------------------------------------------------------------------------------------------
# legs of the GPU arm that are not the headline
# ------------------------------------------------------------------------------------------------------
def _timed_ms(fn, iters, dev):
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / iters


def shape_roofline(name, shape, n_pairs, dtype, dev, peaks, packed_qkv=False, iters=5):
    """K1 on another BASELINE shape: n_pairs AAS pairs (4 attentions each; the kernel runs 2 self + 2 cross per pair) through
    ds_aas_pairs; kernel time from the library's own CUDA events.  packed_qkv: q, k, v are views of one (N,B,S,3,H,D) buffer
    (DiT's qkv(x) layout, diffsim/diffsim_dit.py:22-23)."""
    import torch
    from diffsim_b200 import ops, synth

    B, H, S, D = shape
    n_img = 2 * n_pairs
    q, k, v = synth.device_cache(B, H, S, D, n_img, dtype, dev, seed=77)
    if packed_qkv:
        mem = torch.empty(n_img, B, S, 3, H, D, dtype=dtype, device=dev)
        for j, t in enumerate((q, k, v)):
            mem[:, :, :, j] = t.permute(0, 1, 3, 2, 4)
        q, k, v = (mem[:, :, :, j].permute(0, 1, 3, 2, 4) for j in range(3))
    pairs = torch.arange(n_img, dtype=torch.int32, device=dev).view(n_pairs, 2)
    for _ in range(3):
        ops.aas_pairs(q, k, v, pairs, "cosine")
    ops.profile_enable(True)
    for _ in range(iters):
        ops.aas_pairs(q, k, v, pairs, "cosine")
    ms, n = ops.profile_collect()
    ops.profile_enable(False)
    ms /= max(1, n)
    fl = 4.0 * n_pairs * attn_flops(shape)
    tf = fl / (ms * 1e-3) / 1e12
    return {"kernel": f"aas_attn_kernel<{D}> {name}", "shape_BHSD": list(shape), "pairs_per_launch": n_pairs, "bound": "tensor",
            "achieved": tf, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": tf / peaks["bf16_tflops"], "traffic": None,
            "flops_per_launch": fl, "ms_per_launch": ms, "pairs_per_sec": n_pairs / (ms * 1e-3),
            "layout": "packed qkv (N,B,S,3,H,D)" if packed_qkv else "(N,B,S,H*D) per tensor",
            "inputs_mib": 3 * n_img * B * H * S * D * 2 / 2**20}


def torch_cuda_reference(dtype, dev, n_pairs=64, iters=20):
    """The reference's own lines on the same GPU (SURVEY section 8d-ii): 4 x F.scaled_dot_product_attention + 2 x
    F.cosine_similarity + (a+b)/2 (diffsim/diffsim.py:177-197) on (B,H,S,D) views in the reference layout --
    (a) per pair, one call sequence per pair as the reference executes it; (b) the same arithmetic batched over all pairs;
    (c) flash_attn 2.8 batched, if it runs on this GPU.  CUDA events, >= 20 iterations after warm-up."""
    import torch
    import torch.nn.functional as F
    from diffsim_b200 import synth

    B, H, S, D = SHAPE
    n_img = 2 * n_pairs
    q, k, v = synth.device_cache(B, H, S, D, n_img, dtype, dev, seed=55)   # 0.5 GB at 64 pairs: larger than L2
    fl_pair = 4.0 * attn_flops(SHAPE)
    out = {"shape_BHSD": list(SHAPE), "dtype": str(dtype).replace("torch.", ""), "pairs": n_pairs, "iters": iters,
           "torch": torch.__version__, "what": "4 x SDPA + 2 x cosine_similarity per pair, diffsim/diffsim.py:177-197"}

    def pair(a, b):
        qa, ka, va, qb, kb, vb = q[a], k[a], v[a], q[b], k[b], v[b]
        a_on_b = F.scaled_dot_product_attention(qa, kb, vb, dropout_p=0.0, is_causal=False)
        b_on_a = F.scaled_dot_product_attention(qb, ka, va, dropout_p=0.0, is_causal=False)
        self_a = F.scaled_dot_product_attention(qa, ka, va, dropout_p=0.0, is_causal=False)
        self_b = F.scaled_dot_product_attention(qb, kb, vb, dropout_p=0.0, is_causal=False)
        d1 = F.cosine_similarity(a_on_b.reshape(-1).unsqueeze(0), self_a.reshape(-1).unsqueeze(0))
        d2 = F.cosine_similarity(b_on_a.reshape(-1).unsqueeze(0), self_b.reshape(-1).unsqueeze(0))
        return (d1 + d2) / 2

    def per_pair():
        return [pair(2 * i, 2 * i + 1) for i in range(n_pairs)]

    ia = torch.arange(0, n_img, 2, device=dev)
    ib = ia + 1

    def batched(sdpa):
        qa, ka, va = (t[ia].flatten(0, 1) for t in (q, k, v))   # (P*B,H,S,D) -- the gather is part of the timed work
        qb, kb, vb = (t[ib].flatten(0, 1) for t in (q, k, v))
        a_on_b, b_on_a, self_a, self_b = sdpa(qa, kb, vb), sdpa(qb, ka, va), sdpa(qa, ka, va), sdpa(qb, kb, vb)
        flat = lambda t: t.reshape(n_pairs, -1)  # noqa: E731
        return (F.cosine_similarity(flat(a_on_b), flat(self_a)) + F.cosine_similarity(flat(b_on_a), flat(self_b))) / 2

    try:
        for _ in range(2):
            per_pair()
        reps = max(1, iters // 10)
        ms = _timed_ms(per_pair, reps, dev)
        out["per_pair"] = {"pairs_per_sec": n_pairs / (ms * 1e-3), "tflops": n_pairs * fl_pair / (ms * 1e-3) / 1e12,
                           "ms_per_pair": ms / n_pairs, "pair_evaluations_timed": reps * n_pairs}
        sd = lambda a, b, c: F.scaled_dot_product_attention(a, b, c, dropout_p=0.0, is_causal=False)  # noqa: E731
        for _ in range(3):
            ref_scores = batched(sd)
        ms = _timed_ms(lambda: batched(sd), iters, dev)
        out["batched"] = {"pairs_per_sec": n_pairs / (ms * 1e-3), "tflops": n_pairs * fl_pair / (ms * 1e-3) / 1e12, "ms": ms}
        out["scores_checksum"] = float(ref_scores.float().sum())
    except Exception as e:  # pragma: no cover
        out["error"] = f"{type(e).__name__}: {e}"[:200]
    try:
        from flash_attn import flash_attn_func

        def fa(a, b, c):   # flash_attn wants (batch, seq, heads, dim): a transpose VIEW of the (B,H,S,D) views
            return flash_attn_func(a.transpose(1, 2), b.transpose(1, 2), c.transpose(1, 2), dropout_p=0.0, causal=False).transpose(1, 2)

        for _ in range(3):
            fa_scores = batched(fa)
        ms = _timed_ms(lambda: batched(fa), iters, dev)
        out["flash_attn"] = {"pairs_per_sec": n_pairs / (ms * 1e-3), "tflops": n_pairs * fl_pair / (ms * 1e-3) / 1e12, "ms": ms,
                             "max_abs_diff_to_torch_sdpa": float((fa_scores.float() - ref_scores.float()).abs().max())}
    except Exception as e:
        out["flash_attn"] = {"unavailable": f"{type(e).__name__}: {e}"[:160]}
    return out


def h2d_ceiling(nbytes, dev, barrier, world, dist):
    """Plain pinned-host -> device copy of the same byte count the end-to-end leg moves per step, all ranks at once: the
    ceiling the e2e leg's h2d_gbs is to be read against (max over ranks of the device time)."""
    import torch

    n = min(int(nbytes), 1 << 30)
    host = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    host.fill_(1)
    dst = torch.empty(n, dtype=torch.uint8, device=dev)
    for _ in range(2):
        dst.copy_(host, non_blocking=True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 4
    e0.record()
    for _ in range(reps):
        dst.copy_(host, non_blocking=True)
    e1.record()
    torch.cuda.synchronize(dev)
    t = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    return {"bytes_per_copy": n, "ms": ms, "gbs_per_gpu": n / (ms * 1e-3) / 1e9, "gbs_all_gpus": world * n / (ms * 1e-3) / 1e9,
            "what": "one cudaMemcpyAsync of pinned host memory per rank, all ranks concurrently, max over ranks"}


def retrieval_leg(args, dtype, dev, rank, world, barrier, dist, peaks):
    """BASELINE.json configs[2]: Sref-shaped all-pairs retrieval -- N = 2032 synthetic images (508 styles x 4), the directional
    N x N AAS matrix, images row-block sharded over the ranks, K and V exchanged with one NCCL all_gather each (the only
    data-path collective of the whole port), row blocks gathered at the end.  STRONG scaling: the work is fixed.  Consumer of
    the result: the ranked lists retrieval_vis.py:57-68 parses."""
    import torch
    from diffsim_b200 import ops, retrieval, scoring, synth

    B, H, S, D = SHAPE
    N = args.retrieval_images
    per_style = 4
    r0, r1 = scoring.row_block(N, rank, world)
    cache = scoring.QKVCache(*synth.device_style_cache(B, H, S, D, r0, r1, per_style, dtype, dev))

    def step():
        """ms, max over ranks: [exposed all-gather wait, matrix kernels, gather of the row blocks, total]"""
        if world > 1:
            ev = {}
            dm = scoring.aas_matrix_sharded(cache, "cosine", timings=ev)
            torch.cuda.synchronize(dev)
            t = [ev["own_done"].elapsed_time(ev["exchange_done"]),
                 ev["start"].elapsed_time(ev["own_done"]) + ev["exchange_done"].elapsed_time(ev["block_done"]),
                 ev["block_done"].elapsed_time(ev["end"]), ev["start"].elapsed_time(ev["end"])]
        else:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dm = ops.aas_matrix(cache.q, cache.k, cache.v, cache.k, cache.v, "cosine")
            e1.record()
            torch.cuda.synchronize(dev)
            t = [0.0, e0.elapsed_time(e1), 0.0, e0.elapsed_time(e1)]
        t = torch.tensor(t, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return dm, t.tolist()

    barrier()
    dm, _ = step()   # warm-up: NCCL communicator, tensor maps, workspaces
    best = None
    for _ in range(max(1, args.retrieval_reps)):
        barrier()
        dm, t = step()
        if best is None or t[3] < best[3]:
            best = t
    ms_gather, ms_matrix, ms_rows, ms_total = best
    flops = (N * N + N) * attn_flops(SHAPE)        # N^2 cross attentions (incl. the diagonal) + N self attentions
    kv_bytes = 2 * N * B * H * S * D * 2
    recv = (world - 1) / world * kv_bytes if world > 1 else 0
    res = {"workload": "sref_all_pairs_sd15_512_up0_cosine", "images": N, "shape_BHSD": list(SHAPE), "n_gpus": world,
           "scaling": "strong", "ms_total": ms_total, "ms_matrix_kernels": ms_matrix, "ms_allgather_kv_exposed": ms_gather,
           "ms_gather_rows": ms_rows, "scores_per_sec": N * N / (ms_total * 1e-3),
           "pairs_per_sec": N * (N - 1) / 2 / (ms_total * 1e-3),
           "attn_tflops_whole_job": flops / (ms_matrix * 1e-3) / 1e12,
           "attn_tflops_per_gpu": flops / world / (ms_matrix * 1e-3) / 1e12,
           "frac_of_burst_peak_per_gpu": flops / world / (ms_matrix * 1e-3) / 1e12 / peaks["bf16_tflops"],
           "allgather_recv_bytes_per_rank": recv,
           "allgather_gbs_if_fully_exposed": (recv / (ms_gather * 1e-3) / 1e9) if ms_gather > 0.05 else None,
           "nvlink_peak_gbs_per_dir": 900.0,
           "exchange": "NCCL all_gather_into_tensor of K and of V, issued asynchronously before the rank scores its rows against its "
                       "own columns; ms_allgather_kv_exposed is the wait left AFTER that block (the part not hidden)",
           "timing": "CUDA events on the launching stream, max over ranks, best of %d after one warm-up" % max(1, args.retrieval_reps)}
    if rank == 0:
        labels = [i // per_style for i in range(N)]
        res["retrieval_accuracy"] = retrieval.retrieval_accuracy(scoring.symmetrize(dm), labels, topk=per_style - 1)
        # bitwise check on a sampled row block: rank 0 rebuilds EVERY image (the generator is deterministic per image) and
        # recomputes 8 of its rows against all N columns in one unsharded call
        full = scoring.QKVCache(*synth.device_style_cache(B, H, S, D, 0, N, per_style, dtype, dev))
        rows = [0, 1, 2, 3, (r1 - r0) // 2, (r1 - r0) // 2 + 1, r1 - r0 - 2, r1 - r0 - 1]
        idx = torch.tensor(rows, device=dev)
        mem = [m[idx] for m in full.memory()]
        sub = scoring.QKVCache(*(m.view(len(rows), B, S, H, D).permute(0, 1, 3, 2, 4) for m in mem))
        ref = ops.aas_matrix(sub.q, sub.k, sub.v, full.k, full.v, "cosine")
        res["bitwise_equal_to_rank_local_recompute"] = bool(torch.equal(ref, dm[idx]))
        res["checked_rows"] = rows
        del full, ref
    del cache, dm
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--triplets", type=int, default=2048, help="triplets per step per GPU (device-resident run)")
    ap.add_argument("--e2e-triplets", type=int, default=384, help="triplets per step per GPU in the end-to-end run")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-pairs", type=int, default=512, help="pairs in the bounded CPU-baseline sample")
    ap.add_argument("--dtype", default="float16", choices=["float16", "bfloat16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the K2 / K3 / K4 / cfg4 / cfg5 secondary roofline measurements")
    ap.add_argument("--no-torch-reference", action="store_true", help="skip the torch-CUDA / flash_attn reference timing")
    ap.add_argument("--no-retrieval", action="store_true", help="skip the all-pairs retrieval leg (BASELINE configs[2])")
    ap.add_argument("--retrieval-images", type=int, default=2032)
    ap.add_argument("--retrieval-reps", type=int, default=1)
    ap.add_argument("--no-numa-bind", action="store_true", help="N > 1: do not bind ranks to their GPU's NUMA-local CPUs")
    ap.add_argument("--profiler-range", action="store_true",
                    help="bracket the timed device-resident steps with cudaProfilerStart/Stop (ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (rank 0's ab, ac, counts, flags of "
                         "score_triplets) as DIR/<name>.npy; the inputs are seeded, so runs with the same arguments compare")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist

    from diffsim_b200 import ops, scoring, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE {world}", file=sys.stderr)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # pinned staging buffers of the end-to-end leg should be local to the GPU's socket: bind before allocating them
    from diffsim_b200 import hostbind
    numa = hostbind.bind_to_gpu_node(local_rank) if world > 1 and not args.no_numa_bind else {"bound": False, "why": "single rank"}
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    dtype = getattr(torch, args.dtype)
    B, H, S, D = SHAPE
    T = args.triplets
    # ---- inputs resident in HBM (weak scaling: every rank owns T triplets) -----------------------------------
    q, k, v = synth.device_cache(B, H, S, D, 3 * T, dtype, dev, seed=1000 + rank)
    cache = scoring.QKVCache(q, k, v)
    trips = torch.arange(3 * T, dtype=torch.int32, device=dev).view(T, 3)
    pairs_per_step = 2 * T
    attn_per_step = 7 * T  # ref self + 2 cross, left self + cross, right self + cross
    resident_gib = 3 * T * cache.bytes_per_image / 2**30

    def step():
        return scoring.score_triplets(cache, trips, "cosine")

    for _ in range(max(3, args.warmup)):
        ab, ac, counts, flags = step()
    barrier()
    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    ops.profile_enable(True)
    launches0 = ops.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if args.profiler_range:
        torch.cuda.cudart().cudaProfilerStart()
    e0.record()
    for _ in range(args.steps):
        ab, ac, counts, flags = step()
    e1.record()
    barrier()
    if args.profiler_range:
        torch.cuda.cudart().cudaProfilerStop()
    launches = ops.LAUNCHES - launches0
    kern_ms, kern_n = ops.profile_collect()
    ops.profile_enable(False)
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    ms_total = e0.elapsed_time(e1)
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_per_step = ms_total / args.steps
    value = world * pairs_per_step * args.steps / (ms_total * 1e-3)
    correct = int(counts[0].item())
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"ab": ab, "ac": ac, "counts": counts, "flags": flags})

    # ---- roofline of the dominant kernel ---------------------------------------------------------------------
    peaks = load_peaks()
    kern_ms_per_launch = kern_ms / max(1, kern_n)
    achieved_tflops = attn_per_step * attn_flops(SHAPE) / (kern_ms_per_launch * 1e-3) / 1e12 if kern_n else None
    # Denominator: the BURST bf16 figure of MEASURED_PEAKS.json (north_star's ">= 60% of bf16 tensor-core peak"); the timed
    # region is a power-capped train of this one kernel, so the fraction of the SUSTAINED figure is printed beside it.
    peak = peaks["bf16_tflops"]
    roofline = {
        "kernel": "aas_attn_kernel<160,f16,cos> (fused QK^T -> online softmax -> PV -> cosine partials; tcgen05/TMEM/TMA)",
        "bound": "tensor", "achieved": achieved_tflops, "peak": peak, "unit": "TFLOP/s",
        "frac": (achieved_tflops / peak) if achieved_tflops else None,
        "frac_sustained": (achieved_tflops / peaks["bf16_tflops_sustained"]) if achieved_tflops else None,
        "peak_sustained": peaks["bf16_tflops_sustained"],
        "peak_source": peaks["source"] + ": burst bf16 figure (frac), sustained bf16 figure (frac_sustained)",
        # dram__bytes_read.sum + dram__bytes_write.sum of this kernel, per launch: NOT measured in this run -- the per-triplet
        # figure of the ncu --set full capture named in traffic_source, scaled to this launch's triplet count
        "traffic": DRAM_BYTES_PER_TRIPLET * T, "traffic_algorithmic": 3 * T * cache.bytes_per_image,
        "traffic_source": TRAFFIC_SOURCE,
        "flops_per_launch": attn_per_step * attn_flops(SHAPE), "ms_per_launch": kern_ms_per_launch,
        "launches_timed": kern_n, "share_of_step": (kern_ms_per_launch / ms_per_step) if kern_n else None,
        "algorithmic": "7 directional attentions per triplet x 4*B*H*S*S*D flops (DESIGN.md section 3)",
    }

    # ---- end to end: host buffers, H2D inside the timed region -------------------------------------------------
    e2e = None
    extra = {}
    if not args.no_e2e:
        Te = args.e2e_triplets

        def timed(fn, n_steps):
            barrier()
            t0 = time.perf_counter()
            e0.record()
            for _ in range(n_steps):
                out = fn()
            e1.record()
            torch.cuda.synchronize(dev)
            wall = time.perf_counter() - t0
            te = torch.tensor([max(wall * 1e3, e0.elapsed_time(e1))], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            return float(te.item()), out

        # (1) the headline: hook-input boundary.  Pinned host hidden states -> K4 projection -> K1 scoring
        del cache, q, k, v
        torch.cuda.empty_cache()
        hid_host, weight = synth.device_hidden(B, H, S, D, 3 * Te, dtype, dev, seed=2000 + rank, pin_host=True)
        hscorer = scoring.HostHiddenTripletScorer(SHAPE, weight, None, dtype, dev, chunk_triplets=96)
        hscorer.score(hid_host, Te)  # warm-up
        hscorer.score(hid_host, Te)
        hscorer.h2d_bytes = hscorer.d2h_bytes = 0
        l0 = ops.LAUNCHES
        ms_e, c_e2e = timed(lambda: hscorer.score(hid_host, Te), args.e2e_steps)
        e2e = {"value": world * 2 * Te * args.e2e_steps / (ms_e * 1e-3), "unit": "pairs/s",
               "h2d_bytes_per_step": hscorer.h2d_bytes // args.e2e_steps,
               "d2h_bytes_per_step": hscorer.d2h_bytes // args.e2e_steps,
               "triplets_per_step_per_gpu": Te, "steps": args.e2e_steps, "gpu_launches": ops.LAUNCHES - l0,
               "boundary": "hook input: hidden states (B,S,C) of the target attn1 layer, 3 images per triplet",
               "api": "diffsim_b200.scoring.HostHiddenTripletScorer.score (pinned host hidden states -> ds_qkv_project -> "
                      "ds_aas_triplets -> counts)",
               "h2d_gbs": hscorer.h2d_bytes / (ms_e * 1e-3) / 1e9, "correct": c_e2e[0]}
        e2e["h2d_gbs_all_gpus"] = e2e["h2d_gbs"] * world
        e2e["h2d_ceiling"] = h2d_ceiling(e2e["h2d_bytes_per_step"], dev, barrier, world, dist)
        e2e["h2d_frac_of_ceiling"] = e2e["h2d_gbs"] / e2e["h2d_ceiling"]["gbs_per_gpu"]
        # K4 alone on the resident copy of the same hidden states (secondary roofline)
        hid_dev = hid_host[: 3 * min(Te, 256)].to(dev)
        outs = [torch.empty(hid_dev.shape[:-1] + (H * D,), dtype=dtype, device=dev) for _ in range(3)]
        for _ in range(3):
            ops.qkv_project(hid_dev, weight, None, 3, out=outs)
        e0.record()
        for _ in range(10):
            ops.qkv_project(hid_dev, weight, None, 3, out=outs)
        e1.record()
        torch.cuda.synchronize(dev)
        k4_ms = e0.elapsed_time(e1) / 10
        k4_fl = 2.0 * hid_dev.shape[0] * B * S * (H * D) * (3 * H * D)
        extra["roofline_k4"] = {"kernel": "gemm2_tn_kernel<EPI_16> (QKV projection, tcgen05 cta_group::2 256x256 tiles, TMA-store epilogue)", "bound": "tensor",
                                "achieved": k4_fl / (k4_ms * 1e-3) / 1e12, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                                "frac": k4_fl / (k4_ms * 1e-3) / 1e12 / peaks["bf16_tflops"], "traffic": None,
                                "flops_per_launch": k4_fl, "ms_per_launch": k4_ms, "images_per_launch": hid_dev.shape[0]}
        del hid_dev, outs
        # (2) for comparison: the Q/K/V boundary (what round-1's first bench lines reported)
        dcache = scoring.project_cache(hid_host[: 3 * Te].to(dev), weight, H)
        host = scoring.QKVCache.empty(3 * Te, B, H, S, D, dtype, "cpu", pin=True)
        for hm, dm in zip(host.memory(), dcache.memory()):
            hm.copy_(dm)
        del dcache
        scorer = scoring.HostTripletScorer(SHAPE, dtype, dev, chunk_triplets=96)
        scorer.score(host, Te)  # warm-up
        scorer.h2d_bytes = scorer.d2h_bytes = 0
        ms_q, c_q = timed(lambda: scorer.score(host, Te), args.e2e_steps)
        extra["e2e_qkv_boundary"] = {"value": world * 2 * Te * args.e2e_steps / (ms_q * 1e-3), "unit": "pairs/s",
                                     "h2d_bytes_per_step": scorer.h2d_bytes // args.e2e_steps,
                                     "d2h_bytes_per_step": scorer.d2h_bytes // args.e2e_steps,
                                     "api": "diffsim_b200.scoring.HostTripletScorer.score (pinned host Q/K/V -> ds_aas_triplets)",
                                     "correct": c_q[0]}
        del host, scorer, hscorer, hid_host

    # ---- secondary kernels (rank 0): K2 reductions vs HBM, K3 similarity GEMM vs tensor peak ----------------------
    if rank == 0 and not args.no_secondary:
        torch.cuda.empty_cache()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        E = B * H * S * D
        P2 = 256                                  # 2 x 256 x 1.31 MB = 671 MB of inputs: larger than the 126 MB L2
        g = torch.Generator(device=dev).manual_seed(7)
        x = torch.randn(P2, E, generator=g, device=dev, dtype=torch.float32).to(dtype)
        y = (0.6 * x.float() + 0.4 * torch.randn(P2, E, generator=g, device=dev)).to(dtype)
        for mode in ("cosine", "minmax_cosine"):
            for _ in range(3):
                ops.pair_reduce(x, y, mode)
            e0.record()
            for _ in range(10):
                ops.pair_reduce(x, y, mode)
            e1.record()
            torch.cuda.synchronize(dev)
            ms2 = e0.elapsed_time(e1) / 10
            by = 2.0 * P2 * E * x.element_size() + 4 * P2
            extra["roofline_k2" if mode == "cosine" else "roofline_k2_minmax"] = {
                "kernel": f"pair_reduce_kernel<{args.dtype},{mode}> (batched flat reduction, one pass)", "bound": "hbm",
                "achieved": by / (ms2 * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": by / (ms2 * 1e-3) / 1e9 / peaks["hbm_gbs"], "traffic": None, "bytes_per_launch": by,
                "ms_per_launch": ms2, "pairs_per_launch": P2,
                "algorithmic": "2 * E * sizeof(dtype) read + 4 B written per row pair (DESIGN.md section 3)"}
        del x, y
        Nf, Lf = 2032, E                          # Sref-shaped: 2032 images x flattened (2,256,1280) diffeats features
        feats = torch.empty(Nf, Lf, dtype=dtype, device=dev)
        for i0 in range(0, Nf, 127):
            feats[i0:i0 + 127] = torch.randn(min(127, Nf - i0), Lf, generator=g, device=dev).to(dtype)
        outm = torch.empty(Nf, Nf, dtype=torch.float32, device=dev)
        for _ in range(2):
            ops.simmat(feats, None, "cosine", out=outm)
        e0.record()
        for _ in range(3):
            ops.simmat(feats, None, "cosine", out=outm)
        e1.record()
        torch.cuda.synchronize(dev)
        ms3 = e0.elapsed_time(e1) / 3
        # self-similarity runs the upper-triangle tile schedule: EXECUTED flops = tiles on/above the diagonal x 128 x 256 x 2L
        tm_n, tn_n = (Nf + 127) // 128, (Nf + 255) // 256
        tiles_exec = sum(max(0, tn_n - (tm * 128) // 256) for tm in range(tm_n))
        fl3 = 2.0 * tiles_exec * 128 * 256 * Lf
        extra["roofline_k3"] = {"kernel": "simmat: row statistics + gemm2_tn_kernel<EPI_F32> (CTA pairs, 256x256 upper-triangle tiles, "
                                          "split-K) + normalise/mirror (N x N cosine)",
                                "bound": "tensor", "achieved": fl3 / (ms3 * 1e-3) / 1e12, "peak": peaks["bf16_tflops"],
                                "unit": "TFLOP/s", "frac": fl3 / (ms3 * 1e-3) / 1e12 / peaks["bf16_tflops"], "traffic": None,
                                "flops_per_launch": fl3, "flops_full_matrix": 2.0 * Nf * Nf * Lf, "ms_per_call": ms3,
                                "images": Nf, "feature_len": Lf,
                                "full_matrix_equivalent_tflops": 2.0 * Nf * Nf * Lf / (ms3 * 1e-3) / 1e12,
                                "note": "whole ds_simmat call (one statistics pass + GEMM + finish); achieved counts the flops "
                                        "EXECUTED (36 of 64 256x256 tiles), full_matrix_equivalent the 2*N*N*L of the result",
                                "diag_minus_one_max": float((outm.diagonal() - 1).abs().max())}
        del feats, outm
        torch.cuda.empty_cache()
        # K1 on the shapes of BASELINE.json configs[3] (SDXL 1024^2: the two real up-block layers and the literal "4096 tokens x
        # 1280 channels") and configs[4] (DiT-XL/2 256^2, packed qkv strides, IPref-shaped pair batch)
        extra["roofline_cfg4"] = {
            "sdxl_up0_2x20x1024x64": shape_roofline("SDXL up_blocks[0]", (2, 20, 1024, 64), 64, dtype, dev, peaks),
            "sdxl_up1_2x10x4096x64": shape_roofline("SDXL up_blocks[1]", (2, 10, 4096, 64), 16, dtype, dev, peaks),
            "literal_2x20x4096x64": shape_roofline("literal 4096 tokens x 1280 ch", (2, 20, 4096, 64), 8, dtype, dev, peaks)}
        extra["roofline_cfg5"] = {
            "dit_xl2_2x16x256x72_packed": shape_roofline("DiT-XL/2 blocks[l].attn", (2, 16, 256, 72), 512, dtype, dev, peaks,
                                                         packed_qkv=True)}
        torch.cuda.empty_cache()

    # ---- the reference's own torch lines on this GPU (rank 0) -------------------------------------------------------
    if rank == 0 and not args.no_torch_reference:
        torch.cuda.empty_cache()
        extra["torch_cuda_reference"] = torch_cuda_reference(dtype, dev)
        torch.cuda.empty_cache()

    # ---- all-pairs retrieval, row-block sharded (every rank; strong scaling; NCCL all-gather of K / V) ----------------
    if not args.no_retrieval:
        r = retrieval_leg(args, dtype, dev, rank, world, barrier, dist if world > 1 else None, peaks)
        if rank == 0:
            extra["retrieval"] = r

    # ---- CPU baseline (rank 0, N = 1 only) ----------------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v_cpu, t_cpu = cpu_reference_pairs_per_sec(args.cpu_pairs, threads)
        cpu = {"value": v_cpu, "unit": "pairs/s", "cores": threads, "kind": "port",
               "sample": f"{args.cpu_pairs} pairs of the same shape, fp16, reference torch calls per pair at the hook-input "
                         f"boundary (6 F.linear capture projections + 4 SDPA + 2 cosine), {t_cpu:.1f} s"}

    if world > 1:
        dist.barrier()
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16" if dtype == torch.float16 else "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD, "shape_BHSD": list(SHAPE), "triplets_per_step_per_gpu": T,
                       "pairs_per_step_per_gpu": pairs_per_step, "attentions_per_triplet": 7,
                       "similarity": "cosine", "parallelism": f"pairs sharded over {world} rank(s), no data-path collective",
                       "value_boundary": "Q/K/V of the hooked layer resident in HBM (K1 only); e2e adds the hook-input "
                                         "boundary: H2D of hidden states + K4 projection",
                       "l2": f"inputs {resident_gib:.1f} GiB per step > 126 MB L2 (no flush needed)"},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches,
            "clocks": sampler.summary(), "correct_2afc": correct, "numa_bind": numa,
        }
        line.update(extra)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
