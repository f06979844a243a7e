#!/usr/bin/env python
"""A/B timing of the attention kernel in SM clocks per 128x256x160 item (clock-independent), pairs and triplets.
usage: python tools/perf_attn.py [lib.so ...]   (each library is loaded in its own subprocess, 3 repetitions)"""
import os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def child():
    import torch
    from diffsim_b200 import ops, synth, _native as N
    B, H, S, D = 2, 8, 256, 160
    n_img = 768
    q, k, v = synth.device_cache(B, H, S, D, n_img, torch.float16, "cuda")
    T = n_img // 3
    pairs = torch.tensor([(3 * t, 3 * t + 1) for t in range(T)] + [(3 * t, 3 * t + 2) for t in range(T)], dtype=torch.int32, device="cuda")
    trips = torch.arange(3 * T, dtype=torch.int32, device="cuda").view(T, 3)
    cyc = torch.zeros(8 * 4 + 1, dtype=torch.int64, device="cuda")
    lib = N.load()
    grid = torch.cuda.get_device_properties(0).multi_processor_count   # K1 runs one persistent CTA per SM
    out = []
    for name, fn, attn in (("pairs", lambda: ops.aas_pairs(q, k, v, pairs, "cosine"), 4 * pairs.shape[0]),
                           ("triplets", lambda: ops.aas_triplets(q, k, v, trips, "cosine"), 7 * T)):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        lib.ds_debug_set_trace(cyc.data_ptr(), 4)
        fn()
        torch.cuda.synchronize()
        lib.ds_debug_set_trace(None, 0)
        items = attn * B * H * (S // 128) / grid
        tf = attn * 4 * B * H * S * S * D / ms / 1e9
        out.append(f"{name}: {int(cyc[-1]) / items:.0f} clk/item, {ms:.3f} ms, {tf:.0f} TFLOP/s, {int(cyc[-1]) / ms / 1e6:.2f} GHz")
    print(" | ".join(out))


if __name__ == "__main__":
    if os.environ.get("PERF_CHILD"):
        child()
    else:
        libs = sys.argv[1:] or [os.path.join(ROOT, "diffsim_b200", "_lib", "libdiffsim_b200.so")]
        for rep in range(3):
            for lib in libs:
                env = dict(os.environ, PERF_CHILD="1", DIFFSIM_B200_LIB=os.path.abspath(lib))
                r = subprocess.run([sys.executable, os.path.abspath(__file__)], env=env, capture_output=True, text=True, timeout=300)
                print(f"[{os.path.basename(lib)} rep{rep}] {r.stdout.strip() or r.stderr.strip()[-300:]}", flush=True)
