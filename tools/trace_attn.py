#!/usr/bin/env python
"""Timeline of CTA 0 of the attention kernel (library must be built with DS_EXTRA_NVCC_FLAGS=-DDS_TRACE).
Prints, per role, the (tag, clock) events of a few steady-state items."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from diffsim_b200 import ops, synth, _native as N

CAP = 4096
B, H, S, D = (int(x) for x in os.environ.get("TR_SHAPE", "2,8,256,160").split(","))
n_img = int(os.environ.get("TR_IMAGES", "768"))
q, k, v = synth.device_cache(B, H, S, D, n_img, torch.float16, "cuda")
pairs = torch.tensor([(3 * t, 3 * t + 1) for t in range(n_img // 3)] + [(3 * t, 3 * t + 2) for t in range(n_img // 3)],
                     dtype=torch.int32, device="cuda")
buf = torch.zeros(8 * CAP, dtype=torch.int64, device="cuda")
lib = N.load()
ops.aas_pairs(q, k, v, pairs, "cosine")
torch.cuda.synchronize()
on = lib.ds_debug_set_trace(buf.data_ptr(), CAP)
print("trace compiled in:", on)
ops.aas_pairs(q, k, v, pairs, "cosine")
torch.cuda.synchronize()
lib.ds_debug_set_trace(None, 0)
t = buf.cpu().view(8, CAP)
names = {1: "prod wait kv_empty", 2: "prod got slot", 3: "prod wait q_empty", 4: "prod Q issued",
         10: "mma qkA begin", 11: "mma qkB begin", 12: "mma qkA kv ready", 13: "mma qkB kv ready", 14: "mma qkA committed",
         15: "mma qkB committed", 17: "mma wait q_full", 18: "mma got Q",
         20: "mma pvA begin", 21: "mma pvB begin", 22: "mma pvA p_full ok", 23: "mma pvB p_full ok", 24: "mma pvA o_empty + kv ready",
         25: "mma pvB kv ready", 26: "mma pvA committed", 27: "mma pvB committed",
         30: "sm wait s_full A", 31: "sm wait s_full B", 32: "sm got S_A", 33: "sm got S_B", 34: "sm max A written", 35: "sm max B written",
         36: "sm bar A passed", 37: "sm bar B passed", 38: "sm arrived p_full A", 39: "sm arrived p_full B",
         44: "sm P_A stored (issued)", 45: "sm P_B stored (issued)", 46: "sm st A complete", 47: "sm st B complete",
         48: "sm S_A in registers", 49: "sm S_B in registers",
         40: "epi o_full", 42: "epi released O", 41: "epi done"}
ev = []
for slot in range(8):
    for x in t[slot].tolist():
        if x == 0:
            continue
        tag, clk = (x >> 48) & 0xFFFF, x & 0xFFFFFFFFFFFF
        ev.append((clk, slot, tag))
ev.sort()
if not ev:
    print("no events")
    sys.exit(0)
# steady state window: skip the first 40% of events
t0 = ev[0][0]
lo = int(os.environ.get("TR_LO", "60000")); hi = int(os.environ.get("TR_HI", "85000"))
last = {}
for clk, slot, tag in ev:
    r = clk - t0
    if lo <= r <= hi and (not os.environ.get("TR_SLOT") or str(slot) in os.environ["TR_SLOT"].split(",")):
        d = r - last.get(slot, r)
        print(f"{r:8d} (+{d:5d}) slot{slot} {names.get(tag, tag)}")
    last[slot] = r
# per-item period from the epilogue
epi = [clk for clk, slot, tag in ev if tag == 41]
if len(epi) > 20:
    import statistics
    d = [b - a for a, b in zip(epi[10:-1], epi[11:])]
    print("epilogue-done period: median", statistics.median(d), "mean", sum(d) / len(d), "n", len(d))
