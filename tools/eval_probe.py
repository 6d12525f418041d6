"""Time the full-rank kernels in isolation: python tools/eval_probe.py [n_users] [n_items] [precision ...]

The tensor-core path ("tf32x3") issues three kind::f16 MMA passes per score tile (hi.hi + lo.hi + hi.lo of the
scaled fp16 split): its issued rate is 3 x 2 U I 64 flop (K padded to 64) over the time, set against the dense FP16
data-sheet rate of one B200 (2250 TFLOP/s at 1000 W; a card with a lower power limit clocks lower).  RECAD_TC_DEBUG=2
times the TMA + MMA pipeline alone, RECAD_TC_DEBUG=3 the ranking epilogue with one MMA per tile."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from recad_b200 import ops  # noqa: E402

U = int(sys.argv[1]) if len(sys.argv) > 1 else 37888
I = int(sys.argv[2]) if len(sys.argv) > 2 else 200000
precs = sys.argv[3:] or ["tf32x3", "exact"]
F16_PEAK = 2250.0      # TFLOP/s, dense FP16 / BF16, one B200 (data sheet)
dev = torch.device("cuda:0")
g = torch.Generator(device=dev).manual_seed(0)
ue = torch.randn(U, 64, device=dev, generator=g) * 0.1
ie = torch.randn(I, 64, device=dev, generator=g) * 0.1
deg = 50
ptr = torch.arange(0, (U + 1) * deg, deg, device=dev)
col = torch.sort(torch.randint(0, I, (U, deg), device=dev, generator=g), 1)[0].int().flatten()
users = torch.arange(U, device=dev)
for p in precs:
    for rep in range(2):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = ops.fullrank_eval(ue, ie, users, ptr, col, [0], 20, precision=p)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
    line = f"{p}: {ms:.2f} ms for {U} users x {I} items -> {U / ms * 1e3:.0f} users/s, {2 * U * I * 64 / ms / 1e9:.1f} TFLOP/s useful"
    if p == "tf32x3":
        issued = 3 * 2 * U * I * 64 / ms / 1e9
        line += f", {issued:.1f} TFLOP/s issued on kind::f16 = {issued / F16_PEAK:.3f} of the {F16_PEAK:.0f} data-sheet rate"
    print(line, flush=True)
