"""Quick device-resident sort timing with per-kernel-class breakdown (experiments; not the bench)."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, numpy as np
from ytsaurus_b200 import GpuContext, capi
from ytsaurus_b200.rowset import EValueType as T
n = int(sys.argv[1]) if len(sys.argv) > 1 else 100_000_000
steps = 5
ctx = GpuContext(0)
g = torch.Generator(device="cuda").manual_seed(1)
rows = torch.randint(-2**63, 2**63 - 1, (n, 8), dtype=torch.int64, device="cuda", generator=g).view(torch.uint8).reshape(-1)
out = torch.empty_like(rows)
cols = [(0, 0, T.Uint64, 0, 1)]
for _ in range(2):
    ctx.sort_fixed_rows(rows, 64, cols, out_rows=out)
torch.cuda.synchronize()
ctx.enable_timers(True); ctx.reset_timers()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(steps):
    ctx.sort_fixed_rows(rows, 64, cols, out_rows=out)
e1.record(); torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / steps
k = out.view(torch.int64).reshape(n, 8)[:, 0] ^ (-2**63)
ok = bool((k[1:] >= k[:-1]).all())
names = ["pass", "gather", "extract", "hist", "part", "groupby", "decode"]
parts = {names[i]: round(ctx.kernel_ms(i)[0] / steps, 3) for i in range(4)}
print(f"n={n} ms/step={ms:.3f} rows/s={n/ms*1e3:.3e} sorted={ok} {parts} pass_frac={24*n/(parts['pass']/8*1e-3)/1e9/6564.2:.3f}")
