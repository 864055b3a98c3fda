"""Profiling helper (run from the repo root: PYTHONPATH=. python tools/...): quick WPS timing at config 2 (chr1-scale) - not the bench contract."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import sys, time
import numpy as np, torch, os, ctypes
from finaletoolkit_b200.device import ContigFragments, WpsPlan
from finaletoolkit_b200.synth import synth_fragments
clen = 249_250_621; n = int(sys.argv[1]) if len(sys.argv) > 1 else 80_000_000
t0 = time.time(); st, sp, mq, sd = synth_fragments(clen, n, 0); print("synth", time.time() - t0, flush=True)
fr = ContigFragments(st, sp, mq, sd, device="cuda:0", max_len=600)
edges = np.arange(0, clen + 5000, 5000).clip(max=clen)
plan = WpsPlan(edges[:-1], edges[1:], clen, 180, "cuda:0")
out = torch.empty(plan.n_positions, dtype=torch.int32, device="cuda:0")
for _ in range(3): plan.run(fr, out=out)
torch.cuda.synchronize()
ev = [torch.cuda.Event(enable_timing=True) for _ in range(11)]
for i in range(10):
    ev[i].record(); plan.run(fr, out=out)
ev[10].record(); torch.cuda.synchronize()
ts = [ev[i].elapsed_time(ev[i + 1]) for i in range(10)]
ms = float(np.median(ts)); byt = 9 * n + 4 * plan.n_positions
print(f"tiles={plan.n_tiles} ms={ms:.3f} (min {min(ts):.3f}) GB/s={byt / ms / 1e6:.1f} frags/s={n / ms * 1e3:.3e} pos/s={plan.n_positions / ms * 1e3:.3e} checksum={int(out.sum(dtype=torch.int64))}")
