"""Profiling target (run under ncu on a GPU box): one fused WPS+coverage+histogram step and one fused
adjust (rank median + Savitzky-Golay) call at chr1 scale.
    EXTRAS=1 ncu --set full --clock-control none --import-source on \
        -k regex:"adjust_rank_kernel|wps_stream_kernel|end_motif_kernel|cleavage_tile_kernel|delfi_count_kernel" -c 5 \
        -o gpurun_out/r2b_top python tools/prof_kernels.py
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from finaletoolkit_b200 import device as D
from finaletoolkit_b200.synth import synth_fragments_device

CLEN = int(os.environ.get("CLEN", 249_250_621))
N = int(os.environ.get("NFRAG", round(CLEN * 80_000_000 / 249_250_621)))
dev = D.require_cuda("cuda:0")
st, sp, mq = synth_fragments_device(CLEN, N, 0, dev)
fr = D.ContigFragments(st, sp, mq, None, device=dev, max_len=600)
edges = np.arange(0, CLEN + 5000, 5000, dtype=np.int64).clip(max=CLEN)
plan = D.WpsPlan(edges[:-1], edges[1:], CLEN, 180, dev)
reps = int(os.environ.get("REPS", 1))
for _ in range(reps):
    wps, cov, hist = plan.run_fused(fr, n_bins=601)
aplan = D.AdjustPlan(np.diff(plan.offsets), 1000, True, 21, 2, dev, skip_short=True)
for _ in range(reps):
    out, off = D.adjust_segments(wps, None, plan=aplan)
if os.environ.get("EXTRAS"):
    from finaletoolkit_b200.synth import synth_twobit
    codes, nm = synth_twobit(CLEN, 0)
    ref = D.PackedContig.from_codes(codes, nm, device=dev)
    fr.strand = torch.ones(fr.n, dtype=torch.uint8, device=dev)
    ws = list(range(0, CLEN - 1_000_000, 1_000_000)); we = [a + 1_000_000 for a in ws]
    D.end_motif_hist(fr, ref, ws, we, k=4, strand_mode=0, quality_threshold=30, pooled=True)
    D.cleavage_intervals(fr, edges[:-1], edges[1:], CLEN, None, None, 30)
    bs = np.arange(0, CLEN, 100_000, dtype=np.int64); be = np.minimum(bs + 100_000, CLEN)
    D.delfi_windows(fr, ref, bs, be, quality_threshold=30)
torch.cuda.synchronize()
print("ok", int(cov.sum()), float(out[:3].sum()))
