"""Kernel timing helper (python tools/quick_kernels.py [motif] [bp] [adjust] [delfi] [hist] [cleavage] [depth] [depth-mid]
[vplot] [vplot-dense]
[gc-obs] [gc-exp] [gc-cov] [gc-site] [spectrum]):
CUDA-event time of the secondary kernels at chr1 scale (80 M fragments drawn on the GPU), median of 7 calls after 3
warm-ups (the call: planning and uploads included).  Every op except adjust also prints an order-sensitive checksum
of its output (compare two builds with it) and each kernel's own device time (torch.profiler, a separate run)."""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from finaletoolkit_b200 import device as D
from finaletoolkit_b200.synth import synth_fragments_device, synth_twobit

what = set(sys.argv[1:]) or {"motif", "bp", "adjust"}
CLEN, N = 249_250_621, 80_000_000
dev = D.require_cuda("cuda:0")
st, sp, mq = synth_fragments_device(CLEN, N, 0, dev)
g = torch.Generator(device=dev); g.manual_seed(5)
sd = (torch.rand(N, generator=g, device=dev) < 0.5).to(torch.uint8)
fr = D.ContigFragments(st, sp, mq, sd, device=dev, max_len=600)


def timed(name, fn, nbytes):
    for _ in range(3):
        out = fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(7):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); out = fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ms = timed.ms = float(np.median(ts))
    print(f"{name}: {ms:.3f} ms (min {min(ts):.3f})  {nbytes / ms / 1e6:.0f} GB/s = {nbytes / ms / 1e6 / 6541.1:.1%} of measured HBM peak", flush=True)
    return out


def kernels(fn, reps=5):
    """Device time per call of each ftk:: kernel fn launches (CUPTI through torch.profiler, a separate run)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    for ev in prof.key_averages():
        if "ftk::" in ev.key:
            print(f"  kernel {ev.key.split('(')[0]}: {ev.device_time_total / reps / 1e3:.3f} ms", flush=True)


def checksum(o):
    """Order-sensitive checksum of an output tensor's bits (int64 arithmetic wraps)."""
    x = o.contiguous().flatten()
    if x.is_floating_point():
        x = x.view({8: torch.int64, 4: torch.int32}[x.element_size()])
    x = x.to(torch.int64)
    return int((x * torch.arange(1, x.numel() + 1, dtype=torch.int64, device=x.device)).sum())


def op(name, fn, nbytes, result=lambda o: o):
    o = timed(name, fn, nbytes)
    print("  checksum", checksum(result(o)), flush=True)
    kernels(fn)


if what & {"motif", "bp", "delfi", "gc-obs", "gc-exp", "gc-cov", "gc-site"}:
    codes, nm = synth_twobit(CLEN, 0)
    ref = D.PackedContig.from_codes(codes, nm, device=dev)
    ws = np.arange(0, CLEN, 1_000_000, dtype=np.int64); we = np.minimum(ws + 1_000_000, CLEN)
tiles = np.arange(0, CLEN + 5000, 5000, dtype=np.int64).clip(max=CLEN)
if "motif" in what:
    op("end_motifs k=4", lambda: D.end_motif_hist(fr, ref, ws, we, k=4, strand_mode=0, quality_threshold=30, pooled=True), 10 * N)
    op("end_motifs k=3 (runtime-K variant)", lambda: D.end_motif_hist(fr, ref, ws, we, k=3, strand_mode=0, quality_threshold=30, pooled=True), 10 * N)
if "bp" in what:
    op("breakpoint_motifs k=6", lambda: D.end_motif_hist(fr, ref, ws, we, k=6, strand_mode=0, quality_threshold=30, pooled=True, breakpoint=True), 10 * N)
if "delfi" in what:
    bs = np.arange(0, CLEN, 100_000, dtype=np.int64); be = np.minimum(bs + 100_000, CLEN)
    op("delfi 100-kb bins", lambda: D.delfi_windows(fr, ref, bs, be, quality_threshold=30), 9 * N + CLEN * 3 // 8)
if "cleavage" in what:
    op("cleavage", lambda: D.cleavage_intervals(fr, tiles[:-1], tiles[1:], CLEN, None, None, 30), 10 * N + 8 * CLEN, lambda o: o[0])
for name in ("depth", "depth-mid"):
    if name in what:
        op(name, lambda: D.depth_intervals(fr, tiles[:-1], tiles[1:], CLEN, None, None, 30, name == "depth-mid"), 9 * N + 4 * CLEN,
           lambda o: o[0])
if "hist" in what:
    op("coverage counts (5-kb intervals)", lambda: D.interval_hist(fr, tiles[:-1], tiles[1:], "midpoint", None, None, 30), 9 * N,
       lambda o: o[0])
    op("coverage counts + pooled length histogram",
       lambda: D.interval_hist(fr, tiles[:-1], tiles[1:], "midpoint", None, None, 30, n_bins=601, pooled="hist"), 9 * N,
       lambda o: torch.cat([o[0], o[1].flatten()]))
    op("per-interval length histograms (frag_length_intervals)",
       lambda: D.interval_hist(fr, tiles[:-1], tiles[1:], "midpoint", None, None, 30, n_bins=601, first_seen=True), 9 * N,
       lambda o: torch.cat([o[0], o[1].flatten(), o[2].flatten().to(torch.int64)]))
for name, step in (("vplot", 5000), ("vplot-dense", 500)):
    if name in what:
        # sites every `step` bp (49 850 at 5 kb), strands alternating, flank 1000, lengths 0..600
        vc = np.arange(step // 2, CLEN, step, dtype=np.int64)
        vf = np.arange(vc.size) % 2 == 1
        made = []
        interval_set = D.IntervalSet
        D.IntervalSet = lambda *a, **k: made.append(interval_set(*a, **k)) or made[-1]   # keep the range scratch
        m = D.vplot_sites(fr, vc, vf, 1000, 0, 600, 30)
        D.IntervalSet = interval_set
        rng = made[-1].scratch[: 2 * vc.size].view(-1, 2)
        cand, events = int((rng[:, 1] - rng[:, 0]).sum()), int(m.sum())
        print(f"{name}: {vc.size} sites, {cand} candidates, {events} events", flush=True)
        op(name, lambda: D.vplot_sites(fr, vc, vf, 1000, 0, 600, 30), 9 * cand)
        print(f"  {events / timed.ms / 1e6:.2f} G events/s over the call", flush=True)
# GC bias: one whole-contig region, lengths 50..500, q 30
if "gc-obs" in what:
    o = D.gc_observed(fr, ref, [0], [CLEN], 50, 500, 30)
    reach = min(fr.max_len, 500) >> 1
    cand = int(torch.searchsorted(st, torch.tensor([CLEN], dtype=torch.int32, device=dev)).item()) - \
        int(torch.searchsorted(st, torch.tensor([-reach], dtype=torch.int32, device=dev)).item())
    print(f"gc-obs: {cand} candidates, {int(o.sum())} counted", flush=True)
    op("gc-obs", lambda: D.gc_observed(fr, ref, [0], [CLEN], 50, 500, 30), 9 * cand)
    print(f"  {cand / timed.ms / 1e6:.2f} G candidates/s over the call", flush=True)


def candidates(lo, hi, reach):
    """Sum over units of the candidate range [lower_bound(lo - reach), lower_bound(hi)) of the start column."""
    a = torch.searchsorted(st, torch.tensor(lo - reach, dtype=torch.int32, device=dev))
    b = torch.searchsorted(st, torch.tensor(hi, dtype=torch.int32, device=dev))
    return int((b - a).sum())


# GC-corrected counts: lengths 50..500, q 30, seeded weights (their values do not change the work)
if what & {"gc-cov", "gc-site"}:
    W = torch.rand((451, 501), generator=g, device=dev, dtype=torch.float64)
if "gc-cov" in what:
    cand = candidates(tiles[:-1], tiles[1:], min(fr.max_len, 500) >> 1)
    c, w = D.gc_weighted_intervals(fr, ref, tiles[:-1], tiles[1:], W, 50, 500, 30)
    print(f"gc-cov: {tiles.size - 1} intervals, {cand} candidates, {int(c.sum())} selected", flush=True)
    op("gc-cov", lambda: D.gc_weighted_intervals(fr, ref, tiles[:-1], tiles[1:], W, 50, 500, 30), 9 * cand,
       lambda o: torch.cat([o[0], o[1].view(torch.int64)]))
    print(f"  {cand / timed.ms / 1e6:.2f} G candidates/s over the call", flush=True)
if "gc-site" in what:
    # sites every 5 kb (49 850), strands alternating, flank 1000
    gc_c = np.arange(2500, CLEN, 5000, dtype=np.int64)
    gc_f = np.arange(gc_c.size) % 2 == 1
    cand = candidates(gc_c - 1000, gc_c + 1001, min(fr.max_len, 500) >> 1)
    c, w = D.gc_weighted_sites(fr, ref, gc_c, gc_f, 1000, W, 50, 500, 30)
    print(f"gc-site: {gc_c.size} sites, {cand} candidates, {int(c.sum())} events", flush=True)
    op("gc-site", lambda: D.gc_weighted_sites(fr, ref, gc_c, gc_f, 1000, W, 50, 500, 30), 9 * cand, lambda o: o[0])
    print(f"  {int(c.sum()) / timed.ms / 1e6:.2f} G events/s over the call", flush=True)
if "gc-exp" in what:
    pairs = sum(max(CLEN - L + 1, 0) for L in range(50, 501))   # (m, L) pairs the kernel walks
    op("gc-exp", lambda: D.gc_expected(ref, [0], [CLEN], 50, 500), 0)
    print(f"  {pairs} (m, L) pairs, {pairs / timed.ms / 1e9:.3f} T pairs/s over the call", flush=True)
if "adjust" in what:
    plan = D.WpsPlan(tiles[:-1], tiles[1:], CLEN, 180, dev)
    wps = plan.run(fr)
    ap = D.AdjustPlan(np.diff(plan.offsets), 1000, True, 21, 2, dev, skip_short=True)
    out = torch.empty(ap.n_total, dtype=torch.float64, device=dev)
    timed("adjust_wps fused (median 1000 + SG 21/2)", lambda: ap.run_rank(wps, 0, out), 4 * plan.n_positions + 8 * ap.n_total)
    print("  checksum", float(out.sum()), "flags", int(ap.run_rank(wps, 0, out)[1].sum()))
    ap0 = D.AdjustPlan(np.diff(plan.offsets), 1000, False, 21, 2, dev, skip_short=True)
    timed("adjust_wps median only", lambda: ap0.run_rank(wps, 0, out), 4 * plan.n_positions + 8 * ap.n_total)
if "spectrum" in what:
    # 20 000 windows x 10 kb (the gene-body workload), periods 120..280; the values do not change the work
    n_win, win, lo_p, hi_p = 20_000, 10_000, 120, 280
    xi = torch.randint(-300, 300, (n_win * win,), generator=g, device=dev, dtype=torch.int32)
    off = np.arange(0, n_win * win + 1, win, dtype=np.int64)
    adds = n_win * win * (hi_p - lo_p + 1)            # fold additions: one per (position, period)
    for name, xs in (("spectrum-i32", xi), ("spectrum-f64", xi.to(torch.float64))):
        op(name, lambda: D.spectrum_segments(xs, off, lo_p, hi_p), xs.numel() * xs.element_size())
        print(f"  {adds / timed.ms / 1e9:.1f} T fold additions/s; shared-memory loads "
              f"{adds * xs.element_size() / timed.ms / 1e9:.1f} TB/s", flush=True)
    del xi
