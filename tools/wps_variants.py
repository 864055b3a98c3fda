"""Timings of the plain WPS kernel, the fused pass, the unpack kernel and the e2e pipelines
at chr1 scale (CUDA events, min/mean of several launches).  Run on a GPU box:
    python tools/wps_variants.py [n_frag]
"""
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from finaletoolkit_b200 import device as D
from finaletoolkit_b200.packed import PackedFragments
from finaletoolkit_b200.pipeline import StreamedContig
from finaletoolkit_b200.synth import synth_fragments

CLEN = 249_250_621
N = int(sys.argv[1]) if len(sys.argv) > 1 else 80_000_000


def timed(fn, reps=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    for i in range(reps):
        ev[i].record(); fn()
    ev[reps].record(); torch.cuda.synchronize()
    ts = [ev[i].elapsed_time(ev[i + 1]) for i in range(reps)]
    return {"min_ms": min(ts), "mean_ms": float(np.mean(ts))}


def main():
    dev = D.require_cuda("cuda:0")
    st, sp, mq, sd = synth_fragments(CLEN, N, 0)
    fr = D.ContigFragments(st, sp, mq, sd, device=dev, max_len=600)
    edges = np.arange(0, CLEN + 5000, 5000, dtype=np.int64).clip(max=CLEN)
    plan = D.WpsPlan(edges[:-1], edges[1:], CLEN, 180, dev)
    out = torch.empty(plan.n_positions, dtype=torch.int32, device=dev)
    res = {"n_frag": N}
    plan.ranges(fr)
    res["ranges"] = timed(lambda: plan.ranges(fr))
    res["wps"] = timed(lambda: plan.run(fr, out=out, ranges_ready=True))
    cnt = torch.zeros(plan.n_intervals, dtype=torch.int64, device=dev)
    hist = torch.zeros(601, dtype=torch.int64, device=dev)
    res["fused_wps_cov_hist(incl ranges)"] = timed(lambda: plan.run_fused(fr, n_bins=601, out=out, counts=cnt, hist=hist))
    res["fused_wps_cov_nohist(incl ranges)"] = timed(lambda: plan.run_fused(fr, n_bins=0, out=out, counts=cnt))
    ivl = D.IntervalSet(edges[:-1].tolist(), edges[1:].tolist(), dev)
    c2 = torch.zeros(ivl.n, dtype=torch.int64, device=dev); h2 = torch.zeros((1, 601), dtype=torch.int64, device=dev)
    res["separate_cov_hist"] = timed(lambda: D.interval_hist(fr, intersect_policy="midpoint", quality_threshold=30, n_bins=601,
                                                             pooled="hist", ivl_set=ivl, out=(c2, h2, None)))
    print(json.dumps(res), flush=True)
    # pack / unpack
    t0 = time.time(); pk = PackedFragments(st, sp, mq, None); res["host_pack_s"] = time.time() - t0
    res["wire_bytes"] = pk.wire_bytes(); res["raw_blocks"] = pk.n_raw
    d_words = pk.words.to(dev); d_anch = pk.anchors.to(dev); raw = pk.raw_to_device(dev)
    ds = torch.empty(pk.n_blocks * 64, dtype=torch.int32, device=dev); de = torch.empty_like(ds)
    dq = torch.empty(pk.n_blocks * 64, dtype=torch.uint8, device=dev)
    res["unpack"] = timed(lambda: pk.unpack_into(d_words, d_anch, raw, pk.n, ds, de, dq, None, dev))
    assert torch.equal(ds[:N], fr.start) and torch.equal(de[:N], fr.stop) and torch.equal(dq[:N], fr.mapq)
    del d_words, d_anch, ds, de, dq
    print(json.dumps(res), flush=True)
    # e2e pipelines
    h_st = torch.from_numpy(st).pin_memory(); h_sp = torch.from_numpy(sp).pin_memory(); h_mq = torch.from_numpy(mq).pin_memory()
    for chunks in (8, 16, 32):
        pipe = StreamedContig(None, None, None, edges[:-1], edges[1:], CLEN, max_frag_len=600, n_chunks=chunks, device=dev,
                              packed=pk, wps_dtype="int8")
        res[f"e2e_packed_int8_{chunks}chunks"] = dict(timed(pipe.run, reps=6), h2d=pipe.h2d_bytes, d2h=pipe.d2h_bytes)
        del pipe
    pipe = StreamedContig(h_st, h_sp, h_mq, edges[:-1], edges[1:], CLEN, max_frag_len=600, n_chunks=16, device=dev, wps_dtype="int8")
    res["e2e_columns_int8_16chunks"] = dict(timed(pipe.run, reps=6), h2d=pipe.h2d_bytes, d2h=pipe.d2h_bytes)
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
