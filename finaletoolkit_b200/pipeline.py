"""End-to-end pipeline from HOST fragment columns: chunked H2D -> kernels -> D2H, overlapped.

The device kernels finish a chr1-scale shard in well under a millisecond, so the end-to-end
time of the reference-facing call is PCIe.  This module keeps the link busy and the bytes few:

* fragments cross the link PACKED (``packed.PackedFragments``: 3.06 - 4.06 B per fragment instead of the
  9 B of the int32/int32/uint8 columns) and are unpacked on the device (``ftk_unpack_fragments``);
* the contig is cut into ``n_chunks`` runs of intervals; chunk c's fragment slice (plus halo) is
  copied host->device on one stream while chunk c-1 computes on a second stream and chunk c-2's
  WPS drains device->host on a third (PCIe is full duplex), with double-buffered device
  staging and CUDA events for every hand-off;
* each chunk is ONE sweep over its fragments (``ftk_wps_cov_tiles``): WPS + per-interval midpoint
  coverage + the pooled length histogram of the counted fragments;
* WPS travels back as int16 or, with ``wps_dtype="int8"``, as int8 - both exact: a score that does
  not fit raises the overflow flag and the caller reruns one size up.

Plain pinned int32/int32/uint8 columns are accepted too (9 B per fragment on the wire).
"""
from __future__ import annotations

import numpy as np

from .device import WpsPlan, _launch, none_to_ftk, require_cuda, torch
from .packed import PACK_BLOCK, PackedFragments

__all__ = ["StreamedContig"]


class StreamedContig:
    """Streamed L-WPS (+ coverage + length histogram) of one contig from pinned host columns.

    ``ivl_start/ivl_stop``: intervals sorted by start (e.g. ``multi_wps`` windows; gaps and overlaps
    are fine).  Outputs (pinned host tensors): ``h_wps`` (int16 or int8, all intervals back to back;
    ``offsets`` as in ``WpsPlan``), ``h_cov`` (int64 per interval: fragments whose midpoint lies in
    the interval, frag/_coverage.py:117-130), ``h_hist`` (int64[1, n_bins]: lengths of the counted
    fragments, one entry per (interval, fragment) pair), ``h_total`` (= ``h_cov.sum()``).
    The coverage predicate defaults to ``quality_threshold`` and no length window.
    """

    def __init__(self, h_start, h_stop, h_mapq, ivl_start, ivl_stop, chrom_size, window_size=120,
                 min_length=120, max_length=180, quality_threshold=30, max_frag_len=None, n_chunks=8,
                 device=None, coverage=True, length_hist=True, wps_dtype="int16", packed: PackedFragments | None = None,
                 cov_min_length=None, cov_max_length=None, cov_quality_threshold=None):
        t = torch()
        self.device = require_cuda(device)
        if wps_dtype not in ("int16", "int8"):
            raise ValueError("wps_dtype must be 'int16' or 'int8'")
        self.wps_dtype = wps_dtype
        wire = t.int16 if wps_dtype == "int16" else t.int8
        self.packed = packed
        if packed is None:
            for h in (h_start, h_stop, h_mapq):
                if not h.is_pinned():
                    raise ValueError("host columns must be pinned (tensor.pin_memory())")
            self.h_start, self.h_stop, self.h_mapq = h_start, h_stop, h_mapq
            st_np = h_start.numpy()
            n = st_np.shape[0]
            if max_frag_len is None:
                max_frag_len = int((h_stop.numpy().astype(np.int64) - st_np).max()) if n else 0
        else:
            n = packed.n
            if max_frag_len is None:
                max_frag_len = packed.max_len
        self.n_frag = n
        self.max_frag_len = int(max_frag_len)
        self.params = (int(window_size), min_length, int(max_length), int(quality_threshold))
        self.cov_params = (cov_min_length, cov_max_length,
                           int(quality_threshold if cov_quality_threshold is None else cov_quality_threshold))
        self.fused = bool(coverage or length_hist)
        s = np.asarray(ivl_start, dtype=np.int64); e = np.asarray(ivl_stop, dtype=np.int64)
        n_ivl = len(s)
        self.n_ivl = n_ivl
        n_chunks = max(1, min(int(n_chunks), max(n_ivl, 1)))
        bounds = np.linspace(0, n_ivl, n_chunks + 1).astype(np.int64)
        ln = np.maximum(e - s, 0)
        self.offsets = np.zeros(n_ivl + 1, np.int64); np.cumsum(ln, out=self.offsets[1:])
        self.n_positions = int(self.offsets[-1])
        halo = max(self.max_frag_len, int(max_length) + int(window_size)) + 2
        self.chunks = []
        for c in range(n_chunks):
            i0, i1 = int(bounds[c]), int(bounds[c + 1])
            if i1 <= i0:
                continue
            p_lo, p_hi = int(s[i0:i1].min()), int(e[i0:i1].max())
            if packed is None:
                f0 = int(np.searchsorted(st_np, p_lo - halo, side="left")) & ~(PACK_BLOCK - 1)
                f1 = int(np.searchsorted(st_np, p_hi + halo, side="left"))
            else:   # block granularity: first_start[b] = start of block b's first fragment
                b0 = max(int(np.searchsorted(packed.first_start, p_lo - halo, side="right")) - 1, 0)
                b1 = int(np.searchsorted(packed.first_start, p_hi + halo, side="left"))
                f0, f1 = b0 * PACK_BLOCK, min(n, b1 * PACK_BLOCK)
            f1 = max(f1, f0)
            plan = WpsPlan(s[i0:i1], e[i0:i1], int(chrom_size), int(max_length), self.device)
            self.chunks.append(dict(i0=i0, i1=i1, f0=f0, f1=f1, plan=plan, out_off=int(self.offsets[i0]),
                                    n_pos=plan.n_positions))
        max_f = max([c["f1"] - c["f0"] for c in self.chunks] + [0]) + PACK_BLOCK
        max_f = (max_f + PACK_BLOCK - 1) // PACK_BLOCK * PACK_BLOCK
        max_p = max([c["n_pos"] for c in self.chunks] + [1])
        self.d_start = [t.empty(max_f, dtype=t.int32, device=self.device) for _ in range(2)]
        self.d_stop = [t.empty(max_f, dtype=t.int32, device=self.device) for _ in range(2)]
        self.d_mapq = [t.empty(max_f, dtype=t.uint8, device=self.device) for _ in range(2)]
        if packed is not None:
            self.d_words = [t.empty(max_f // PACK_BLOCK * packed.words_per_block, dtype=t.int32, device=self.device)
                            for _ in range(2)]
            self.d_anchors = [t.empty(max_f // PACK_BLOCK, dtype=t.int32, device=self.device) for _ in range(2)]
            self.d_raw = packed.raw_to_device(self.device)
        self.d_out = [t.empty(max_p, dtype=wire, device=self.device) for _ in range(2)]
        self.d_flag = t.zeros(1, dtype=t.int32, device=self.device)
        self.n_bins = (self.max_frag_len + 1) if length_hist else 0
        self.d_cov = t.zeros(max(n_ivl, 1), dtype=t.int64, device=self.device)
        self.d_hist = t.zeros((1, max(self.n_bins, 1)), dtype=t.int64, device=self.device)
        self.h_wps = t.empty(max(self.n_positions, 1), dtype=wire).pin_memory()
        self.h_cov = t.empty(max(n_ivl, 1), dtype=t.int64).pin_memory()
        self.h_hist = t.empty((1, max(self.n_bins, 1)), dtype=t.int64).pin_memory()
        self.h_total = t.zeros(1, dtype=t.int64)
        self.h_flag = t.zeros(1, dtype=t.int32).pin_memory()
        self.s_in, self.s_comp, self.s_out = (t.cuda.Stream(self.device) for _ in range(3))
        self.ev_in = [t.cuda.Event() for _ in range(2)]
        self.ev_comp = [t.cuda.Event() for _ in range(2)]
        self.ev_out = [t.cuda.Event() for _ in range(2)]
        if packed is None:
            self.h2d_bytes = sum((c["f1"] - c["f0"]) * 9 for c in self.chunks)
        else:
            self.h2d_bytes = sum(packed.wire_bytes(c["f0"], c["f1"]) for c in self.chunks) + packed.raw_bytes()
        self.d2h_bytes = self.n_positions * (2 if wps_dtype == "int16" else 1) + n_ivl * 8 + self.n_bins * 8 + 4
        self.kernel_launches = 0
        # The pass is a fixed DAG of copies and kernels over fixed buffers: after one eager pass it is
        # captured as a CUDA graph and replayed (no per-chunk host work, no launch gaps between the ~10 nodes
        # of a chunk).  FTK_PIPE_GRAPH=0 keeps the eager three-stream form.
        import os
        self.use_graph = os.environ.get("FTK_PIPE_GRAPH", "1") != "0"
        self._graph = None
        self._warm = False

    def _stage_in(self, c, b):
        """H2D of chunk c's fragment slice into staging set b (on s_in)."""
        f0, f1 = c["f0"], c["f1"]
        nf = f1 - f0
        if nf == 0:
            return
        if self.packed is None:
            self.d_start[b][:nf].copy_(self.h_start[f0:f1], non_blocking=True)
            self.d_stop[b][:nf].copy_(self.h_stop[f0:f1], non_blocking=True)
            self.d_mapq[b][:nf].copy_(self.h_mapq[f0:f1], non_blocking=True)
        else:
            nb = (nf + PACK_BLOCK - 1) // PACK_BLOCK
            b0 = f0 // PACK_BLOCK
            wpb = self.packed.words_per_block
            self.d_words[b][: nb * wpb].copy_(self.packed.words[b0 * wpb: (b0 + nb) * wpb], non_blocking=True)
            self.d_anchors[b][:nb].copy_(self.packed.anchors[b0: b0 + nb], non_blocking=True)

    def run(self):
        """One end-to-end pass; returns after every result is in the pinned host buffers."""
        t = torch()
        with t.cuda.device(self.device):     # the graph is captured and replayed on the buffers' device
            if self.use_graph and self._warm:
                if self._graph is None:
                    g = t.cuda.CUDAGraph()
                    cap = t.cuda.Stream(self.device)
                    cap.wait_stream(t.cuda.current_stream(self.device))
                    with t.cuda.graph(g, stream=cap):
                        self._enqueue()
                    self._graph = g
                self._graph.replay()
            else:
                self._enqueue()
                self._warm = True
        t.cuda.current_stream(self.device).synchronize()
        if int(self.h_flag[0]):
            raise OverflowError(f"WPS does not fit {self.wps_dtype} on this input; rerun with "
                                + ("wps_dtype='int16'" if self.wps_dtype == "int8" else "the int32 path (WpsPlan.run)"))
        self.h_total[0] = int(self.h_cov[: self.n_ivl].sum()) if self.n_ivl else 0
        return self.h_wps, self.h_cov, self.h_hist, self.h_total

    def _enqueue(self):
        """Put one pass on the streams (no host synchronisation; capturable)."""
        t = torch()
        W, lo, hi, q = self.params
        c_lo, c_hi, c_q = self.cov_params
        kind = 1 if self.wps_dtype == "int16" else 2
        wps_tiles = "ftk_wps_tiles_i16" if self.wps_dtype == "int16" else "ftk_wps_tiles_i8"
        cur = t.cuda.current_stream(self.device)
        for s_ in (self.s_in, self.s_comp, self.s_out):
            s_.wait_stream(cur)
        with t.cuda.stream(self.s_comp):
            self.d_cov.zero_(); self.d_hist.zero_(); self.d_flag.zero_()
        launches = 0
        for k, c in enumerate(self.chunks):
            b = k & 1
            nf = c["f1"] - c["f0"]
            with t.cuda.stream(self.s_in):
                if k >= 2:
                    self.s_in.wait_event(self.ev_comp[b])        # staging buffer b consumed
                self._stage_in(c, b)
                self.ev_in[b].record(self.s_in)
            with t.cuda.stream(self.s_comp):
                self.s_comp.wait_event(self.ev_in[b])
                if k >= 2:
                    self.s_comp.wait_event(self.ev_out[b])       # output buffer b drained
                if self.packed is not None and nf:
                    self.packed.unpack_into(self.d_words[b], self.d_anchors[b], self.d_raw, nf, self.d_start[b],
                                            self.d_stop[b], self.d_mapq[b], None, self.device)
                    launches += 1
                plan = c["plan"]
                if plan.n_tiles:
                    fs, fe, mq = self.d_start[b].data_ptr(), self.d_stop[b].data_ptr(), self.d_mapq[b].data_ptr()
                    if self.packed is not None and not self.packed.has_mapq:
                        mq = 0
                    if self.fused:
                        _launch(
                            self.device, "ftk_wps_cov_tiles", fs, fe, mq, nf, self.max_frag_len,
                            plan.tile_p0.data_ptr(), plan.tile_len.data_ptr(), plan.tile_mid_lo.data_ptr(),
                            plan.tile_mid_hi.data_ptr(), plan.tile_out_off.data_ptr(), plan.tile_ivl.data_ptr(),
                            plan.n_tiles, W, none_to_ftk(lo), hi, q, none_to_ftk(c_lo), none_to_ftk(c_hi), c_q,
                            self.n_bins, 0, plan.scratch.data_ptr(), kind, self.d_out[b].data_ptr(),
                            self.d_flag.data_ptr(), self.d_cov[c["i0"]:].data_ptr(),
                            self.d_hist.data_ptr() if self.n_bins else 0)
                    else:
                        _launch(
                            self.device, wps_tiles, fs, fe, mq, nf, plan.tile_p0.data_ptr(), plan.tile_len.data_ptr(),
                            plan.tile_mid_lo.data_ptr(), plan.tile_mid_hi.data_ptr(), plan.tile_out_off.data_ptr(),
                            plan.n_tiles, W, none_to_ftk(lo), hi, q, 0, plan.scratch.data_ptr(),
                            self.d_out[b].data_ptr(), self.d_flag.data_ptr())
                    launches += 2
                self.ev_comp[b].record(self.s_comp)
            with t.cuda.stream(self.s_out):
                self.s_out.wait_event(self.ev_comp[b])
                if c["n_pos"]:
                    self.h_wps[c["out_off"]: c["out_off"] + c["n_pos"]].copy_(self.d_out[b][:c["n_pos"]], non_blocking=True)
                self.ev_out[b].record(self.s_out)
        with t.cuda.stream(self.s_out):
            self.s_out.wait_stream(self.s_comp)
            self.h_cov.copy_(self.d_cov, non_blocking=True)
            self.h_hist.copy_(self.d_hist, non_blocking=True)
            self.h_flag.copy_(self.d_flag, non_blocking=True)
        cur.wait_stream(self.s_out)
        cur.wait_stream(self.s_in)
        cur.wait_stream(self.s_comp)
        self.kernel_launches = launches
