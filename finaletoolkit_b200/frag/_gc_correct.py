"""The fragment GC model applied: ``gc_corrected_coverage`` and ``gc_corrected_profile``.

Additions with no reference function of that name.  Each fragment is weighted by ``1 / ratio[L, g]`` of a ``gc_bias``
model (Benjamini & Speed 2012; Griffin's GC-corrected profiles), with no smoothing of the model.  The weight table
``W`` has the model's shape; ``W[i, g] = 1 / ratio[i, g]`` where the ratio is finite and positive, 0 elsewhere.
A fragment ``[s, e)`` (``L = e - s``, midpoint ``m = (s + e) // 2``) is selected when ``mapq >= quality_threshold``
and ``min_length <= L <= max_length`` and ``m`` passes the position test (in an interval, or within ``flank`` of a
site centre).  Every selected fragment adds 1 to ``count``; it adds ``W[L - min_length, g]`` to ``corrected`` when
``s >= 0``, ``e <= contig length`` and none of its bases is N (the placement rule ``gc_bias`` counts by; g = its C/G
bases).  The counting runs in the CUDA kernels behind ``ftk_gc_weighted_intervals_f64`` and
``ftk_gc_weighted_sites_f64``.
"""
from __future__ import annotations

import os
import time
import warnings
from dataclasses import dataclass
from sys import stderr
from typing import NamedTuple

import numpy as np

from ..io.fragments import as_table
from ..io.reference import open_reference
from ..utils import get_intervals
from ._common import check_tsv_output, dist_context, group_by_contig, is_writer, per_fetch, write_text
from ._gc_bias import GCBias, gc_bias as fit_gc_bias, read_gc_bias
from ._vplot import _read_sites

__all__ = ["gc_corrected_coverage", "gc_corrected_profile", "GCCoverageResult", "GCSiteProfile", "gc_weights"]


class GCCoverageResult(NamedTuple):
    contig: str
    start: int
    stop: int
    name: str
    count: int          # selected fragments whose midpoint lies in [start, stop)
    corrected: float    # their GC weights summed


@dataclass
class GCSiteProfile:
    """Midpoint counts by offset ``-flank .. flank`` from the site centres, summed over ``n_sites`` sites (those on
    contigs both the input and the reference hold)."""
    count: np.ndarray       # int64 [2 * flank + 1]
    corrected: np.ndarray   # float64 [2 * flank + 1]
    flank: int
    n_sites: int


def gc_weights(model: GCBias) -> np.ndarray:
    """``1 / model.ratio`` where the ratio is finite and positive, 0 elsewhere (float64, the model's shape)."""
    r = np.asarray(model.ratio, np.float64)
    w = np.zeros(r.shape, np.float64)
    ok = np.isfinite(r) & (r > 0)
    w[ok] = 1.0 / r[ok]
    return w


def _model(input_file, refseq_file, gc_bias, gc_regions, min_length, max_length, quality_threshold,
           reference_file) -> GCBias:
    """The model given (a ``GCBias`` or the path of a ``gc-bias`` table), or one fitted over ``gc_regions``."""
    if gc_bias is None:
        return fit_gc_bias(input_file, refseq_file, gc_regions, min_length=50 if min_length is None else min_length,
                           max_length=500 if max_length is None else max_length,
                           quality_threshold=quality_threshold, reference_file=reference_file)
    if gc_regions is not None:
        raise ValueError("gc_regions applies only when the model is fitted here (gc_bias=None)")
    if isinstance(gc_bias, GCBias):
        model = gc_bias
    elif isinstance(gc_bias, (str, os.PathLike)):
        model = read_gc_bias(gc_bias)
    else:
        raise TypeError(f"gc_bias must be a GCBias, the path of a gc-bias table or None, got {type(gc_bias)}")
    for name, given, have in (("min_length", min_length, model.min_length), ("max_length", max_length,
                                                                               model.max_length)):
        if given is not None and int(given) != have:
            raise ValueError(f"{name}={given} differs from the GC model's {name} {have}")
    return model


def _warn_missing(missing, what, where):
    if missing:
        warnings.warn(f"{where}: {what} on contigs that the input or the reference lacks count 0: "
                      f"{', '.join(missing)}", UserWarning, stacklevel=3)


def gc_corrected_coverage(input_file, refseq_file, interval_file, output_file=None, gc_bias=None, gc_regions=None,
                          min_length=None, max_length=None, quality_threshold=30, workers=1, verbose=0,
                          reference_file=None) -> list:
    """Plain and GC-corrected fragment counts of every BED interval, in input order.

    A fragment counts in an interval when its midpoint lies in ``[start, stop)``; intervals may overlap and need not
    be sorted.  ``gc_bias``: a ``GCBias``, the path of a ``gc-bias`` table, or None to fit one first with ``gc_bias``
    on the same input over ``gc_regions`` (BED; default the whole contigs) with the same ``quality_threshold``.
    ``min_length`` / ``max_length`` default to the model's range (50 and 500 when fitting).  Intervals on contigs the
    input or the reference lacks count 0, with one ``UserWarning``.  ``output_file``: None, ``.tsv``, ``.tsv.gz`` or
    '-' (header ``contig start stop name count corrected``).  BAM input: each interval's fragments are those an
    indexed fetch of the interval yields.  ``workers`` is accepted for compatibility (one process per GPU)."""
    from ..device import gc_weighted_intervals, gc_weights_to_device, require_cuda
    if verbose:
        start_time = time.time()
    check_tsv_output(output_file, "the GC-corrected counts")
    intervals = get_intervals(interval_file)
    model = _model(input_file, refseq_file, gc_bias, gc_regions, min_length, max_length, quality_threshold,
                   reference_file)
    lo, hi = model.min_length, model.max_length
    ref = open_reference(refseq_file)
    table = as_table(input_file, reference_file)
    usable = set(table.contigs) & set(ref.chroms)
    ctx = dist_context()   # torch.distributed initialised: contigs sharded over the ranks, one all-reduce
    mine = None
    if ctx is not None:
        from ..distributed import owned_contigs
        mine = set(owned_contigs(table, ctx))
    dev = require_cuda()
    W = gc_weights_to_device(gc_weights(model), model.ratio.shape, dev)
    counts = np.zeros(len(intervals), np.int64)
    corrected = np.zeros(len(intervals), np.float64)
    missing = []
    for contig, idx in group_by_contig([iv[0] for iv in intervals]).items():
        if contig not in usable:
            missing.append(contig)
            continue
        if (mine is not None and contig not in mine) or table.n_fragments(contig) == 0:
            continue
        s, e = [intervals[i][1] for i in idx], [intervals[i][2] for i in idx]
        dev_ref = ref.device_contig(contig, dev)

        def run(tab, sel, contig=contig, s=s, e=e, dev_ref=dev_ref):
            if tab.n_fragments(contig) == 0:
                return [(0, 0.0)] * len(sel)
            c, w = gc_weighted_intervals(tab.device(contig, dev), dev_ref, [s[k] for k in sel], [e[k] for k in sel], W,
                                         lo, hi, quality_threshold)
            return list(zip(c.cpu().tolist(), w.cpu().tolist()))

        # the region handed to the fetch is the interval itself
        for i, (c, w) in zip(idx, per_fetch(table, contig, s, e, run)):
            counts[i], corrected[i] = c, w
    _warn_missing(missing, "intervals", "gc_corrected_coverage")
    if ctx is not None:
        import torch
        # each interval is counted on one rank and is 0 on every other, so summing the fp64 bit patterns as int64
        # moves them exactly: the result is bit-identical to one GPU's
        buf = torch.from_numpy(np.stack([counts, corrected.view(np.int64)])).to(dev)
        ctx.all_reduce_sum(buf)
        host = buf.cpu().numpy()
        counts, corrected = host[0].copy(), host[1].copy().view(np.float64)
        if not is_writer(ctx):
            output_file = None
    res = [GCCoverageResult(c, s, e, n, int(k), float(w))
           for (c, s, e, n), k, w in zip(intervals, counts.tolist(), corrected.tolist())]
    if output_file is not None:
        write_text(output_file, "contig\tstart\tstop\tname\tcount\tcorrected\n" +
                   "".join(f"{r.contig}\t{r.start}\t{r.stop}\t{r.name}\t{r.count}\t{r.corrected!r}\n" for r in res))
    if verbose:
        stderr.write(f"gc_corrected_coverage took {time.time() - start_time} s to complete\n")
    return res


def gc_corrected_profile(input_file, refseq_file, site_bed, output_file=None, flank=1000, gc_bias=None,
                         gc_regions=None, min_length=None, max_length=None, quality_threshold=30, workers=1, verbose=0,
                         reference_file=None) -> GCSiteProfile:
    """Plain and GC-corrected fragment-midpoint profiles around the sites of ``site_bed``, summed over the sites.

    Sites are read as ``vplot`` reads them: centre ``(start + stop) // 2``, mirrored when column 6 is '-'.  A
    selected fragment whose midpoint ``m`` lies within ``flank`` of a centre ``c`` adds at offset ``m - c``
    (``c - m`` for '-' sites), once per such site.  ``gc_bias``, ``gc_regions``, ``min_length`` / ``max_length`` and
    missing contigs are as for ``gc_corrected_coverage``.  ``output_file``: None, ``.tsv``, ``.tsv.gz`` or '-' (header
    ``offset count corrected``).  BAM input: each site's fragments are those an indexed fetch of
    ``[c - flank, c + flank + 1)`` yields.  The corrected sums are fp64 atomics on the GPU, so their last bits may
    vary between runs.  ``workers`` is accepted for compatibility (one process per GPU)."""
    from ..device import VPLOT_MAX_FLANK, gc_weighted_sites, gc_weights_to_device, require_cuda, torch
    if verbose:
        start_time = time.time()
    if input_file == "-" and site_bed == "-":
        raise ValueError("input_file and site_bed cannot both read from stdin")
    if isinstance(flank, bool) or int(flank) != flank or not 0 <= int(flank) <= VPLOT_MAX_FLANK:
        raise ValueError(f"flank must be an integer in [0, {VPLOT_MAX_FLANK}], got {flank!r}")
    flank = int(flank)
    check_tsv_output(output_file, "the GC-corrected profile")
    contigs, centers, flips = _read_sites(site_bed)
    model = _model(input_file, refseq_file, gc_bias, gc_regions, min_length, max_length, quality_threshold,
                   reference_file)
    lo, hi = model.min_length, model.max_length
    ref = open_reference(refseq_file)
    table = as_table(input_file, reference_file)
    usable = set(table.contigs) & set(ref.chroms)
    ctx = dist_context()   # torch.distributed initialised: contigs sharded over the ranks, one all-reduce
    held = set(usable)
    if ctx is not None:
        from ..distributed import owned_contigs
        held &= set(owned_contigs(table, ctx))
    t = torch()
    dev = require_cuda()
    W = gc_weights_to_device(gc_weights(model), model.ratio.shape, dev)
    acc = (t.zeros(2 * flank + 1, dtype=t.int64, device=dev), t.zeros(2 * flank + 1, dtype=t.float64, device=dev))
    missing, n_sites = [], 0
    for contig, idx in group_by_contig(contigs).items():
        if contig not in usable:
            missing.append(contig)
            continue
        n_sites += len(idx)
        if contig not in held or table.n_fragments(contig) == 0:
            continue
        c = [centers[i] for i in idx]
        f = [flips[i] for i in idx]
        dev_ref = ref.device_contig(contig, dev)

        def run(tab, sel, contig=contig, c=c, f=f, dev_ref=dev_ref):
            if tab.n_fragments(contig):
                gc_weighted_sites(tab.device(contig, dev), dev_ref, [c[k] for k in sel], [f[k] for k in sel], flank, W,
                                  lo, hi, quality_threshold, out=acc)
            return [None] * len(sel)

        # the region an indexed fetch is asked for: the site's window, clamped at 0
        per_fetch(table, contig, [max(x - flank, 0) for x in c], [x + flank + 1 for x in c], run)
    _warn_missing(missing, "sites", "gc_corrected_profile")
    count, corr = acc[0].cpu().numpy().astype(np.int64), acc[1].cpu().numpy().astype(np.float64)
    if ctx is not None:
        # one fp64 all-reduce of both rows (counts below 2^53 are exact in fp64)
        buf = t.from_numpy(np.stack([count.astype(np.float64), corr])).to(dev)
        ctx.all_reduce_sum(buf)
        host = buf.cpu().numpy()
        count, corr = host[0].astype(np.int64), host[1].copy()
        if not is_writer(ctx):
            output_file = None
    res = GCSiteProfile(count, corr, flank, n_sites)
    if output_file is not None:
        write_text(output_file, "offset\tcount\tcorrected\n" +
                   "".join(f"{d}\t{k}\t{w!r}\n" for d, k, w in zip(range(-flank, flank + 1), count.tolist(),
                                                                    corr.tolist())))
    if verbose:
        stderr.write(f"gc_corrected_profile took {time.time() - start_time} s to complete\n")
    return res
