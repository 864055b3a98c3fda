"""GC-corrected per-base depth tracks: ``gc_corrected_coverage_profile`` / ``multi_gc_corrected_coverage_profile``.

Additions with no reference function of that name: the depth tracks of ``coverage_profile`` with every fragment
weighted by a ``gc_bias`` model, as ``gc_corrected_coverage`` weights its counts (the track deepTools builds with
``correctGCBias`` and then ``bamCoverage``).  The weight table ``W = gc_weights(model)`` is quantised to
``Q = rint(W * 2^32)`` (int64).  A fragment ``[s, e)`` (``L = e - s``) is selected when ``mapq >= quality_threshold``
and ``min_length <= L <= max_length`` (the model's range); it weighs ``Q[L - min_length, g]`` when ``s >= 0``,
``e <= contig length`` and none of its bases is N (g = its C/G bases), 0 otherwise.  The value at a position ``p`` is
``fp64(S(p)) * 2^-32`` with ``S(p)`` the int64 sum of the weights of the selected fragments with ``s <= p < e``
(``midpoint=True``: with ``(s + e) // 2 == p``): exact, exactly 0.0 where no weighted fragment counts, and the same
bits whatever the run or the intervals batched with it.  The sums run in the CUDA kernel behind
``ftk_gc_depth_tiles_f64``; interval handling, BAM fetch semantics and writers are those of ``coverage_profile``.
"""
from __future__ import annotations

import time
from sys import stderr

import numpy as np

from ..io.fragments import as_table
from ..io.reference import open_reference
from ..utils import chrom_sizes_to_dict, chrom_sizes_to_list
from ._cleavage_profile import _check_output_file, _read_intervals, _write_tracks
from ._common import group_by_contig, per_fetch
from ._gc_correct import _model, _warn_missing, gc_weights

__all__ = ["gc_corrected_coverage_profile", "multi_gc_corrected_coverage_profile"]

_DEPTH_DTYPE = [("contig", "U16"), ("pos", "i8"), ("depth", "f8")]


def _result(contig, start, values) -> np.ndarray:
    res = np.zeros(len(values), dtype=_DEPTH_DTYPE)
    res["contig"] = contig
    res["pos"] = np.arange(start, start + len(values))
    res["depth"] = values
    return res


def gc_corrected_coverage_profile(input_file, refseq_file, chrom_size, contig, start, stop, left=0, right=0,
                                  gc_bias=None, gc_regions=None, min_length=None, max_length=None, quality_threshold=30,
                                  midpoint=False, verbose=0, reference_file=None) -> np.ndarray:
    """GC-corrected fragment depth of every base of ``contig:[start-left, stop+right)`` (clamped to
    ``[0, chrom_size)``): ('contig', 'pos', 'depth' float64).  ``gc_bias``: a ``GCBias``, the path of a ``gc-bias``
    table, or None to fit one first over ``gc_regions``; ``min_length`` / ``max_length`` default to the model's range
    (50 and 500 when fitting).  A contig the input or the reference lacks gives zeros, with a ``UserWarning``."""
    from ..device import gc_depth_intervals, require_cuda
    if verbose:
        start_time = time.time()
    model = _model(input_file, refseq_file, gc_bias, gc_regions, min_length, max_length, quality_threshold,
                   reference_file)
    adj_start = max(start - left, 0)
    adj_stop = min(stop + right, chrom_size)
    n = max(adj_stop - adj_start, 0)
    if n == 0:
        return _result(contig, adj_start, np.zeros(0))
    ref = open_reference(refseq_file)
    table = as_table(input_file, reference_file)
    if contig not in set(table.contigs) & set(ref.chroms):
        _warn_missing([contig], "positions", "gc_corrected_coverage_profile")
        return _result(contig, adj_start, np.zeros(n))
    if table.has_read1(contig):   # BAM: what an indexed fetch of the padded region yields
        table = table.fetched(contig, adj_start, adj_stop)
    if table.n_fragments(contig) == 0:
        return _result(contig, adj_start, np.zeros(n))
    dev = require_cuda()
    out, _ = gc_depth_intervals(table.device(contig, dev), ref.device_contig(contig, dev), [adj_start], [adj_stop],
                                chrom_size, gc_weights(model), model.min_length, model.max_length, quality_threshold,
                                midpoint)
    if verbose:
        stderr.write(f"gc_corrected_coverage_profile took {time.time() - start_time} s to complete\n")
    return _result(contig, adj_start, out.cpu().numpy())


def multi_gc_corrected_coverage_profile(input_file, refseq_file, interval_file, chrom_sizes, output_file="-", left=0,
                                        right=0, gc_bias=None, gc_regions=None, min_length=None, max_length=None,
                                        quality_threshold=30, midpoint=False, scale_factor=1.0, normalize=False,
                                        workers=1, verbose=0, reference_file=None) -> str:
    """GC-corrected fragment depth tracks over the intervals of a (sorted) BED, expanded by ``left`` / ``right``,
    clamped and merged like ``multi_coverage_profile``; ``.bw`` / ``.bed.gz`` / ``bedgraph.gz``.  Written value:
    ``depth * scale_factor`` (float64); ``normalize=True`` divides ``scale_factor`` by the number of passing fragments
    in the whole file (plain counts, lengths in the model's range), as ``multi_coverage_profile`` does.  The model is
    given or fitted as for ``gc_corrected_coverage``.  Intervals on contigs the input or the reference lacks are
    written as zeros, with one ``UserWarning``.  ``workers`` is accepted for compatibility (one process per GPU)."""
    from ..device import gc_depth_intervals, require_cuda
    from ._coverage import _count_intervals
    if verbose:
        start_time = time.time()
    if input_file == "-" and interval_file == "-":
        raise ValueError("input_file and site_bed cannot both read from stdin")
    if chrom_sizes is None:
        raise ValueError("chrom_sizes must be specified.")
    header = chrom_sizes_to_list(chrom_sizes)
    chrom_dict = chrom_sizes_to_dict(chrom_sizes)
    contigs, starts, stops = _read_intervals(interval_file, left, right, chrom_dict)
    _check_output_file(output_file, input_file)
    model = _model(input_file, refseq_file, gc_bias, gc_regions, min_length, max_length, quality_threshold,
                   reference_file)
    lo, hi = model.min_length, model.max_length
    ref = open_reference(refseq_file)
    table = as_table(input_file, reference_file)
    if normalize:
        total = _count_intervals(table, [(None, 0, None)], lo, hi, "midpoint", quality_threshold)[0]
        scale_factor /= total   # ZeroDivisionError for a file without a passing fragment, like coverage()
    usable = set(table.contigs) & set(ref.chroms)
    W = gc_weights(model)
    size_dict = dict(header)
    results: list = [None] * len(contigs)
    missing = []
    dev = None
    for contig, idx in group_by_contig(contigs).items():
        s = [starts[i] for i in idx]
        e = [stops[i] for i in idx]
        if contig not in usable:
            missing.append(contig)
            for i in idx:
                results[i] = np.zeros(max(stops[i] - starts[i], 0))
            continue
        dev = require_cuda() if dev is None else dev
        dev_ref = ref.device_contig(contig, dev)

        def run(tab, sel, contig=contig, s=s, e=e, dev_ref=dev_ref):
            if tab.n_fragments(contig) == 0:
                return [np.zeros(max(e[k] - s[k], 0)) for k in sel]
            out, off = gc_depth_intervals(tab.device(contig, dev), dev_ref, [s[k] for k in sel], [e[k] for k in sel],
                                          size_dict[contig], W, lo, hi, quality_threshold, midpoint)
            host = out.cpu().numpy()
            return [host[off[j]: off[j + 1]] for j in range(len(sel))]

        for i, depth in zip(idx, per_fetch(table, contig, s, e, run)):
            results[i] = depth * scale_factor
    _warn_missing(missing, "intervals", "multi_gc_corrected_coverage_profile")
    _write_tracks(output_file, header, contigs, starts, results)
    if verbose:
        stderr.write(f"GC-corrected coverage profile took {time.time() - start_time} s to complete\n")
    return output_file
