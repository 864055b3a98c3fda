"""Per-base fragment depth tracks: ``coverage_profile`` / ``multi_coverage_profile``.

An addition with no reference function of that name: the ``coverage`` array of the reference's
``_coverage_and_ends`` (frag/_cleavage_profile.py:33-90) as an output of its own, or with
``midpoint=True`` the number of fragments whose midpoint ``(start + stop) // 2`` falls on each base.
A fragment passes when ``mapq >= quality_threshold`` and ``min_length <= stop - start <= max_length``
(None = unbounded).  The depth runs in the CUDA tile kernel behind ``ftk_depth_tiles_i32``; interval
handling, BAM fetch semantics, writers and errors are those of the cleavage profile drivers.
"""
from __future__ import annotations

import time
from sys import stderr

import numpy as np

from ..io.fragments import as_table
from ..utils import chrom_sizes_to_dict, chrom_sizes_to_list
from ._cleavage_profile import _check_output_file, _read_intervals, _write_tracks
from ._common import group_by_contig, per_fetch

__all__ = ["coverage_profile", "multi_coverage_profile"]

_DEPTH_DTYPE = [("contig", "U16"), ("pos", "i8"), ("depth", "i8")]


def _result(contig, start, values) -> np.ndarray:
    res = np.zeros(len(values), dtype=_DEPTH_DTYPE)
    res["contig"] = contig
    res["pos"] = np.arange(start, start + len(values))
    res["depth"] = values
    return res


def coverage_profile(input_file, chrom_size, contig, start, stop, left=0, right=0, min_length=None, max_length=None,
                     quality_threshold=30, midpoint=False, verbose=0, reference_file=None) -> np.ndarray:
    """Fragment depth of every base of ``contig:[start-left, stop+right)`` (clamped to ``[0, chrom_size)``):
    ('contig', 'pos', 'depth').  Span depth counts the passing fragments with ``start <= pos < stop``;
    ``midpoint=True`` counts those with ``(start + stop) // 2 == pos``."""
    from ..device import depth_intervals
    if verbose:
        start_time = time.time()
    adj_start = max(start - left, 0)
    adj_stop = min(stop + right, chrom_size)
    table = as_table(input_file, reference_file)
    if adj_stop <= adj_start:
        return _result(contig, adj_start, np.zeros(0, np.int64))
    if table.has_read1(contig):   # BAM: what an indexed fetch of the padded region yields
        table = table.fetched(contig, adj_start, adj_stop)
    out, _ = depth_intervals(table.device(contig), [adj_start], [adj_stop], chrom_size, min_length, max_length,
                             quality_threshold, midpoint)
    if verbose:
        stderr.write(f"coverage_profile took {time.time() - start_time} s to complete\n")
    return _result(contig, adj_start, out.cpu().numpy())


def multi_coverage_profile(input_file, interval_file, chrom_sizes, output_file="-", left=0, right=0, min_length=None,
                           max_length=None, quality_threshold=30, midpoint=False, scale_factor=1.0, normalize=False,
                           workers=1, verbose=0, reference_file=None) -> str:
    """Fragment depth tracks over the intervals of a (sorted) BED, expanded by ``left`` / ``right``, clamped and
    merged like ``multi_cleavage_profile``; ``.bw`` / ``.bed.gz`` / ``bedgraph.gz``.  Written value:
    ``depth * scale_factor`` (float64); ``normalize=True`` divides ``scale_factor`` by the number of passing
    fragments in the whole file (the total of ``coverage(normalize=True)``), so ``scale_factor=1e6`` gives
    depth per million fragments."""
    from ..device import depth_intervals
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
    table = as_table(input_file, reference_file)
    if normalize:
        total = _count_intervals(table, [(None, 0, None)], min_length, max_length, "midpoint", quality_threshold)[0]
        scale_factor /= total   # ZeroDivisionError for a file without a passing fragment, like coverage()
    size_dict = dict(header)
    results: list = [None] * len(contigs)
    for contig, idx in group_by_contig(contigs).items():
        s = [starts[i] for i in idx]
        e = [stops[i] for i in idx]

        def run(tab, sel, contig=contig, s=s, e=e):
            if tab.n_fragments(contig) == 0:
                return [np.zeros(max(e[k] - s[k], 0), np.int32) for k in sel]
            out, off = depth_intervals(tab.device(contig), [s[k] for k in sel], [e[k] for k in sel],
                                       size_dict[contig], min_length, max_length, quality_threshold, midpoint)
            host = out.cpu().numpy()
            return [host[off[j]: off[j + 1]] for j in range(len(sel))]

        for i, depth in zip(idx, per_fetch(table, contig, s, e, run)):
            results[i] = depth.astype(np.float64) * scale_factor
    _write_tracks(output_file, header, contigs, starts, results)
    if verbose:
        stderr.write(f"coverage profile took {time.time() - start_time} s to complete\n")
    return output_file
