"""Nucleosome periodicity spectra from WPS: ``wps_spectrum``.

An addition with no reference function of that name: the gene-body analysis of Snyder et al. (2016), who took the
strength of the ~190 bp nucleosome repeat from a Fourier transform of the long-fragment WPS at periods of 120-280 bp.
Each BED row ``[start, stop)``, clipped to ``[0, contig length)``, is one window (rows may overlap and need not be
sorted; the strand column is ignored, since the magnitude does not change when a series is reversed).  Its series
``x`` is the L-WPS ``multi_wps`` computes for that interval, or (``adjust=True``) the series ``adjust_segments``
returns for it (windows too short for the filters give an empty series, as in ``adjust_wps_genome``).  With
``N = len(x)`` and mean ``mu``, for every integer period ``P``:

    I(P) = |sum_{n<N} (x[n] - mu) exp(-2 pi i (n mod P) / P)|^2 / N        (float64; NaN when N = 0)

WPS, adjustment and spectra stay on the GPU (``WpsPlan``, ``AdjustPlan`` / ``adjust_segments``, and the CUDA kernel
behind ``ftk_spectrum_i32_f64`` / ``ftk_spectrum_f64_f64``); only the ``[windows, periods]`` matrix is downloaded.
"""
from __future__ import annotations

import time
import warnings
from dataclasses import dataclass
from sys import stderr

import numpy as np

from ..io.fragments import as_table
from ..utils import get_intervals
from ._common import check_tsv_output, dist_context, group_by_contig, is_writer, per_fetch, resolve_length_aliases, \
    write_text
from ._multi_wps import _read_header
from ._wps import fetch_window

__all__ = ["wps_spectrum", "WpsSpectrum", "LAST_TIMINGS"]

# wall-clock split of the most recent wps_spectrum call (seconds): decode = file -> columns, compute = uploads +
# kernels + the download of the matrix, write = output file
LAST_TIMINGS: dict = {}


@dataclass
class WpsSpectrum:
    """Periodograms of the BED rows, in input order."""
    intervals: list          # (contig, start, stop, name) as given in the BED
    n: np.ndarray            # int64 [windows]: length of each series (0: empty, a row of NaN)
    periods: np.ndarray      # int64 [periods]: min_period .. max_period
    intensity: np.ndarray    # float64 [windows, periods]: I(P)


def _check_filters(median_window_size, savgol, savgol_window_size, savgol_poly_deg):
    from ..device import savgol_tables
    w = median_window_size
    if isinstance(w, bool) or int(w) != w or w < 2 or w % 2:
        raise ValueError(f"median_window_size must be an even integer >= 2, got {w!r}")
    if savgol:
        savgol_tables(savgol_window_size, savgol_poly_deg)    # ValueError for an even window or a degree >= window


def spectrum_text(res: WpsSpectrum) -> str:
    """The TSV of ``wps_spectrum``: ``contig start stop name n p<P>...``, floats written with ``repr``."""
    head = "contig\tstart\tstop\tname\tn\t" + "\t".join(f"p{p}" for p in res.periods.tolist()) + "\n"
    return head + "".join(f"{c}\t{s}\t{e}\t{name}\t{n}\t" + "\t".join(map(repr, row)) + "\n"
                          for (c, s, e, name), n, row in zip(res.intervals, res.n.tolist(), res.intensity.tolist()))


def wps_spectrum(input_file, site_bed, chrom_sizes=None, output_file=None, min_period=120, max_period=280, adjust=True,
                 median_window_size=1000, savgol=True, savgol_window_size=21, savgol_poly_deg=2, window_size=120,
                 min_length=120, max_length=180, quality_threshold=30, workers=1, verbose=0, fraction_low=None,
                 fraction_high=None, reference_file=None) -> WpsSpectrum:
    """Periodogram of the (adjusted) L-WPS of every BED row at the integer periods ``min_period .. max_period``.

    WPS arguments as for ``multi_wps`` (``chrom_sizes`` is required unless the input is a BAM / CRAM with a header);
    ``adjust`` and the filter arguments as for ``adjust_wps``.  Rows on contigs the sizes do not list become rows of
    NaN with ``n = 0``, with one ``UserWarning``.  ``output_file``: None, ``.tsv``, ``.tsv.gz`` or '-'.  BAM input:
    each window's fragments are those an indexed fetch of its padded WPS window yields, as in ``multi_wps``.  Under
    ``torch.distributed`` every rank computes the rows of its contigs and one all-reduce combines them; each row is
    bit-identical to a one-GPU run.  ``workers`` is accepted for compatibility (one process per GPU)."""
    from ..device import AdjustPlan, require_cuda, spectrum_check, torch
    from .. import device as D
    if verbose:
        start_time = time.time()
    if input_file == "-" and site_bed == "-":
        raise ValueError("input_file and site_bed cannot both read from stdin")
    n_p = spectrum_check(min_period, max_period)
    min_length, max_length = resolve_length_aliases(min_length, max_length, fraction_low, fraction_high)
    if adjust:
        _check_filters(median_window_size, savgol, savgol_window_size, savgol_poly_deg)
    check_tsv_output(output_file, "the WPS spectra")
    t_begin = time.perf_counter()
    intervals = get_intervals(site_bed)
    table = as_table(input_file, reference_file)
    sizes = dict(_read_header(input_file, table, chrom_sizes))
    width = int(round(max_length))

    # the windows clipped to their contig (a contig the sizes lack has length 0), and the length of each series
    lo = np.array([max(iv[1], 0) for iv in intervals], dtype=np.int64)
    hi = np.array([min(iv[2], sizes.get(iv[0], 0)) for iv in intervals], dtype=np.int64)
    n = np.maximum(hi - lo, 0)
    if adjust:
        n = AdjustPlan.output_lengths(n, median_window_size, savgol, savgol_window_size)
    missing = list(dict.fromkeys(iv[0] for iv in intervals if iv[0] not in sizes))

    t = torch()
    dev = require_cuda()
    ctx = dist_context()   # torch.distributed initialised: contigs sharded over the ranks, one all-reduce
    mine = None
    if ctx is not None:
        from ..distributed import owned_contigs
        mine = set(owned_contigs(table, ctx))
    filters = dict(median_window_size=median_window_size, savgol=savgol, savgol_window_size=savgol_window_size,
                   savgol_poly_deg=savgol_poly_deg)
    # rows not computed here stay 0: a contig without fragments has WPS 0 everywhere, so every I(P) is 0
    out = t.zeros((len(intervals), n_p), dtype=t.float64, device=dev)
    t_decode = time.perf_counter() - t_begin
    t_compute = 0.0
    for contig, idx in group_by_contig([iv[0] for iv in intervals]).items():
        idx = [i for i in idx if n[i] > 0]
        if not idx or (mine is not None and contig not in mine):
            continue
        t0 = time.perf_counter()
        table.host(contig)      # lazy tables decode here: keep it out of the compute share
        t1 = time.perf_counter()
        t_decode += t1 - t0
        if table.n_fragments(contig) == 0:
            continue
        size = sizes[contig]

        def run(tab, sel, contig=contig, idx=idx, size=size):
            if not sel or tab.n_fragments(contig) == 0:
                return [None] * len(sel)
            rows = [idx[k] for k in sel]
            plan = D.WpsPlan(lo[rows], hi[rows], size, width, dev)
            x = plan.run(tab.device(contig, dev), int(window_size), min_length, width, quality_threshold)
            off = plan.offsets
            if adjust:
                aplan = AdjustPlan(np.diff(off), median_window_size, savgol, savgol_window_size, savgol_poly_deg, dev,
                                   skip_short=True)
                x, off = D.adjust_segments(x, np.diff(off), plan=aplan, **filters)
            out[t.as_tensor(rows, dtype=t.int64, device=dev)] = D.spectrum_segments(x, off, min_period, max_period)
            return [None] * len(sel)

        # every window is one wps() call of the reference, which fetches from its own padded window
        bam = table.has_read1(contig)
        fetch = [fetch_window(lo[i], hi[i], max_length, size) if bam else (None, None) for i in idx]
        per_fetch(table, contig, [f[0] for f in fetch], [f[1] for f in fetch], run)
        t_compute += time.perf_counter() - t1
    t0 = time.perf_counter()
    if ctx is not None:
        # every row is computed on one rank and is 0 on every other, so summing the fp64 bit patterns as int64
        # moves them exactly: the result is bit-identical to one GPU's
        ctx.all_reduce_sum(out.view(t.int64))
        if not is_writer(ctx):
            output_file = None
    intensity = out.cpu().numpy()
    intensity[n == 0] = np.nan
    t_compute += time.perf_counter() - t0
    if missing:
        warnings.warn(f"wps_spectrum: rows on contigs missing from the chromosome sizes are NaN: {', '.join(missing)}",
                      UserWarning, stacklevel=2)
    res = WpsSpectrum(intervals, n, np.arange(int(min_period), int(max_period) + 1, dtype=np.int64), intensity)
    t0 = time.perf_counter()
    if output_file is not None:
        write_text(output_file, spectrum_text(res))
    t_write = time.perf_counter() - t0
    LAST_TIMINGS.clear()
    LAST_TIMINGS.update(decode=t_decode, compute=t_compute, write=t_write, total=time.perf_counter() - t_begin)
    if verbose:
        stderr.write(f"wps_spectrum took {time.time() - start_time} s to complete\n")
    return res
