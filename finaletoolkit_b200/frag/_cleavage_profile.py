"""Cleavage profile (Zhou et al., 2022) - API mirror of reference frag/_cleavage_profile.py.

``_coverage_and_ends`` + the proportion step (frag/_cleavage_profile.py:33-90, 190-217) run in the
CUDA tile kernel behind ``ftk_cleavage_tiles_f64``; the drivers (interval expansion / merging,
writers, errors) follow the reference.
"""
from __future__ import annotations

import time
import warnings
from sys import stderr, stdin

import numpy as np

from ..io import bigwig as pbw
from ..io.textout import GzipTextWriter
from ..io.fragments import as_table
from ..utils import chrom_sizes_to_dict, chrom_sizes_to_list
from ._common import group_by_contig, per_fetch, resolve_length_aliases

__all__ = ["cleavage_profile", "multi_cleavage_profile"]

_CLEAVAGE_DTYPE = [("contig", "U16"), ("pos", "i8"), ("proportion", "f8")]


def _result(contig, start, values) -> np.ndarray:
    res = np.zeros(len(values), dtype=_CLEAVAGE_DTYPE)
    res["contig"] = contig
    res["pos"] = np.arange(start, start + len(values))
    res["proportion"] = values
    return res


def cleavage_profile(input_file, chrom_size, contig, start, stop, left=0, right=0, min_length=None,
                     max_length=None, quality_threshold=30, verbose=0, fraction_low=None, fraction_high=None,
                     reference_file=None) -> np.ndarray:
    """Cleavage proportion (percent) over ``contig:[start-left, stop+right)``: ('contig','pos','proportion')."""
    from ..device import cleavage_intervals
    if verbose:
        start_time = time.time()
    min_length, max_length = resolve_length_aliases(min_length, max_length, fraction_low, fraction_high)
    adj_start = max(start - left, 0)
    adj_stop = min(stop + right, chrom_size)
    table = as_table(input_file, reference_file)
    if adj_stop <= adj_start:
        return _result(contig, adj_start, np.zeros(0))
    if table.has_read1(contig):   # BAM: what an indexed fetch of the padded region yields (:193-202)
        table = table.fetched(contig, adj_start, adj_stop)
    out, _ = cleavage_intervals(table.device(contig), [adj_start], [adj_stop], chrom_size, min_length, max_length,
                                quality_threshold)
    if verbose:
        stderr.write(f"cleavage_profile took {time.time() - start_time} s to complete\n")
    return _result(contig, adj_start, out.cpu().numpy())


def _read_intervals(interval_file, left, right, chrom_dict):
    """frag/_cleavage_profile.py:411-449: expand, clamp, merge overlapping neighbours."""
    contigs, starts, stops = [], [], []
    bed = stdin if interval_file == "-" else open(interval_file)
    try:
        prev_contig, prev_start, prev_stop = None, 0, 0
        for line in bed:
            contents = line.split()
            contig = contents[0].strip()
            start, stop = int(contents[1]), int(contents[2])
            if contig not in chrom_dict:
                warnings.warn(f"Skipping interval {contig}:{start}-{stop} from interval_file "
                              f"({contig} not in chrom_sizes)", UserWarning)
                continue
            start = max(0, start - left)
            stop = min(stop + right, chrom_dict[contig])
            if prev_contig == contig and start < prev_stop:
                prev_stop = max(prev_stop, stop)
            else:
                contigs.append(prev_contig); starts.append(prev_start); stops.append(prev_stop)
                prev_contig, prev_start, prev_stop = contig, start, stop
        contigs.append(prev_contig); starts.append(prev_start); stops.append(prev_stop)
    finally:
        if interval_file != "-":
            bed.close()
    return contigs[1:], starts[1:], stops[1:]


def _check_output_file(output_file, input_file):
    """``output_file`` must be None or a ``.bw`` / ``.bed.gz`` / ``bedgraph.gz`` path or '-'."""
    if isinstance(output_file, str):
        if not (output_file.endswith(".bw") or output_file.endswith(".bed.gz") or output_file.endswith("bedgraph.gz")
                or output_file == "-"):
            raise ValueError("output_file can only have suffix .bw, .bedgraph.gz, or .bed.gz.")
    elif output_file is not None:
        raise TypeError(f'output_file is unsupported type "{type(input_file)}". output_file should be a string '
                        "specifying the path of the file to output scores to.")


def _write_tracks(output_file, header, contigs, starts, results):
    """Per-base values of every interval (float64 arrays) as bigWig entries (``.bw``) or gzipped bedGraph lines."""
    if isinstance(output_file, str):
        if output_file.endswith(".bw"):
            with pbw.open(output_file, "w") as bigwig:
                bigwig.addHeader(header)
                for contig, start, scores in zip(contigs, starts, results):
                    if len(scores) == 0:
                        continue
                    try:
                        bigwig.addEntries(contig, max(start, 0), values=scores.astype(np.float64), step=1, span=1)
                    except RuntimeError as e:  # frag/_cleavage_profile.py:472-483
                        stderr.write(f"{contig}:{start}-{start + len(scores)}\n")
                        stderr.write("invalid or out of order interval encountered. Skipping to next.\n")
                        stderr.write(f"captured error:\n{e}\n")
                        continue
        else:
            with GzipTextWriter(output_file) as bedgraph:   # float text stays Python's repr; deflate is threaded
                for contig, start, scores in zip(contigs, starts, results):
                    pos = max(start, 0)
                    bedgraph.write("".join(f"{contig}\t{p}\t{p + 1}\t{v}\n"
                                           for p, v in zip(range(pos, pos + len(scores)), scores.tolist())))


def multi_cleavage_profile(input_file, interval_file, chrom_sizes, left=0, right=0, min_length=None,
                           max_length=None, quality_threshold=30, output_file="-", workers=1, verbose=0,
                           fraction_low=None, fraction_high=None, reference_file=None) -> str:
    """Cleavage profiles over the intervals of a (sorted) BED; ``.bw`` / ``.bed.gz`` / ``bedgraph.gz``."""
    from ..device import cleavage_intervals
    if verbose:
        start_time = time.time()
    min_length, max_length = resolve_length_aliases(min_length, max_length, fraction_low, fraction_high)
    if input_file == "-" and interval_file == "-":
        raise ValueError("input_file and site_bed cannot both read from stdin")
    if chrom_sizes is None:
        raise ValueError("chrom_sizes must be specified.")
    header = chrom_sizes_to_list(chrom_sizes)
    chrom_dict = chrom_sizes_to_dict(chrom_sizes)
    contigs, starts, stops = _read_intervals(interval_file, left, right, chrom_dict)
    _check_output_file(output_file, input_file)
    table = as_table(input_file, reference_file)
    size_dict = dict(header)
    results: list = [None] * len(contigs)
    for contig, idx in group_by_contig(contigs).items():
        # cleavage_profile() re-clamps each interval (left = right = 0 here, frag/_cleavage_profile.py:352-353)
        s = [max(starts[i], 0) for i in idx]
        e = [min(stops[i], size_dict[contig]) for i in idx]

        def run(tab, sel, contig=contig, s=s, e=e):
            if tab.n_fragments(contig) == 0:
                return [np.zeros(max(e[k] - s[k], 0)) for k in sel]
            out, off = cleavage_intervals(tab.device(contig), [s[k] for k in sel], [e[k] for k in sel],
                                          size_dict[contig], min_length, max_length, quality_threshold)
            host = out.cpu().numpy()
            return [host[off[j]: off[j + 1]] for j in range(len(sel))]

        for i, scores in zip(idx, per_fetch(table, contig, s, e, run)):
            results[i] = scores
    _write_tracks(output_file, header, contigs, starts, results)
    if verbose:
        stderr.write(f"cleavage profile took {time.time() - start_time} s to complete\n")
    return output_file
