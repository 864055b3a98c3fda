"""Orientation-aware fragment end profiles at open chromatin: ``ocf``.

An addition with no reference function of that name: the orientation-aware cfDNA fragmentation (OCF) measure of
Sun et al. (Genome Research 2019).  At an open-chromatin region the nucleosome just right of the centre leaves
fragments whose upstream (left) ends sit at about +60 bp, and the nucleosome just left of it leaves downstream
(right) ends at about -60 bp; summed over a tissue's regions, the imbalance measures how much of the sample's
cfDNA comes from that tissue.

Each BED file is one site set (its label is the file's basename without ``.bed``).  For every site (centre
``c = (start + stop) // 2``, mirrored when column 6 is '-') and every passing fragment ``[s, e)`` (``mapq >=
quality_threshold``, ``L = e - s >= 1``, ``min_length <= L <= max_length``), the upstream end offset ``s - c``
and the downstream end offset ``e - 1 - c`` (mirrored: ``c - (e - 1)`` and ``c - s``) each add 1 to their row of
the set when within ``flank``.  The counting runs in the CUDA kernel behind ``ftk_ocf_u64``; the OCF value is
computed on the host from the integer counts.
"""
from __future__ import annotations

import os
import time
from dataclasses import dataclass
from sys import stderr

import numpy as np

from ..io.fragments import as_table
from ._common import check_tsv_output, dist_context, group_by_contig, is_writer, per_fetch, write_text
from ._vplot import _read_sites

__all__ = ["ocf", "OcfResult"]


@dataclass
class OcfResult:
    """End profiles and OCF values of each site set.

    ``labels[k]`` names set k; ``n_sites[k]`` counts its sites on contigs the input holds; ``upstream[k, x + flank]``
    and ``downstream[k, x + flank]`` count the fragment ends at offset x from a site centre (int64); ``ocf[k]`` is
    the set's OCF value (NaN when it has no end in the window)."""
    labels: list
    n_sites: np.ndarray
    upstream: np.ndarray
    downstream: np.ndarray
    ocf: np.ndarray
    flank: int
    peak_offset: int
    peak_width: int


def _set_labels(site_beds):
    """(paths, labels) of the site files: a label is the basename without a trailing ``.bed``."""
    paths = [site_beds] if isinstance(site_beds, (str, os.PathLike)) else list(site_beds)
    if not paths:
        raise ValueError("ocf needs at least one site BED file")
    paths = [os.fspath(p) for p in paths]
    if "-" in paths and len(paths) > 1:
        raise ValueError("'-' (stdin) can only be the single site file")
    labels = []
    for p in paths:
        name = os.path.basename(p)
        labels.append(name[:-4] if name.endswith(".bed") else name)
    if len(set(labels)) != len(labels):
        raise ValueError(f"two site files have the same label: {labels}")
    return paths, labels


def ocf_values(counts: np.ndarray, flank: int, peak_offset: int, peak_width: int) -> np.ndarray:
    """OCF of every set from its end counts ``counts[k] = (U, D)`` (int64 ``[S, 2, 2 flank + 1]``).

    With ``P+ = [o - w // 2, o - w // 2 + w)`` and ``P- = -P+``: ``num = sum_{P+} (U - D) + sum_{P-} (D - U)`` and
    ``T = sum U + sum D`` over the window; ``OCF = num * 2 (2 flank + 1) / T``, one correctly rounded division of
    exact integers (NaN when ``T = 0``)."""
    lo = peak_offset - peak_width // 2
    plus = slice(flank + lo, flank + lo + peak_width)
    minus = slice(flank - lo - peak_width + 1, flank - lo + 1)
    out = np.empty(counts.shape[0], np.float64)
    for k in range(counts.shape[0]):
        u, d = counts[k, 0], counts[k, 1]
        num = int(u[plus].sum()) - int(d[plus].sum()) + int(d[minus].sum()) - int(u[minus].sum())
        total = int(u.sum()) + int(d.sum())
        out[k] = num * 2 * (2 * flank + 1) / total if total else float("nan")
    return out


def ocf_summary_text(res: OcfResult) -> str:
    """Header ``set\\tsites\\tends\\tocf``, then one row per set (``repr`` floats, ``nan`` when undefined)."""
    lines = ["set\tsites\tends\tocf"]
    for k, label in enumerate(res.labels):
        ends = int(res.upstream[k].sum()) + int(res.downstream[k].sum())
        lines.append(f"{label}\t{int(res.n_sites[k])}\t{ends}\t{float(res.ocf[k])!r}")
    return "\n".join(lines) + "\n"


def ocf_profile_text(res: OcfResult) -> str:
    """Header ``set\\tend\\t-flank\\t...\\tflank``, then the rows ``label\\tU\\t...`` and ``label\\tD\\t...`` per set."""
    lines = ["\t".join(["set", "end"] + [str(x) for x in range(-res.flank, res.flank + 1)])]
    for k, label in enumerate(res.labels):
        for end, row in (("U", res.upstream[k]), ("D", res.downstream[k])):
            lines.append("\t".join([label, end] + [str(v) for v in row.tolist()]))
    return "\n".join(lines) + "\n"


def ocf(input_file, site_beds, output_file=None, profile_file=None, flank=1000, peak_offset=60, peak_width=20,
        min_length=None, max_length=None, quality_threshold=30, workers=1, verbose=0,
        reference_file=None) -> OcfResult:
    """Orientation-aware fragment end profiles and OCF values around the sites of each BED file of ``site_beds``.

    ``site_beds`` is one path or a sequence of paths; each file is one site set.  For every site of a set and every
    passing fragment, the upstream end (offset ``s - c``; mirrored sites ``c - (e - 1)``) and the downstream end
    (``e - 1 - c``; mirrored ``c - s``) each add 1 at their offset when it lies within ``flank``.  A fragment passes
    when ``mapq >= quality_threshold`` and ``max(1, min_length) <= L <= max_length`` (None = unbounded).

    OCF: with ``P+ = [peak_offset - peak_width // 2, peak_offset - peak_width // 2 + peak_width)`` (``[50, 69]`` at
    the defaults) and ``P- = -P+``, ``OCF = (sum_{P+} (U - D) + sum_{P-} (D - U)) / mu`` with ``mu = T / (2 (2 flank
    + 1))`` and ``T`` the set's ends over the whole window, i.e. the window sums of the mean-normalised signals
    ``U / mu`` and ``D / mu`` (computed as one division of exact integers; NaN when ``T = 0``).  This normalisation
    is this package's choice: it has not been checked against the exact scaling of Sun et al. (2019), and the raw
    counts are returned so that any other scaling can be applied.  Phased nucleosomes flanking an open site give a positive value.

    Returns an ``OcfResult``.  ``output_file``: None, ``.tsv``, ``.tsv.gz`` or '-' for the per-set table
    (``set sites ends ocf``); ``profile_file`` likewise for the U and D rows of every set.  BAM input: each site's
    fragments are those an indexed fetch of ``[c - flank, c + flank + 1)`` yields.  ``workers`` is accepted for
    compatibility (one process per GPU)."""
    from ..device import ocf_check, ocf_length_check, ocf_sites, require_cuda, torch
    if verbose:
        start_time = time.time()
    paths, labels = _set_labels(site_beds)
    if input_file == "-" and "-" in paths:
        raise ValueError("input_file and the site file cannot both read from stdin")
    shape = ocf_check(flank, peak_offset, peak_width, len(paths))
    flank, peak_offset, peak_width = int(flank), int(peak_offset), int(peak_width)
    ocf_length_check(min_length, max_length)
    check_tsv_output(output_file, "the OCF table")
    check_tsv_output(profile_file, "the OCF end profiles")
    if output_file == "-" and profile_file == "-":
        raise ValueError("output_file and profile_file cannot both write to stdout")
    contigs, centers, flips, sets = [], [], [], []
    for k, path in enumerate(paths):
        cs, xs, fs = _read_sites(path)
        contigs += cs; centers += xs; flips += fs; sets += [k] * len(cs)
    table = as_table(input_file, reference_file)
    ctx = dist_context()   # torch.distributed initialised: contigs sharded over the ranks, one all-reduce
    present = set(table.contigs)
    held = set(present)
    if ctx is not None:
        from ..distributed import owned_contigs
        held &= set(owned_contigs(table, ctx))
    n_sites = np.bincount([s for s, c in zip(sets, contigs) if c in present], minlength=shape[0]).astype(np.int64)
    acc = None   # the one device tensor every launch accumulates into
    for contig, idx in group_by_contig(contigs).items():
        if contig not in held or table.n_fragments(contig) == 0:
            continue
        c = [centers[i] for i in idx]
        f = [flips[i] for i in idx]
        s = [sets[i] for i in idx]

        def run(tab, sel, contig=contig, c=c, f=f, s=s):
            nonlocal acc
            if tab.n_fragments(contig):
                acc = ocf_sites(tab.device(contig), [c[k] for k in sel], [f[k] for k in sel], [s[k] for k in sel],
                                shape[0], flank, min_length, max_length, quality_threshold, out=acc)
            return [None] * len(sel)

        # the region an indexed fetch is asked for: the site's window, clamped at 0
        per_fetch(table, contig, [max(x - flank, 0) for x in c], [x + flank + 1 for x in c], run)
    if ctx is not None:
        t = torch()
        if acc is None:
            acc = t.zeros(shape, dtype=t.int64, device=require_cuda())
        ctx.all_reduce_sum(acc)
        if not is_writer(ctx):
            output_file = profile_file = None
    counts = np.zeros(shape, np.int64) if acc is None else acc.cpu().numpy().astype(np.int64, copy=False)
    res = OcfResult(labels, n_sites, counts[:, 0].copy(), counts[:, 1].copy(),
                    ocf_values(counts, flank, peak_offset, peak_width), flank, peak_offset, peak_width)
    if output_file is not None:
        write_text(output_file, ocf_summary_text(res))
    if profile_file is not None:
        write_text(profile_file, ocf_profile_text(res))
    if verbose:
        stderr.write(f"ocf took {time.time() - start_time} s to complete\n")
    return res
