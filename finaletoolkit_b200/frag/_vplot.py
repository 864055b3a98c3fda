"""Site-centred fragment V-plots: ``vplot``.

An addition with no reference function of that name.  A V-plot counts fragments by length and by the offset of
their midpoint from a site centre, summed over many sites (TSS, CTCF or TF sites); nucleosome and TF footprints
show as the arms of a "V".  For every site of the BED (centre ``c = (start + stop) // 2``, mirrored for '-'
sites) and every passing fragment (``mapq >= quality_threshold``, ``min_length <= L <= max_length``) whose
midpoint ``m = (start + stop) // 2`` lies within ``flank`` of ``c``, ``M[L - min_length, m - c + flank] += 1``
(``c - m`` for '-' sites).  The counting runs in the CUDA kernel behind ``ftk_vplot_u64``.
"""
from __future__ import annotations

import time
from sys import stderr, stdin

import numpy as np

from ..io.fragments import as_table
from ._common import check_tsv_output, dist_context, group_by_contig, is_writer, per_fetch, write_text

__all__ = ["vplot"]


def _read_sites(site_bed):
    """(contigs, centres, flips) of every BED row: centre (start + stop) // 2, flipped when column 6 is '-'."""
    contigs, centers, flips = [], [], []
    bed = stdin if site_bed == "-" else open(site_bed)
    try:
        for line in bed:
            if not line.strip() or line.startswith(("#", "track", "browser")):
                continue
            contents = line.split()
            if len(contents) < 3:
                raise ValueError(f"{site_bed}: a site needs contig, start and stop columns, got {line.strip()!r}")
            contig, start, stop = contents[0], int(contents[1]), int(contents[2])
            if start > stop:
                raise ValueError(f"[vplot] {contig}:{start}-{stop} is invalid. Please be sure start coordinate "
                                 f"occurs before stop for all sites in {site_bed}.")
            contigs.append(contig)
            centers.append((start + stop) // 2)
            flips.append(len(contents) >= 6 and contents[5] == "-")
    finally:
        if site_bed != "-":
            bed.close()
    return contigs, centers, flips


def vplot_text(matrix: np.ndarray, flank: int, min_length: int) -> str:
    """Header ``length\\t-flank\\t...\\tflank``, then ``L\\tcount\\t...`` for every length."""
    lines = ["\t".join(["length"] + [str(d) for d in range(-flank, flank + 1)])]
    for j, row in enumerate(matrix.tolist()):
        lines.append("\t".join([str(min_length + j)] + [str(v) for v in row]))
    return "\n".join(lines) + "\n"


def vplot(input_file, site_bed, output_file=None, flank=1000, min_length=0, max_length=500, quality_threshold=30,
          workers=1, verbose=0, reference_file=None) -> np.ndarray:
    """Fragment-length x midpoint-offset counts around the sites of ``site_bed``, summed over the sites.

    Returns int64 of shape ``(max_length - min_length + 1, 2 * flank + 1)``: row ``L - min_length``, column
    ``offset + flank``.  A fragment counts once for every site whose window holds its midpoint; sites on contigs
    the input does not hold contribute nothing.  ``output_file``: None (nothing written), ``.tsv``, ``.tsv.gz`` or
    '-' (stdout).  BAM input: each site's fragments are those an indexed fetch of ``[c - flank, c + flank + 1)``
    yields.  ``workers`` is accepted for compatibility (one process per GPU)."""
    from ..device import require_cuda, torch, vplot_check, vplot_sites
    if verbose:
        start_time = time.time()
    if input_file == "-" and site_bed == "-":
        raise ValueError("input_file and site_bed cannot both read from stdin")
    shape = vplot_check(flank, min_length, max_length)
    flank, min_length, max_length = int(flank), int(min_length), int(max_length)
    check_tsv_output(output_file, "the V-plot")
    contigs, centers, flips = _read_sites(site_bed)
    table = as_table(input_file, reference_file)
    ctx = dist_context()   # torch.distributed initialised: contigs sharded over the ranks, one all-reduce
    held = set(table.contigs)
    if ctx is not None:
        from ..distributed import owned_contigs
        held &= set(owned_contigs(table, ctx))
    acc = None   # the one device matrix every launch accumulates into
    for contig, idx in group_by_contig(contigs).items():
        if contig not in held or table.n_fragments(contig) == 0:
            continue
        c = [centers[i] for i in idx]
        f = [flips[i] for i in idx]

        def run(tab, sel, contig=contig, c=c, f=f):
            nonlocal acc
            if tab.n_fragments(contig):
                acc = vplot_sites(tab.device(contig), [c[k] for k in sel], [f[k] for k in sel], flank, min_length,
                                  max_length, quality_threshold, out=acc)
            return [None] * len(sel)

        # the region an indexed fetch is asked for: the site's window, clamped at 0
        per_fetch(table, contig, [max(x - flank, 0) for x in c], [x + flank + 1 for x in c], run)
    if ctx is not None:
        t = torch()
        if acc is None:
            acc = t.zeros(shape, dtype=t.int64, device=require_cuda())
        ctx.all_reduce_sum(acc)
        if not is_writer(ctx):
            output_file = None
    result = np.zeros(shape, np.int64) if acc is None else acc.cpu().numpy().astype(np.int64, copy=False)
    if output_file is not None:
        write_text(output_file, vplot_text(result, flank, min_length))
    if verbose:
        stderr.write(f"vplot took {time.time() - start_time} s to complete\n")
    return result
