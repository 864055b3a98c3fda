"""Fragment GC bias: ``gc_bias``.

An addition with no reference function of that name: the fragment-level GC model (Benjamini & Speed 2012; deepTools
``computeGCBias``), all integers and no third-party smoother.  Fragments are counted by (length L, G+C bases g); the
observed counts come from the sample, the expected counts from every place a fragment of length L could sit in the
same regions.  A placement ``[p, p + L)`` counts when ``p >= 0``, ``p + L <= contig length``, its midpoint
``p + L // 2`` lies in a region and none of its bases is N.  Their per-length ratio
``(O[i, g] / O[i].sum()) / (E[i, g] / E[i].sum())`` is the bias (NaN where ``E[i, g] == 0`` or ``O[i].sum() == 0``).
The counting runs in the CUDA kernels behind ``ftk_gc_observed_u64`` and ``ftk_gc_expected_u64``.
"""
from __future__ import annotations

import time
import warnings
from dataclasses import dataclass
from sys import stderr, stdin

import numpy as np

from ..io.fragments import as_table
from ..io.reference import open_reference
from ._common import check_tsv_output, dist_context, is_writer, per_fetch, write_text

__all__ = ["gc_bias", "GCBias", "read_gc_bias"]


@dataclass
class GCBias:
    """Counts by (length, G+C bases): row ``L - min_length``, column ``g`` (``0 <= g <= max_length``)."""
    observed: np.ndarray   # int64, the sample's fragments
    expected: np.ndarray   # int64, every placement of each length in the regions
    ratio: np.ndarray      # float64, (O / O.sum(row)) / (E / E.sum(row)); NaN where undefined
    min_length: int
    max_length: int


def gc_ratio(O: np.ndarray, E: np.ndarray) -> np.ndarray:
    """``(O[i, g] / O[i].sum()) / (E[i, g] / E[i].sum())`` in fp64, NaN where ``E[i, g] == 0`` or ``O[i].sum() == 0``."""
    o_sum = O.sum(axis=1, keepdims=True)
    e_sum = E.sum(axis=1, keepdims=True)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = (O / o_sum) / (E / e_sum)
    r[(E == 0) | (o_sum == 0)] = np.nan
    return r


def gc_text(res: GCBias) -> str:
    """Header ``length\\tgc\\tobserved\\texpected\\tratio``, then one row per ``(L, g)`` with ``g <= L``."""
    lines = [_HEADER]
    O, E, R = res.observed.tolist(), res.expected.tolist(), res.ratio.tolist()
    for i in range(len(O)):
        L = res.min_length + i
        o, e, r = O[i], E[i], R[i]
        lines.extend(f"{L}\t{g}\t{o[g]}\t{e[g]}\t{r[g]!r}" for g in range(L + 1))
    return "\n".join(lines) + "\n"


_HEADER = "length\tgc\tobserved\texpected\tratio"


def read_gc_bias(path) -> GCBias:
    """The ``GCBias`` a ``gc_bias`` / ``gc-bias`` table (``.tsv`` or ``.tsv.gz``) holds; the inverse of ``gc_text``.

    Ratios are read back as written (``repr`` floats and ``nan`` round-trip exactly).  ValueError for a table that
    is not one row per ``(L, g)``, ``0 <= g <= L``, for consecutive lengths within ``[1, 1024]``."""
    import gzip
    import os
    path = os.fspath(path)
    with (gzip.open(path, "rt") if path.endswith(".gz") else open(path)) as fh:
        lines = fh.read().splitlines()
    if not lines or lines[0] != _HEADER:
        raise ValueError(f"{path}: not a GC-bias table (expected the header {_HEADER!r})")
    rows = []
    for k, line in enumerate(lines[1:], 2):
        f = line.split("\t")
        try:
            if len(f) != 5:
                raise ValueError
            rows.append((int(f[0]), int(f[1]), int(f[2]), int(f[3]), float(f[4])))
        except ValueError:
            raise ValueError(f"{path}:{k}: malformed GC-bias row {line!r}") from None
    if not rows:
        raise ValueError(f"{path}: the GC-bias table has no rows")
    lo, hi = rows[0][0], rows[-1][0]
    if not 1 <= lo <= hi <= 1024 or len(rows) != sum(L + 1 for L in range(lo, hi + 1)):
        raise ValueError(f"{path}: the GC-bias table does not hold every (length, gc) of lengths {lo}..{hi}")
    keys = np.array([(r[0], r[1]) for r in rows], np.int64)
    want = np.array([(L, g) for L in range(lo, hi + 1) for g in range(L + 1)], np.int64)
    if not np.array_equal(keys, want):
        raise ValueError(f"{path}: the GC-bias rows are not one per (length, gc) in order")
    shape = (hi - lo + 1, hi + 1)
    O, E = np.zeros(shape, np.int64), np.zeros(shape, np.int64)
    R = np.full(shape, np.nan)
    i, g = keys[:, 0] - lo, keys[:, 1]
    O[i, g] = [r[2] for r in rows]
    E[i, g] = [r[3] for r in rows]
    R[i, g] = [r[4] for r in rows]
    return GCBias(O, E, R, lo, hi)


def read_regions(interval_file, chrom_len: dict) -> dict:
    """{contig: (starts, stops) int64} of a BED: rows clipped to ``[0, chrom_len[contig]]``, sorted and merged where
    they overlap or touch.  Rows on contigs outside ``chrom_len`` are skipped with one ``UserWarning``."""
    rows: dict = {}
    missing = []
    bed = stdin if interval_file == "-" else open(interval_file)
    try:
        for line in bed:
            if not line.strip() or line.startswith(("#", "track", "browser")):
                continue
            contents = line.split()
            if len(contents) < 3:
                raise ValueError(f"{interval_file}: a region needs contig, start and stop columns, got {line.strip()!r}")
            contig, start, stop = contents[0], int(contents[1]), int(contents[2])
            if start > stop:
                raise ValueError(f"[gc_bias] {contig}:{start}-{stop} is invalid. Please be sure start coordinate "
                                 f"occurs before stop for all regions in {interval_file}.")
            if contig not in chrom_len:
                if contig not in missing:
                    missing.append(contig)
                continue
            start, stop = max(start, 0), min(stop, chrom_len[contig])
            if stop > start:
                rows.setdefault(contig, []).append((start, stop))
    finally:
        if interval_file != "-":
            bed.close()
    if missing:
        warnings.warn(f"gc_bias: regions on contigs that the input or the reference lacks were skipped: "
                      f"{', '.join(missing)}", UserWarning, stacklevel=3)
    merged = {}
    for contig, iv in rows.items():
        iv.sort()
        s, e = [iv[0][0]], [iv[0][1]]
        for a, b in iv[1:]:
            if a <= e[-1]:
                e[-1] = max(e[-1], b)
            else:
                s.append(a); e.append(b)
        merged[contig] = (np.array(s, np.int64), np.array(e, np.int64))
    return merged


def gc_bias(input_file, refseq_file, interval_file=None, output_file=None, min_length=50, max_length=500,
            quality_threshold=30, workers=1, verbose=0, reference_file=None) -> GCBias:
    """Observed and expected fragment counts by (length, G+C bases) and their ratio.

    Regions: the whole of every contig both ``refseq_file`` and the input hold, or the rows of ``interval_file``
    (BED, clipped to the contig and merged, so each position counts at most once).  A fragment counts when
    ``mapq >= quality_threshold``, ``min_length <= L <= max_length``, its midpoint ``(start + stop) // 2`` lies in a
    region, it lies within the contig and touches no N.  ``1 <= min_length <= max_length <= 1024``.
    ``output_file``: None (nothing written), ``.tsv``, ``.tsv.gz`` or '-' (stdout).  BAM input: each region's
    fragments are those an indexed fetch of the region yields.  ``workers`` is accepted for compatibility (one
    process per GPU)."""
    from ..device import gc_check, gc_expected, gc_observed, require_cuda, torch
    if verbose:
        start_time = time.time()
    shape = gc_check(min_length, max_length)
    min_length, max_length = int(min_length), int(max_length)
    check_tsv_output(output_file, "the GC-bias table")
    ref = open_reference(refseq_file)
    table = as_table(input_file, reference_file)
    common = [c for c in table.contigs if c in ref.chroms]
    chrom_len = {c: int(ref.chroms[c]) for c in common}
    if interval_file is None:
        regions = {c: (np.zeros(1, np.int64), np.array([n], np.int64)) for c, n in chrom_len.items() if n > 0}
    else:
        regions = read_regions(interval_file, chrom_len)
    ctx = dist_context()   # torch.distributed initialised: contigs sharded over the ranks, one all-reduce
    if ctx is not None:
        from ..distributed import owned_contigs
        mine = set(owned_contigs(table, ctx))
        regions = {c: r for c, r in regions.items() if c in mine}
    t = torch()
    acc = None   # [observed, expected]: one buffer every launch accumulates into, all-reduced at once
    for contig, (rs, re) in regions.items():
        if acc is None:
            acc = t.zeros((2,) + shape, dtype=t.int64, device=require_cuda())
        dev_ref = ref.device_contig(contig, acc.device)
        gc_expected(dev_ref, rs, re, min_length, max_length, out=acc[0])
        if table.n_fragments(contig) == 0:
            continue

        def run(tab, sel, contig=contig, rs=rs, re=re, dev_ref=dev_ref):
            if tab.n_fragments(contig):
                gc_observed(tab.device(contig, acc.device), dev_ref, rs[sel], re[sel], min_length, max_length,
                            quality_threshold, out=acc[1])
            return [None] * len(sel)

        per_fetch(table, contig, rs.tolist(), re.tolist(), run)
    if ctx is not None:
        if acc is None:
            acc = t.zeros((2,) + shape, dtype=t.int64, device=require_cuda())
        ctx.all_reduce_sum(acc)
        if not is_writer(ctx):
            output_file = None
    host = np.zeros((2,) + shape, np.int64) if acc is None else acc.cpu().numpy().astype(np.int64, copy=False)
    O, E = host[1].copy(), host[0].copy()
    res = GCBias(O, E, gc_ratio(O, E), min_length, max_length)
    if output_file is not None:
        write_text(output_file, gc_text(res))
    if verbose:
        stderr.write(f"gc_bias took {time.time() - start_time} s to complete\n")
    return res
