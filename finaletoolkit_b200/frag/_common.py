"""Shared helpers of the feature modules: alias resolution, device access, text writers."""
from __future__ import annotations

import warnings

import numpy as np


def resolve_length_aliases(min_length, max_length, fraction_low, fraction_high, stacklevel=3):
    """Deprecated ``fraction_low/high`` aliases (frag/_wps.py:110-140, frag/_motif_common.py:97-138):
    an alias alone warns; alias + modern spelling raises ValueError."""
    if fraction_low is not None and min_length is None:
        min_length = fraction_low
        warnings.warn("fraction_low is deprecated. Use min_length instead.", category=DeprecationWarning,
                      stacklevel=stacklevel)
    elif fraction_low is not None and min_length is not None:
        warnings.warn("fraction_low is deprecated. Use min_length instead.", category=DeprecationWarning,
                      stacklevel=stacklevel)
        raise ValueError("fraction_low and min_length cannot both be specified")
    if fraction_high is not None and max_length is None:
        max_length = fraction_high
        warnings.warn("fraction_high is deprecated. Use max_length instead.", category=DeprecationWarning,
                      stacklevel=stacklevel)
    elif fraction_high is not None and max_length is not None:
        warnings.warn("fraction_high is deprecated. Use max_length instead.", category=DeprecationWarning,
                      stacklevel=stacklevel)
        raise ValueError("fraction_high and max_length cannot both be specified")
    return min_length, max_length


def dist_context():
    """``DistContext`` when ``torch.distributed`` is initialised with more than one rank (one process
    per GPU; contigs are then LPT-sharded over the ranks and genome-wide totals all-reduced), else None."""
    import sys
    if "torch.distributed" not in sys.modules and "torch" not in sys.modules:
        return None
    from ..sharding import DistContext
    ctx = DistContext()
    return ctx if ctx.on and ctx.world > 1 else None


def is_writer(ctx) -> bool:
    """Under a multi-rank launch only rank 0 writes output files / stdout."""
    return ctx is None or ctx.rank == 0


def group_by_contig(contigs):
    """{contig: [indices]} preserving first-appearance order."""
    groups: dict = {}
    for i, c in enumerate(contigs):
        groups.setdefault(c, []).append(i)
    return groups


def per_fetch(table, contig, fetch_starts, fetch_stops, run, fetch_only: bool = False):
    """The per-interval results ``run`` produces, with the READ-level region selection a BAM query makes.

    ``run(tab, sel) -> list`` computes the intervals at positions ``sel`` of the caller's list from the
    fragment table ``tab`` (one entry per position, in order); ``fetch_starts[k], fetch_stops[k]`` is the
    region the reference hands to ``AlignmentWrapper.fetch`` for interval k (None = unbounded).  For a
    fragment file that region test is the kernels' own fragment predicate and everything is ONE call on the
    whole table.  For BAM input the fetch returns the fragments whose READ 1 overlaps the region
    (io/alignment.py:245) - a per-(fragment, interval) condition - so the intervals that hold a fragment
    the two rules treat differently (``FragmentTable.read1_affected``: those whose edge cuts a fragment
    between its read 1 and its mate) are computed from the rows the fetch would have yielded
    (``FragmentTable.fetched_union``).  Such intervals share a launch whenever no fragment can reach two of
    them (``FragmentTable.fetch_groups``: a tiling of 5-kb windows is two groups, even and odd), so a BAM
    costs a few batched calls per contig, not one per interval; all unaffected intervals go through one
    call on the whole table.

    ``fetch_only``: the caller applies NO fragment-level test after the fetch (the motif counters,
    frag/_end_motifs.py:115-120), so a dovetailed pair whose read 1 runs past its own template counts wherever
    the read reaches.  The fetched tables are then selected by the whole read and ``run(tab, sel, widen)`` is
    asked to query them with bounds widened by ``widen`` = ``FragmentTable.fetch_reach`` - every row of the
    sub-table passes the kernel's overlap test for its own region, and the groups are spaced so that it
    passes for no other."""
    n = len(fetch_starts)
    if n == 0 or not table.has_read1(contig):
        return run(table, list(range(n)))
    affected = table.read1_affected(contig, fetch_starts, fetch_stops, fetch_only)
    out: list = [None] * n
    clean = np.flatnonzero(~affected).tolist()
    if clean:
        for k, r in zip(clean, run(table, clean)):
            out[k] = r
    todo = np.flatnonzero(affected)
    if todo.size:
        lo = [fetch_starts[k] for k in todo.tolist()]
        hi = [fetch_stops[k] for k in todo.tolist()]
        extra = (table.fetch_reach(contig),) if fetch_only else ()
        for members in table.fetch_groups(contig, lo, hi, fetch_only):
            sel = todo[members].tolist()
            rows = table.fetched_union(contig, [lo[m] for m in members.tolist()], [hi[m] for m in members.tolist()],
                                       fetch_only)
            for k, r in zip(sel, run(rows, sel, *extra)):
                out[k] = r
    return out


def bedgraph_lines(contig: str, start: int, scores: np.ndarray) -> str:
    """``contig\\tpos\\tpos+1\\tscore\\n`` per position (frag/_multi_wps.py:328-341), vectorised."""
    n = scores.shape[0]
    if n == 0:
        return ""
    pos = np.arange(start, start + n, dtype=np.int64)
    a = np.char.add(contig + "\t", pos.astype(str))
    a = np.char.add(np.char.add(a, "\t"), (pos + 1).astype(str))
    a = np.char.add(np.char.add(a, "\t"), scores.astype(np.int64).astype(str))
    return "\n".join(a.tolist()) + "\n"


def check_tsv_output(output_file, what: str) -> None:
    """``output_file`` must be None, a ``.tsv`` / ``.tsv.gz`` path or '-'; ``what`` names the table in the error."""
    if isinstance(output_file, str):
        if not (output_file.endswith(".tsv") or output_file.endswith(".tsv.gz") or output_file == "-"):
            raise ValueError("output_file can only have suffix .tsv or .tsv.gz, or be '-'.")
    elif output_file is not None:
        raise TypeError(f'output_file is unsupported type "{type(output_file)}". output_file should be a string '
                        f"specifying the path of the file to output {what} to.")


def write_text(output_file: str, text: str) -> None:
    """``text`` to stdout ('-'), a gzip file (``.gz``) or a plain file."""
    import sys
    if output_file == "-":
        sys.stdout.write(text)
    elif output_file.endswith(".gz"):
        from ..io.textout import GzipTextWriter
        with GzipTextWriter(output_file) as out:
            out.write(text)
    else:
        with open(output_file, "w") as out:
            out.write(text)
