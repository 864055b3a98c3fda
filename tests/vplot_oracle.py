"""Brute-force numpy definition of the site-centred fragment V-plot (``vplot``), for the tests.

Sites: one per BED row (blank lines and lines starting with '#', 'track' or 'browser' skipped), centre
``c = (start + stop) // 2``, mirrored when column 6 is '-'.  A fragment passes when ``mapq >= q`` and
``min_length <= L <= max_length`` with ``L = stop - start``; its midpoint is ``m = (start + stop) // 2`` and its
offset ``d = m - c`` (``c - m`` for a mirrored site).  For every site and every passing fragment with
``|d| <= flank``: ``M[L - min_length, d + flank] += 1`` (int64).

This lives beside the tests rather than in ``oracle/oracle.py``: that module restates functions of the reference,
which has no V-plot.  The definition here is plain numpy, one site at a time, and shares nothing with the kernel.
"""
import numpy as np


def read_sites(lines):
    """[(contig, centre, flipped)] of the BED text lines."""
    out = []
    for line in lines:
        if not line.strip() or line.startswith(("#", "track", "browser")):
            continue
        f = line.split()
        out.append((f[0], (int(f[1]) + int(f[2])) // 2, len(f) >= 6 and f[5] == "-"))
    return out


def vplot(start, stop, mapq, centers, flips, flank, min_length, max_length, q=30) -> np.ndarray:
    st = np.asarray(start, np.int64)
    sp = np.asarray(stop, np.int64)
    L = sp - st
    ok = (np.asarray(mapq).astype(np.int64) >= q) & (L >= min_length) & (L <= max_length)
    m = (st + sp) // 2
    M = np.zeros((max_length - min_length + 1, 2 * flank + 1), np.int64)
    for c, flip in zip(centers, flips):
        d = (c - m) if flip else (m - c)
        sel = ok & (np.abs(d) <= flank)
        np.add.at(M, (L[sel] - min_length, d[sel] + flank), 1)
    return M
