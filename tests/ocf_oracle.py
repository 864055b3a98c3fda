"""Brute-force numpy definition of the orientation-aware fragment end profiles (``ocf``), for the tests.

A fragment ``[s, e)`` passes when ``mapq >= q``, ``L = e - s >= 1`` and ``min_length <= L <= max_length`` (None =
unbounded).  For a site of centre ``c`` the upstream end offset is ``x_U = s - c`` and the downstream one
``x_D = (e - 1) - c``; for a mirrored site ``x_U = c - (e - 1)`` and ``x_D = c - s``.  For every site of set k and
every passing fragment, ``U[k, x_U + F] += 1`` when ``|x_U| <= F`` and ``D[k, x_D + F] += 1`` when ``|x_D| <= F``.

The OCF value is written independently of the package: explicit loops over the peak windows and an exact
``fractions.Fraction``, rounded once to float.  Plain numpy, one site at a time; shares nothing with the kernel.
"""
from fractions import Fraction

import numpy as np


def ends(start, stop, mapq, centers, flips, sets, n_sets, flank, min_length=None, max_length=None, q=30):
    """int64 ``[n_sets, 2, 2 flank + 1]``: the U row, then the D row, of every set."""
    st = np.asarray(start, np.int64)
    sp = np.asarray(stop, np.int64)
    L = sp - st
    ok = (np.asarray(mapq).astype(np.int64) >= q) & (L >= 1)
    if min_length is not None:
        ok &= L >= min_length
    if max_length is not None:
        ok &= L <= max_length
    out = np.zeros((n_sets, 2, 2 * flank + 1), np.int64)
    for c, flip, k in zip(centers, flips, sets):
        xu = (c - (sp - 1)) if flip else (st - c)
        xd = (c - st) if flip else (sp - 1 - c)
        for row, x in ((0, xu), (1, xd)):
            sel = ok & (np.abs(x) <= flank)
            np.add.at(out[k, row], x[sel] + flank, 1)
    return out


def ocf_value(u, d, flank, peak_offset=60, peak_width=20):
    """OCF of one set: (sum over P+ of U - D plus sum over P- of D - U) / (T / (2 (2 flank + 1)))."""
    first = peak_offset - peak_width // 2
    num = 0
    for x in range(first, first + peak_width):
        num += int(u[x + flank]) - int(d[x + flank])
        num += int(d[-x + flank]) - int(u[-x + flank])
    total = sum(int(v) for v in u) + sum(int(v) for v in d)
    if total == 0:
        return float("nan")
    return float(Fraction(num) / Fraction(total, 2 * (2 * flank + 1)))
