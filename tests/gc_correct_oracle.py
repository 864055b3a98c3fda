"""Plain numpy restatement of the GC-corrected counts (``gc_corrected_coverage`` / ``gc_corrected_profile``,
DESIGN.md 4.11) on ``gc_oracle.prefix``.

A fragment [s, e) (L = e - s, m = (s + e) // 2) is selected when mapq >= q and min_length <= L <= max_length and m
passes the position test.  It adds 1 to the count, and W[L - min_length, g] to the corrected sum when s >= 0,
e <= contig_len and none of its bases is N.  Corrected sums are ``math.fsum`` per interval or offset."""
import math

import numpy as np

import gc_oracle as GO


def weights(ratio):
    """1 / ratio where the ratio is finite and > 0, else 0."""
    r = np.asarray(ratio, np.float64)
    w = np.zeros(r.shape, np.float64)
    ok = np.isfinite(r) & (r > 0)
    w[ok] = 1.0 / r[ok]
    return w


def fragment_weights(st, sp, mq, codes, nmask, clen, W, min_length, max_length, q):
    """(selected by mapq and length, midpoint, weight (0 where undefined), weight defined) per fragment."""
    st = np.asarray(st, np.int64); sp = np.asarray(sp, np.int64); mq = np.asarray(mq, np.int64)
    L = sp - st
    sel = (mq >= q) & (L >= min_length) & (L <= max_length)
    placed = sel & (st >= 0) & (sp <= clen)
    pg, pn = GO.prefix(codes, nmask)
    s, e = np.where(placed, st, 0), np.where(placed, sp, 0)
    defined = placed & (pn[e] - pn[s] == 0)
    w = np.zeros(st.size, np.float64)
    w[defined] = np.asarray(W, np.float64)[L[defined] - min_length, (pg[e] - pg[s])[defined]]
    return sel, (st + sp) // 2, w, defined


def intervals(st, sp, mq, codes, nmask, clen, ivl_start, ivl_stop, W, min_length, max_length, q):
    """(count int64[n], corrected float64[n]); None bounds are unbounded."""
    sel, m, w, _ = fragment_weights(st, sp, mq, codes, nmask, clen, W, min_length, max_length, q)
    count = np.zeros(len(ivl_start), np.int64)
    corr = np.zeros(len(ivl_start), np.float64)
    for k, (a, b) in enumerate(zip(ivl_start, ivl_stop)):
        hit = sel.copy()
        if a is not None:
            hit &= m >= a
        if b is not None:
            hit &= m < b
        count[k] = int(hit.sum())
        corr[k] = math.fsum(w[hit].tolist())
    return count, corr


def sites(st, sp, mq, codes, nmask, clen, centers, flips, flank, W, min_length, max_length, q):
    """(count int64[2 flank + 1], corrected float64[2 flank + 1]) summed over the sites."""
    sel, m, w, _ = fragment_weights(st, sp, mq, codes, nmask, clen, W, min_length, max_length, q)
    bins, vals = [], []
    for c, f in zip(centers, flips):
        d = (c - m) if f else (m - c)
        hit = sel & (np.abs(d) <= flank)
        bins.append(d[hit] + flank); vals.append(w[hit])
    bins = np.concatenate(bins) if bins else np.zeros(0, np.int64)
    vals = np.concatenate(vals) if vals else np.zeros(0)
    count = np.bincount(bins, minlength=2 * flank + 1).astype(np.int64)
    corr = np.zeros(2 * flank + 1, np.float64)
    order = np.argsort(bins, kind="stable")
    sb, sv = bins[order], vals[order]
    cuts = np.flatnonzero(np.diff(sb)) + 1
    for b, chunk in zip(np.split(sb, cuts), np.split(sv, cuts)):
        if b.size:
            corr[b[0]] = math.fsum(chunk.tolist())
    return count, corr


def coverage_text(rows):
    """rows: (contig, start, stop, name, count, corrected)."""
    return "contig\tstart\tstop\tname\tcount\tcorrected\n" + "".join(
        f"{c}\t{s}\t{e}\t{n}\t{int(k)}\t{float(w)!r}\n" for c, s, e, n, k, w in rows)


def profile_text(count, corrected, flank):
    return "offset\tcount\tcorrected\n" + "".join(
        f"{d}\t{int(k)}\t{float(w)!r}\n" for d, k, w in zip(range(-flank, flank + 1), count, corrected))
