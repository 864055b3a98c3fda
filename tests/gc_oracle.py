"""Plain numpy restatement of the fragment GC-bias definition (``gc_bias``, DESIGN.md 4.10).

A placement [p, p + L) of a contig counts when p >= 0, p + L <= contig_len, its midpoint p + L // 2 lies in a
merged region and no base of it is N; its key is (L - min_length, g), g = C/G bases in it.  Observed: one placement
per fragment with mapq >= q and min_length <= L <= max_length.  Expected: one per (p, L)."""
import warnings

import numpy as np


def prefix(codes, nmask):
    """(G/C prefix, N prefix), int64[n + 1] each: G/C = code C or G and not N."""
    codes = np.asarray(codes); nmask = np.asarray(nmask, bool)
    gc = ((codes == 1) | (codes == 2)) & ~nmask
    z = np.zeros(1, np.int64)
    return np.concatenate([z, np.cumsum(gc, dtype=np.int64)]), np.concatenate([z, np.cumsum(nmask, dtype=np.int64)])


def in_regions(m, reg_start, reg_stop):
    """m lies in one of the sorted, disjoint regions."""
    s = np.asarray(reg_start, np.int64); e = np.asarray(reg_stop, np.int64)
    m = np.asarray(m, np.int64)
    if s.size == 0:
        return np.zeros(m.shape, bool)
    i = np.searchsorted(e, m, side="right")
    ok = i < s.size
    return ok & (s[np.minimum(i, s.size - 1)] <= m)


def observed(st, sp, mq, codes, nmask, clen, reg_start, reg_stop, min_length, max_length, q):
    O = np.zeros((max_length - min_length + 1, max_length + 1), np.int64)
    st = np.asarray(st, np.int64); sp = np.asarray(sp, np.int64); mq = np.asarray(mq, np.int64)
    L = sp - st
    ok = (mq >= q) & (L >= min_length) & (L <= max_length) & (st >= 0) & (sp <= clen)
    ok &= in_regions((st + sp) // 2, reg_start, reg_stop)
    pg, pn = prefix(codes, nmask)
    s, e, L = st[ok], sp[ok], L[ok]
    clean = pn[e] - pn[s] == 0
    np.add.at(O, (L[clean] - min_length, (pg[e] - pg[s])[clean]), 1)
    return O


def expected(codes, nmask, clen, reg_start, reg_stop, min_length, max_length):
    E = np.zeros((max_length - min_length + 1, max_length + 1), np.int64)
    pg, pn = prefix(codes, nmask)
    for L in range(min_length, max_length + 1):
        h = L // 2
        ps = [np.arange(max(a - h, 0), min(b - h, clen - L + 1), dtype=np.int64) for a, b in zip(reg_start, reg_stop)]
        p = np.concatenate(ps) if ps else np.zeros(0, np.int64)
        p = p[pn[p + L] - pn[p] == 0]
        E[L - min_length] = np.bincount(pg[p + L] - pg[p], minlength=max_length + 1)
    return E


def ratio(O, E):
    """(O[i, g] / O[i].sum()) / (E[i, g] / E[i].sum()), NaN where E[i, g] == 0 or O[i].sum() == 0."""
    os_ = O.sum(axis=1, keepdims=True); es = E.sum(axis=1, keepdims=True)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = (O / os_) / (E / es)
    r[(E == 0) | (os_ == 0)] = np.nan
    return r


def merge_regions(rows, chrom_len):
    """{contig: (starts, stops)}: BED rows (contig, start, stop) clipped to [0, chrom_len[contig]], sorted and
    merged where they overlap or touch; rows on contigs outside ``chrom_len`` dropped (one warning)."""
    out, missing = {}, []
    for c, a, b in rows:
        if c not in chrom_len:
            missing.append(c)
            continue
        a, b = max(int(a), 0), min(int(b), chrom_len[c])
        if b > a:
            out.setdefault(c, []).append((a, b))
    if missing:
        warnings.warn(f"regions on contigs missing from the input or the reference skipped: {sorted(set(missing))}")
    merged = {}
    for c, iv in out.items():
        iv.sort()
        m = [list(iv[0])]
        for a, b in iv[1:]:
            if a <= m[-1][1]:
                m[-1][1] = max(m[-1][1], b)
            else:
                m.append([a, b])
        merged[c] = (np.array([x[0] for x in m], np.int64), np.array([x[1] for x in m], np.int64))
    return merged


def text(O, E, R, min_length):
    lines = ["length\tgc\tobserved\texpected\tratio"]
    for i in range(O.shape[0]):
        L = min_length + i
        for g in range(L + 1):
            lines.append(f"{L}\t{g}\t{int(O[i, g])}\t{int(E[i, g])}\t{float(R[i, g])!r}")
    return "\n".join(lines) + "\n"
