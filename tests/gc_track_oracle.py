"""Plain numpy restatement of the GC-corrected depth tracks (``gc_corrected_coverage_profile``, DESIGN.md 4.14) on
``gc_correct_oracle.fragment_weights`` and ``gc_oracle.prefix``.

Q = rint(W * 2^32) (int64).  A fragment [s, e) selected by mapq and length weighs Q[L - min_length, g] where its
placement is defined, 0 elsewhere.  S(p) = the int64 sum of the weights of the selected fragments with s <= p < e
(span: np.add.at difference + cumsum) or (s + e) // 2 == p (midpoint: np.add.at, as np.bincount would sum the
weights in fp64); the track is fp64(S(p)) * 2^-32."""
import numpy as np

import gc_correct_oracle as CO
import gc_oracle as GO


def quantise(W):
    q = np.rint(np.asarray(W, np.float64) * 2.0 ** 32)
    assert q.size == 0 or q.max() < 2.0 ** 62
    return q.astype(np.int64)


def fragment_q(st, sp, mq, codes, nmask, clen, W, min_length, max_length, q):
    """(selected, int64 quantised weight, 0 where the placement is undefined) per fragment."""
    st = np.asarray(st, np.int64); sp = np.asarray(sp, np.int64)
    sel, _, _, defined = CO.fragment_weights(st, sp, mq, codes, nmask, clen, np.zeros_like(W), min_length, max_length, q)
    pg, _ = GO.prefix(codes, nmask)
    s, e = st[defined], sp[defined]
    wq = np.zeros(st.size, np.int64)
    wq[defined] = quantise(W)[e - s - min_length, pg[e] - pg[s]]
    return sel, wq


def sums(st, sp, mq, codes, nmask, clen, a, b, W, min_length, max_length, q, midpoint=False):
    """int64[max(b - a, 0)]: S(p) for every p of [a, b)."""
    n = max(int(b) - int(a), 0)
    sel, wq = fragment_q(st, sp, mq, codes, nmask, clen, W, min_length, max_length, q)
    keep = sel & (wq != 0)
    s = np.asarray(st, np.int64)[keep]; e = np.asarray(sp, np.int64)[keep]; w = wq[keep]
    if midpoint:
        m = (s + e) // 2 - a
        ok = (m >= 0) & (m < n)
        out = np.zeros(n, np.int64)
        np.add.at(out, m[ok], w[ok])
        return out
    lo = np.clip(s - a, 0, n); hi = np.clip(e - a, 0, n)
    ok = hi > lo
    d = np.zeros(n + 1, np.int64)
    np.add.at(d, lo[ok], w[ok])
    np.add.at(d, hi[ok], -w[ok])
    return np.cumsum(d[:n])


def to_track(S):
    return np.asarray(S, np.int64).astype(np.float64) * 2.0 ** -32


def track(st, sp, mq, codes, nmask, clen, a, b, W, min_length, max_length, q, midpoint=False):
    return to_track(sums(st, sp, mq, codes, nmask, clen, a, b, W, min_length, max_length, q, midpoint))


def track_intervals(st, sp, mq, codes, nmask, clen, ivl_start, ivl_stop, W, min_length, max_length, q,
                    midpoint=False):
    """Every interval back to back + offsets (the return shape of ``device.gc_depth_intervals``)."""
    parts = [track(st, sp, mq, codes, nmask, clen, a, b, W, min_length, max_length, q, midpoint)
             for a, b in zip(ivl_start, ivl_stop)]
    off = np.zeros(len(parts) + 1, np.int64)
    np.cumsum([len(p) for p in parts], out=off[1:])
    return (np.concatenate(parts) if parts else np.zeros(0)), off
