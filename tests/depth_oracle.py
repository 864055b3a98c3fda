"""Brute-force numpy definition of the per-base fragment depth tracks (``coverage_profile``), for the tests.

A fragment passes when ``mapq >= q`` and ``min_length <= stop - start <= max_length`` (None = unbounded);
``stop < start`` never passes (the loaders never produce it and the kernels skip it).
  span:     depth[p] = #{passing fragments with start <= p < stop}          (np.add.at + cumsum)
  midpoint: depth[p] = #{passing fragments with (start + stop) // 2 == p}   (np.bincount)
A zero-length fragment (start == stop) that passes counts at its start in midpoint mode.

This lives beside the tests rather than in ``oracle/oracle.py``: that module restates functions of the reference and
is pinned to the reference's outputs, and the reference has no per-base depth function to restate.  The definition
here is plain numpy and shares nothing with the kernel.
"""
import numpy as np


def passing(start, stop, mapq, min_length=None, max_length=None, q=30):
    L = np.asarray(stop, np.int64) - np.asarray(start, np.int64)
    ok = (np.asarray(mapq).astype(np.int64) >= q) & (L >= 0)
    if min_length is not None:
        ok &= L >= min_length
    if max_length is not None:
        ok &= L <= max_length
    return ok


def depth(start, stop, mapq, a, b, min_length=None, max_length=None, q=30, midpoint=False) -> np.ndarray:
    """int64[max(b - a, 0)]: the depth of every position of [a, b)."""
    n = max(int(b) - int(a), 0)
    ok = passing(start, stop, mapq, min_length, max_length, q)
    st = np.asarray(start, np.int64)[ok]
    sp = np.asarray(stop, np.int64)[ok]
    if midpoint:
        m = (st + sp) // 2 - a
        return np.bincount(m[(m >= 0) & (m < n)], minlength=n)[:n].astype(np.int64)
    s = np.clip(st - a, 0, n)
    e = np.clip(sp - a, 0, n)
    keep = e > s
    d = np.zeros(n + 1, np.int64)
    np.add.at(d, s[keep], 1)
    np.add.at(d, e[keep], -1)
    return np.cumsum(d[:n])


def depth_intervals(start, stop, mapq, ivl_start, ivl_stop, min_length=None, max_length=None, q=30, midpoint=False):
    """Every interval back to back + offsets (the return shape of ``device.depth_intervals``)."""
    parts = [depth(start, stop, mapq, a, b, min_length, max_length, q, midpoint) for a, b in zip(ivl_start, ivl_stop)]
    off = np.zeros(len(parts) + 1, np.int64)
    np.cumsum([len(p) for p in parts], out=off[1:])
    return (np.concatenate(parts) if parts else np.zeros(0, np.int64)), off
