"""TEST SHIM: the device layer replaced by the oracle, so that the host-side orchestration of the public API
(interval grouping, index bookkeeping, writers) can be replayed on a machine without a GPU.

``install(monkeypatch, seqs)`` swaps ``FragmentTable.device`` / ``ReferenceWrapper.device_contig`` and the
kernel wrappers of ``finaletoolkit_b200.device`` for functions with the same signatures and return shapes that
compute with ``oracle/`` on host columns (torch CPU tensors stand in for device tensors).  Nothing in the
package imports this; it exists only for ``-m "not gpu"`` tests of host logic whose numeric core is covered
against the same oracle by the ``-m gpu`` tests.
"""
import numpy as np
import torch

from oracle import oracle as O


class HostFrags:
    """Stand-in for ``device.ContigFragments``."""

    def __init__(self, st, sp, mq, sd):
        self.fr = O.Frags(st, sp, mq, sd)
        self.n, self.max_len = self.fr.n, self.fr.max_len
        self.device = torch.device("cpu")


class HostWpsPlan:
    """Stand-in for ``device.WpsPlan`` (``run`` + ``offsets``)."""

    def __init__(self, ivl_start, ivl_stop, chrom_size, max_length, device=None):
        self.s = np.asarray(ivl_start, np.int64); self.e = np.asarray(ivl_stop, np.int64)
        self.chrom_size = int(chrom_size)
        self.offsets = np.zeros(len(self.s) + 1, np.int64)
        np.cumsum(np.maximum(self.e - self.s, 0), out=self.offsets[1:])

    def run(self, frags, window_size=120, min_length=120, max_length=180, quality_threshold=30, out=None):
        got, _ = O.wps_intervals(frags.fr, self.s, self.e, self.chrom_size, window_size, min_length, max_length,
                                 quality_threshold)
        return torch.from_numpy(got)


def interval_hist(frags, ivl_start=None, ivl_stop=None, intersect_policy="midpoint", min_length=None, max_length=None,
                  quality_threshold=30, n_bins=0, pooled=False, first_seen=False, ivl_set=None, out=None):
    n = len(ivl_start)
    assert not pooled or n == 1
    counts = np.zeros(max(n, 1), np.int64)
    hist = np.zeros((max(n, 1), n_bins), np.int64) if n_bins else None
    first = np.full((max(n, 1), n_bins), 2 ** 31 - 1, np.int32) if (n_bins and first_seen) else None
    for i, (s, e) in enumerate(zip(ivl_start, ivl_stop)):
        d = O.length_dist(frags.fr, s, e, min_length, max_length, intersect_policy, quality_threshold)
        counts[i] = sum(d.values())
        if hist is not None:
            for rank, (ln, c) in enumerate(d.items()):
                hist[i, ln] = c
                if first is not None:
                    first[i, ln] = rank
    t = torch.from_numpy
    return t(counts[:n]), None if hist is None else t(hist), None if first is None else t(first)


def frag_lengths(frags, start=None, stop=None, intersect_policy="midpoint", min_length=0, max_length=1000000000,
                 quality_threshold=30):
    return torch.from_numpy(O.frag_lengths(frags.fr, start, stop, intersect_policy, quality_threshold))


def end_motif_hist(frags, ref, ivl_start, ivl_stop, k=4, strand_mode=0, quality_threshold=20, pooled=False,
                   counts=None, breakpoint=False):
    fn = O.region_breakpoint_motifs if breakpoint else O.region_end_motifs
    rows = np.array([fn(frags.fr, ref, s, e, k, strand_mode == 0, strand_mode == 2, quality_threshold)
                     for s, e in zip(ivl_start, ivl_stop)], np.int64).reshape(-1, 4 ** k)
    if pooled:
        add = torch.from_numpy(rows.sum(axis=0, keepdims=True))
        return add if counts is None else counts.add_(add)
    return torch.from_numpy(rows)


def cleavage_intervals(frags, ivl_start, ivl_stop, chrom_size, min_length=None, max_length=None, quality_threshold=30):
    parts = [O.cleavage_profile(frags.fr, chrom_size, s, e, 0, 0, min_length, max_length, quality_threshold)[1]
             for s, e in zip(ivl_start, ivl_stop)]
    off = np.zeros(len(parts) + 1, np.int64)
    np.cumsum([len(p) for p in parts], out=off[1:])
    return torch.from_numpy(np.concatenate(parts) if parts else np.zeros(0)), off


def delfi_windows(frags, ref, win_start, win_stop, blacklist=None, gaps=None, quality_threshold=30):
    rows = [O.delfi_counts(frags.fr, ref, int(s), int(e), blacklist, gaps, quality_threshold)
            for s, e in zip(win_start, win_stop)]
    return torch.from_numpy(np.array(rows, np.int64).reshape(-1, 4))


def adjust_segments(x, seg_lengths, median_window_size=1000, use_mean=False, savgol=True, savgol_window_size=21,
                    savgol_poly_deg=2, subtract_edges=False, edge_size=500, **_):
    """frag/_adjust_wps.py:119-140 per segment with the reference's own numpy / scipy calls (oracle.adjust_core)."""
    x = np.asarray(x.cpu() if torch.is_tensor(x) else x, dtype=np.float64)
    seg = np.asarray(seg_lengths, np.int64)
    off = np.zeros(len(seg) + 1, np.int64); np.cumsum(seg, out=off[1:])
    if median_window_size > 0 and np.any(seg < median_window_size):
        raise ValueError("median_window_size cannot be greater than the length of interval")
    parts = []
    for a, b in zip(off[:-1], off[1:]):
        v = x[a:b].copy()
        if subtract_edges:
            v -= np.mean([np.mean(v[:edge_size]), np.mean(v[-edge_size:])])
        parts.append(O.adjust_core(v, median_window_size, use_mean, savgol, savgol_window_size, savgol_poly_deg))
    out_off = np.zeros(len(seg) + 1, np.int64); np.cumsum([len(p) for p in parts], out=out_off[1:])
    return torch.from_numpy(np.concatenate(parts) if parts else np.zeros(0)), out_off


def agg_signal(rows, strand, trim_lo, out_len, device=None):
    """utils/_agg_bw.py:84-123: the accepted rows added in file order, '-' rows flipped, NaN -> 0, fp64."""
    out = np.zeros(int(out_len), np.float64)
    for row, sd in zip(np.asarray(rows, np.float32), strand):
        if sd == 0:
            continue
        v = np.nan_to_num(np.asarray(row, np.float64)[trim_lo: trim_lo + out_len])
        out = out + (v if sd > 0 else v[::-1])
    return torch.from_numpy(out)


def _import_whole_package():
    """Import every module of the package now, while ``device`` still holds the real classes: a module first
    imported under the patch (``pipeline`` is imported lazily) would keep a stand-in from its
    ``from .device import ...`` after the monkeypatch is undone, and hand it to later tests."""
    import importlib
    import importlib.util
    import pkgutil
    import finaletoolkit_b200 as F
    for m in pkgutil.walk_packages(F.__path__, F.__name__ + "."):
        if not m.name.endswith(".__main__") and importlib.util.find_spec(m.name).origin.endswith(".py"):
            importlib.import_module(m.name)     # (the walk also lists libftk_b200.so, a ctypes library)


def install(monkeypatch, seqs: dict):
    """``seqs``: {contig: ASCII reference sequence (bytes)} for the motif / DELFI wrappers."""
    _import_whole_package()
    import finaletoolkit_b200.device as D
    from finaletoolkit_b200.io.fragments import FragmentTable
    from finaletoolkit_b200.io.reference import ReferenceWrapper
    monkeypatch.setattr(FragmentTable, "device", lambda self, contig, device=None: HostFrags(*self.host(contig)))
    monkeypatch.setattr(ReferenceWrapper, "device_contig", lambda self, contig, device=None: seqs[contig])
    for name, fn in (("interval_hist", interval_hist), ("frag_lengths", frag_lengths), ("end_motif_hist", end_motif_hist),
                     ("cleavage_intervals", cleavage_intervals), ("delfi_windows", delfi_windows), ("WpsPlan", HostWpsPlan),
                     ("adjust_segments", adjust_segments), ("agg_signal", agg_signal)):
        monkeypatch.setattr(D, name, fn)
