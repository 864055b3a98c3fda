"""Device-resident fragment columns and the CUDA op wrappers.

PyTorch is plumbing here (HBM allocations, streams); every computation is a
call into ``libftk_b200.so`` through the C ABI of ``include/ftk_b200.h``.
"""
from __future__ import annotations

import functools
from ctypes import POINTER, c_int32, c_int64

import numpy as np

from ._lib import FTK_NONE, FtkLibraryError, check, lib

__all__ = ["ContigFragments", "WpsPlan", "AdjustPlan", "IntervalSet", "PackedContig", "interval_hist", "frag_lengths",
           "end_motif_hist", "delfi_windows", "blacklist_in_windows", "agg_signal", "require_cuda", "none_to_ftk", "policy_code",
           "vplot_sites", "ocf_sites", "gc_observed", "gc_expected", "gc_weighted_intervals", "gc_weighted_sites",
           "gc_depth_intervals", "spectrum_segments"]

_torch = None


def torch():
    global _torch
    if _torch is None:
        import torch as t
        _torch = t
    return _torch


def require_cuda(device=None):
    """Return a CUDA ``torch.device`` with its index (the current device when ``device`` names none) or raise:
    there is no CPU compute path."""
    t = torch()
    if not t.cuda.is_available():
        raise FtkLibraryError(
            "finaletoolkit_b200 needs a CUDA device (sm_100a); no CPU fallback exists")
    lib()  # fail loudly if the extension is missing
    dev = t.device("cuda") if device is None else t.device(device)
    if dev.type == "cuda" and dev.index is None:
        return t.device("cuda", t.cuda.current_device())
    return dev


def none_to_ftk(v) -> int:
    return FTK_NONE if v is None else int(v)


def _stream_ptr(device) -> int:
    return int(torch().cuda.current_stream(device).cuda_stream)


def _launch(dev, name: str, *args) -> None:
    """``libftk_b200.<name>(*args, stream)`` on device ``dev`` and its current stream, result checked.

    The library launches on the calling thread's current CUDA device, so the call runs with ``dev`` made current:
    tensors on a device other than the current one are worked on where they live.  Nothing changes when ``dev`` is
    already current (e.g. inside a CUDA graph capture)."""
    with torch().cuda.device(dev):
        check(getattr(lib(), name)(*args, _stream_ptr(dev)), name)


def _same_device(dev, *objs) -> None:
    """ValueError unless every object (tensor, ``ContigFragments``, ``PackedContig``, plan) lives on ``dev``."""
    for o in objs:
        if o.device != dev:
            raise ValueError(f"inputs on {o.device} and {dev}: every input of a call must be on one device")


def _np_ptr(a, ctype):
    return a.ctypes.data_as(POINTER(ctype))


class _PinnedStaging:
    """Two reusable pinned host buffers for the big host -> device uploads.

    ``cudaHostAlloc`` of a fresh buffer per column costs ~0.3 s per GB - more than the copy itself.  The
    staging buffers are allocated once (grown on demand), a column is memcpy'd into the free one and
    sent with an asynchronous copy; the buffer is reused only after the event recorded behind that copy
    has completed, so back-to-back uploads overlap the next memcpy with the previous DMA."""

    def __init__(self):
        self.bufs = [None, None]
        self.events = [None, None]
        self.turn = 0

    def upload(self, a: np.ndarray, device):
        t = torch()
        i = self.turn
        self.turn ^= 1
        nbytes = a.nbytes
        if self.events[i] is not None:
            self.events[i].synchronize()
        if self.bufs[i] is None or self.bufs[i].numel() < nbytes:
            self.bufs[i] = None
            self.bufs[i] = t.empty(max(nbytes, 1 << 26), dtype=t.uint8).pin_memory()
        stage = self.bufs[i][:nbytes]
        stage.numpy()[:] = a.reshape(-1).view(np.uint8)
        out = t.empty(a.shape, dtype=t.from_numpy(a[:0]).dtype, device=device)
        out.view(t.uint8).reshape(-1).copy_(stage, non_blocking=True)
        ev = t.cuda.Event()
        ev.record(t.cuda.current_stream(device))
        self.events[i] = ev
        return out


_STAGING: dict = {}


def _to_device(a: np.ndarray, device, dtype):
    """H2D through pinned staging (async on the current stream)."""
    t = torch()
    a = np.ascontiguousarray(a, dtype=dtype)
    if a.nbytes >= (1 << 23):   # big columns go through the reusable pinned staging buffers
        key = str(device)
        if key not in _STAGING:
            _STAGING[key] = _PinnedStaging()
        return _STAGING[key].upload(a, device)
    return t.from_numpy(a).to(device, non_blocking=True)


class ContigFragments:
    """Start-sorted fragments of one contig as columns in HBM.

    ``start``/``stop`` int32, ``mapq``/``strand`` uint8 (strand 1 = '+'), the
    columnar form of the reference's fragment stream
    (utils/_frag_generator.py:124-130 yields contig,start,stop,mapq,is_forward).
    """

    def __init__(self, start, stop, mapq=None, strand=None, device=None, contig=None,
                 max_len=None):
        t = torch()
        self.device = require_cuda(device)
        self.contig = contig
        if isinstance(start, np.ndarray) or not t.is_tensor(start):
            start = np.asarray(start)
            stop = np.asarray(stop)
            if start.size and not np.all(start[1:] >= start[:-1]):
                order = np.argsort(start, kind="stable")
                start, stop = start[order], stop[order]
                mapq = None if mapq is None else np.asarray(mapq)[order]
                strand = None if strand is None else np.asarray(strand)[order]
            if max_len is None:
                max_len = int((stop.astype(np.int64) - start).max()) if start.size else 0
            self.start = _to_device(start, self.device, np.int32)
            self.stop = _to_device(stop, self.device, np.int32)
            self.mapq = None if mapq is None else _to_device(mapq, self.device, np.uint8)
            self.strand = None if strand is None else _to_device(strand, self.device, np.uint8)
        else:
            self.start = start.to(self.device, t.int32).contiguous()
            self.stop = stop.to(self.device, t.int32).contiguous()
            self.mapq = None if mapq is None else mapq.to(self.device, t.uint8).contiguous()
            self.strand = None if strand is None else strand.to(self.device, t.uint8).contiguous()
            if max_len is None:
                max_len = int((self.stop - self.start).max().item()) if self.start.numel() else 0
        self.n = int(self.start.numel())
        self.max_len = max(int(max_len), 0)

    def ptrs(self):
        return (self.start.data_ptr(), self.stop.data_ptr(),
                0 if self.mapq is None else self.mapq.data_ptr())


class WpsPlan:
    """Tile table for a set of intervals of one contig (host-planned, HBM-resident).

    Mirrors what ``multi_wps`` hands to ``wps`` per interval
    (frag/_multi_wps.py:176-191): (start, stop, chrom_size) plus the padded
    fetch window of frag/_wps.py:156-157, expanded into <= FTK_WPS_TILE tiles.
    """

    def __init__(self, ivl_start, ivl_stop, chrom_size: int, max_length: int, device=None):
        self._install(self.host_tiles(ivl_start, ivl_stop, chrom_size, max_length), max_length, device)

    @staticmethod
    def host_tiles(ivl_start, ivl_stop, chrom_size: int, max_length: int) -> dict:
        """Plan the tiles of one contig's intervals on the host (``ftk_wps_plan_tiles``): numpy arrays
        ``p0, len, mid_lo, mid_hi`` (int32), ``out_off`` (int64), ``ivl`` (int32, bit 31 = the
        interval's first tile), ``offsets`` (int64[n_intervals + 1]: output offset of every interval)."""
        s = np.ascontiguousarray(ivl_start, dtype=np.int64)
        e = np.ascontiguousarray(ivl_stop, dtype=np.int64)
        ln = np.maximum(e - s, 0)
        offsets = np.zeros(len(s) + 1, dtype=np.int64)
        np.cumsum(ln, out=offsets[1:])
        L = lib()
        i64p, i32p = POINTER(c_int64), POINTER(c_int32)
        null32, null64 = i32p(), i64p()
        n_tiles = L.ftk_wps_plan_tiles(_np_ptr(s, c_int64), _np_ptr(e, c_int64), _np_ptr(offsets, c_int64),
                                       len(s), int(chrom_size), int(max_length), null32, null32, null32, null32, null64)
        check(n_tiles, "ftk_wps_plan_tiles")
        n_tiles = int(n_tiles)
        p0 = np.empty(n_tiles, np.int32)
        tl = np.empty(n_tiles, np.int32)
        mlo = np.empty(n_tiles, np.int32)
        mhi = np.empty(n_tiles, np.int32)
        off = np.empty(n_tiles, np.int64)
        if n_tiles:
            check(L.ftk_wps_plan_tiles(_np_ptr(s, c_int64), _np_ptr(e, c_int64), _np_ptr(offsets, c_int64),
                                       len(s), int(chrom_size), int(max_length), _np_ptr(p0, c_int32), _np_ptr(tl, c_int32),
                                       _np_ptr(mlo, c_int32), _np_ptr(mhi, c_int32), _np_ptr(off, c_int64)),
                  "ftk_wps_plan_tiles")
        # interval of each tile (empty intervals own no position, hence no tile)
        ivl = np.searchsorted(offsets[1:], off, side="right").astype(np.int64)
        first = off == offsets[np.minimum(ivl, len(s) - 1)] if n_tiles else np.zeros(0, bool)
        ivl = np.where(first, ivl - (1 << 31), ivl).astype(np.int32)   # bit 31: the interval's first tile
        return {"p0": p0, "len": tl, "mid_lo": mlo, "mid_hi": mhi, "out_off": off, "ivl": ivl, "offsets": offsets}

    @classmethod
    def from_tiles(cls, tiles: dict, max_length: int, device=None, n_positions: int | None = None):
        """A plan over an already planned (possibly merged, see ``distributed.GenomeShard``) tile table."""
        self = cls.__new__(cls)
        self._install(tiles, max_length, device, n_positions)
        return self

    def _install(self, tiles: dict, max_length: int, device=None, n_positions: int | None = None):
        t = torch()
        self.device = require_cuda(device)
        self.offsets = tiles["offsets"]
        self.n_positions = int(self.offsets[-1]) if n_positions is None else int(n_positions)
        self.max_length = int(max_length)
        self.n_tiles = int(len(tiles["p0"]))
        self.tile_p0 = _to_device(tiles["p0"], self.device, np.int32)
        self.tile_len = _to_device(tiles["len"], self.device, np.int32)
        self.tile_mid_lo = _to_device(tiles["mid_lo"], self.device, np.int32)
        self.tile_mid_hi = _to_device(tiles["mid_hi"], self.device, np.int32)
        self.tile_out_off = _to_device(tiles["out_off"], self.device, np.int64)
        self.n_intervals = len(self.offsets) - 1
        self.tile_ivl = _to_device(tiles["ivl"], self.device, np.int32)
        self.scratch = t.empty(2 * max(self.n_tiles, 1), dtype=t.int64, device=self.device)

    def ranges(self, frags: ContigFragments, window_size=120):
        """Only the per-tile fragment-range prepass (lets a caller time the main kernel alone)."""
        if self.n_tiles:
            _launch(self.device, "ftk_wps_tile_ranges", frags.start.data_ptr(), frags.n, self.tile_p0.data_ptr(),
                    self.tile_len.data_ptr(), self.n_tiles, int(window_size), self.max_length,
                    self.scratch.data_ptr())

    def run(self, frags: ContigFragments, window_size=120, min_length=120, max_length=180,
            quality_threshold=30, out=None, ranges_ready=False):
        """Launch the WPS kernels on the current stream; returns int32[n_positions] (device)."""
        t = torch()
        if int(max_length) != self.max_length:
            raise ValueError("plan was built for a different max_length")
        _same_device(self.device, frags)
        if out is None:
            out = t.empty(self.n_positions, dtype=t.int32, device=self.device)
        elif out.dtype != t.int32 or out.numel() < self.n_positions or not out.is_contiguous():
            raise ValueError("out must be a contiguous int32 tensor with n_positions elements")
        if self.n_tiles == 0:
            return out
        fs, fe, mq = frags.ptrs()
        _launch(self.device, "ftk_wps_tiles_i32",
            fs, fe, mq, frags.n,
            self.tile_p0.data_ptr(), self.tile_len.data_ptr(), self.tile_mid_lo.data_ptr(),
            self.tile_mid_hi.data_ptr(), self.tile_out_off.data_ptr(), self.n_tiles,
            int(window_size), none_to_ftk(min_length), int(max_length), int(quality_threshold),
            int(bool(ranges_ready)), self.scratch.data_ptr(), out.data_ptr())
        return out

    def ranges_fused(self, frags: ContigFragments, window_size=120, cov_max_length=None, zero_counts=None,
                     zero_hist=None):
        """Only the fragment-range prepass of ``run_fused`` (lets a caller time the main kernel alone).
        ``zero_counts`` / ``zero_hist``: int64 accumulators the prepass clears on the way (no extra launch)."""
        if self.n_tiles:
            _launch(self.device, "ftk_wps_cov_tile_ranges",
                frags.start.data_ptr(), frags.n, self.tile_p0.data_ptr(), self.tile_len.data_ptr(), self.n_tiles,
                int(window_size), self.max_length, none_to_ftk(cov_max_length), frags.max_len, self.scratch.data_ptr(),
                0 if zero_counts is None else zero_counts.data_ptr(), 0 if zero_counts is None else zero_counts.numel(),
                0 if zero_hist is None else zero_hist.data_ptr(), 0 if zero_hist is None else zero_hist.numel())
        else:
            for z in (zero_counts, zero_hist):
                if z is not None:
                    z.zero_()

    def run_fused(self, frags: ContigFragments, window_size=120, min_length=120, max_length=180,
                  quality_threshold=30, cov_min_length=None, cov_max_length=None, cov_quality_threshold=30,
                  n_bins=0, out=None, counts=None, hist=None, overflow=None, ranges_ready=False, zero_counts=False):
        """ONE pass over the fragments: WPS of every interval + per-interval midpoint coverage
        (``counts`` int64[n_intervals]) + the pooled length histogram of the counted fragments
        (``hist`` int64[n_bins]).  ``counts``/``hist`` are ACCUMULATED into (pass zeroed tensors to
        reuse buffers; ``zero_counts=True`` lets the range prepass clear ``counts`` first); ``out`` may be
        int32 / int16 / int8 (the narrow types need ``overflow``, an int32[1] flag the caller zeroes).
        Returns ``(wps, counts, hist)`` device tensors."""
        t = torch()
        if int(max_length) != self.max_length:
            raise ValueError("plan was built for a different max_length")
        _same_device(self.device, frags)
        if out is None:
            out = t.empty(self.n_positions, dtype=t.int32, device=self.device)
        kind = {t.int32: 0, t.int16: 1, t.int8: 2}.get(out.dtype)
        if kind is None or out.numel() < self.n_positions or not out.is_contiguous():
            raise ValueError("out must be a contiguous int32/int16/int8 tensor with n_positions elements")
        if kind and overflow is None:
            raise ValueError("int16/int8 output needs an overflow flag tensor")
        if counts is None:
            counts = t.zeros(max(self.n_intervals, 1), dtype=t.int64, device=self.device)
        if hist is None and n_bins:
            hist = t.zeros(int(n_bins), dtype=t.int64, device=self.device)
        if zero_counts and not ranges_ready:   # the range prepass clears ``counts`` on the way: no memset launch
            self.ranges_fused(frags, window_size, cov_max_length, zero_counts=counts)
            ranges_ready = True
        if self.n_tiles == 0:
            return out, counts[: self.n_intervals], hist
        fs, fe, mq = frags.ptrs()
        _launch(self.device, "ftk_wps_cov_tiles",
            fs, fe, mq, frags.n, frags.max_len,
            self.tile_p0.data_ptr(), self.tile_len.data_ptr(), self.tile_mid_lo.data_ptr(),
            self.tile_mid_hi.data_ptr(), self.tile_out_off.data_ptr(), self.tile_ivl.data_ptr(), self.n_tiles,
            int(window_size), none_to_ftk(min_length), int(max_length), int(quality_threshold),
            none_to_ftk(cov_min_length), none_to_ftk(cov_max_length), int(cov_quality_threshold), int(n_bins),
            int(bool(ranges_ready)), self.scratch.data_ptr(), kind, out.data_ptr(), 0 if overflow is None else overflow.data_ptr(),
            counts.data_ptr(), 0 if hist is None else hist.data_ptr())
        return out, counts[: self.n_intervals], hist


_POLICY = {"midpoint": 0, "any": 1}
_TARGET_CTAS = 148 * 8  # SM count x resident CTAs: enough slices to fill the chip
_UNIT_FRAGS = 8192      # fragments per (interval, split) unit: 8 K measured best for Mb-scale bins (2 K: +10 %, 32 K: +7 %)


def policy_code(intersect_policy: str) -> int:
    """utils/_frag_generator.py:52-53: unknown policy -> InvalidInputError."""
    try:
        return _POLICY[intersect_policy]
    except KeyError:
        from .exceptions import InvalidInputError
        raise InvalidInputError(f"{intersect_policy} is not a valid policy") from None


def _splits_for(n_ivl: int, n_frag: int, unit_frags: int | None = None) -> int:
    """Slices per interval.  A unit (one warp, or one CTA for per-interval histograms) should hold
    about ``_UNIT_FRAGS`` candidate fragments - few enough that its loads are all in flight at
    once, many enough to amortise its descriptor fetch - and there should be at least a few
    waves of units; estimated from the contig-wide mean fragments per interval."""
    if n_ivl <= 0:
        return 1
    unit = _UNIT_FRAGS if unit_frags is None else int(unit_frags)
    by_size = -(-(n_frag // max(n_ivl, 1)) // unit)
    by_grid = -(-4 * _TARGET_CTAS // n_ivl)
    return int(max(1, min(max(by_size, by_grid), 65536)))


def _ivl_to_device(ivl_start, ivl_stop, device):
    if isinstance(ivl_start, np.ndarray) and isinstance(ivl_stop, np.ndarray) and ivl_start.dtype.kind in "iu" \
            and ivl_stop.dtype.kind in "iu":
        lim = 2 ** 31 - 1
        return (_to_device(np.clip(ivl_start, -lim, lim), device, np.int32),
                _to_device(np.clip(ivl_stop, -lim, lim), device, np.int32))
    s = np.array([FTK_NONE if v is None else int(v) for v in ivl_start], dtype=np.int64)
    e = np.array([FTK_NONE if v is None else int(v) for v in ivl_stop], dtype=np.int64)
    lim = 2 ** 31 - 1
    s = np.where(s == FTK_NONE, FTK_NONE, np.clip(s, -lim, lim)).astype(np.int32)
    e = np.where(e == FTK_NONE, FTK_NONE, np.clip(e, -lim, lim)).astype(np.int32)
    return _to_device(s, device, np.int32), _to_device(e, device, np.int32)


class IntervalSet:
    """Interval table of one contig resident in HBM (+ the per-interval range scratch)."""

    def __init__(self, ivl_start, ivl_stop, device=None):
        self.device = require_cuda(device)
        self.n = len(ivl_start)
        if self.n:
            self.start, self.stop = _ivl_to_device(ivl_start, ivl_stop, self.device)
        else:
            self.start = self.stop = None
        self.scratch = torch().empty(2 * max(self.n, 1), dtype=torch().int64, device=self.device)


def interval_hist(frags: ContigFragments, ivl_start=None, ivl_stop=None, intersect_policy="midpoint",
                  min_length=None, max_length=None, quality_threshold=30, n_bins=0,
                  pooled=False, first_seen=False, ivl_set: IntervalSet | None = None, out=None):
    """Counts (and optional length histograms) of the fragment stream of each interval.

    Returns device tensors ``(counts int64[rows], hist int64[rows, n_bins] | None,
    first int32[rows, n_bins] | None)``; rows = 1 when ``pooled``.  ``ivl_set`` /
    ``out=(counts, hist, first)`` let a caller reuse device buffers (outputs accumulate).
    """
    t = torch()
    dev = frags.device
    if ivl_set is None:
        ivl_set = IntervalSet(ivl_start, ivl_stop, dev)
    n_ivl = ivl_set.n
    pool_mode = {False: 0, True: 1, "hist": 2}[pooled]   # "hist": per-interval counts + one pooled histogram
    rows = 1 if pool_mode == 1 else n_ivl
    if out is not None:
        counts, hist, first = out
    else:
        hrows = 1 if pool_mode else rows
        counts = t.zeros(max(rows, 1), dtype=t.int64, device=dev)
        hist = t.zeros((max(hrows, 1), n_bins), dtype=t.int64, device=dev) if n_bins else None
        first = (t.full((max(hrows, 1), n_bins), 2 ** 31 - 1, dtype=t.int32, device=dev)
                 if (n_bins and first_seen) else None)
    if n_ivl == 0:
        return counts[:rows], hist, first
    fs, fe, mq = frags.ptrs()
    _launch(dev, "ftk_interval_hist_u64",
        fs, fe, mq, frags.n, frags.max_len, ivl_set.start.data_ptr(), ivl_set.stop.data_ptr(), n_ivl,
        policy_code(intersect_policy), none_to_ftk(min_length), none_to_ftk(max_length),
        int(quality_threshold), int(n_bins), pool_mode, _splits_for(n_ivl, frags.n),
        ivl_set.scratch.data_ptr(), counts.data_ptr(), 0 if hist is None else hist.data_ptr(),
        0 if first is None else first.data_ptr())
    return counts[:rows], hist, first


VPLOT_MAX_FLANK = 1 << 20
VPLOT_MAX_CELLS = 1 << 27


def vplot_check(flank, min_length, max_length):
    """ValueError unless ``0 <= min_length <= max_length`` (integers), ``0 <= flank <= 2**20`` and the matrix has at
    most 2**27 cells; returns its shape ``(max_length - min_length + 1, 2 * flank + 1)``."""
    if min_length is None or max_length is None:
        raise ValueError("min_length and max_length must both be given (the rows of the V-plot matrix)")
    flank, min_length, max_length = int(flank), int(min_length), int(max_length)
    if min_length < 0 or max_length < min_length:
        raise ValueError(f"need 0 <= min_length <= max_length, got {min_length} and {max_length}")
    if flank < 0 or flank > VPLOT_MAX_FLANK:
        raise ValueError(f"flank must lie in [0, {VPLOT_MAX_FLANK}], got {flank}")
    shape = (max_length - min_length + 1, 2 * flank + 1)
    if shape[0] * shape[1] > VPLOT_MAX_CELLS:
        raise ValueError(f"a {shape[0]} x {shape[1]} V-plot exceeds {VPLOT_MAX_CELLS} cells")
    return shape


def _site_windows(c: np.ndarray, site_flip, flank: int, dev):
    """The windows ``[c - flank, c + flank + 1)`` of site centres ``c`` (int64, non-empty) as an ``IntervalSet``, and
    the flip flags as a device uint8 column."""
    lim = 2 ** 31 - 1
    if int(c.min()) - flank < -lim or int(c.max()) > lim:
        raise ValueError("site centres must lie within the int32 coordinate range")
    # centre = window start + flank; a window that ends past 2**31 - 1 has no upper bound (None), since a stop
    # clipped to 2**31 - 1 would drop a fragment starting there
    hi = c + flank + 1
    sites = IntervalSet(c - flank, hi if int(hi.max()) <= lim else [None if v > lim else v for v in hi.tolist()], dev)
    flip = _to_device(np.asarray(site_flip, dtype=bool).reshape(-1).astype(np.uint8), dev, np.uint8)
    return sites, flip


def vplot_sites(frags: ContigFragments, site_center, site_flip, flank, min_length, max_length, quality_threshold=30,
                out=None):
    """Fragment-length x midpoint-offset counts summed over the sites of one contig (``ftk_vplot_u64``).

    Site k is centred on ``site_center[k]`` and mirrored when ``site_flip[k]`` is true; a passing fragment (mapq >=
    ``quality_threshold``, ``min_length <= L <= max_length``) whose midpoint ``(start + stop) // 2`` lies within
    ``flank`` of the centre adds 1 at ``[L - min_length, offset + flank]``.  Returns the device int64 matrix of
    shape ``(max_length - min_length + 1, 2 * flank + 1)``; ``out`` (such a matrix) is accumulated into."""
    t = torch()
    shape = vplot_check(flank, min_length, max_length)
    dev = frags.device
    if out is None:
        out = t.zeros(shape, dtype=t.int64, device=dev)
    elif out.dtype != t.int64 or tuple(out.shape) != shape or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous int64 tensor of shape {shape}")
    c = np.asarray(site_center, dtype=np.int64).reshape(-1)
    n = c.size
    if n == 0:
        return out
    flank = int(flank)
    sites, flip = _site_windows(c, site_flip, flank, dev)
    fs, fe, mq = frags.ptrs()
    _launch(dev, "ftk_vplot_u64",
        fs, fe, mq, frags.n, frags.max_len, sites.start.data_ptr(), sites.stop.data_ptr(), flip.data_ptr(), n,
        flank, int(min_length), int(max_length), int(quality_threshold), _splits_for(n, frags.n),
        sites.scratch.data_ptr(), out.data_ptr())
    return out


OCF_MAX_FLANK = 8192          # FTK_OCF_MAX_FLANK
OCF_MAX_CELLS = 1 << 27       # FTK_OCF_MAX_CELLS
# A CTA of the OCF kernel adds its 32-bit shared counters to the output before the candidate fragments it has taken
# since its last flush could pass this (one candidate adds at most 1 to a counter).  Tests set it small.
OCF_FLUSH_CANDIDATES = 2 ** 32 - 1


def _ocf_shape(flank, n_sets):
    if isinstance(flank, bool) or int(flank) != flank or not 0 <= int(flank) <= OCF_MAX_FLANK:
        raise ValueError(f"flank must be an integer in [0, {OCF_MAX_FLANK}], got {flank!r}")
    if isinstance(n_sets, bool) or int(n_sets) != n_sets or int(n_sets) < 1:
        raise ValueError(f"need at least one site set, got {n_sets!r}")
    shape = (int(n_sets), 2, 2 * int(flank) + 1)
    if shape[0] * shape[1] * shape[2] > OCF_MAX_CELLS:
        raise ValueError(f"{shape[0]} site sets x 2 x {shape[2]} offsets exceed {OCF_MAX_CELLS} cells")
    return shape


def ocf_check(flank, peak_offset, peak_width, n_sets):
    """ValueError unless ``0 <= flank <= 8192``, ``n_sets >= 1`` and the peak windows ``P+ = [o - w // 2,
    o - w // 2 + w)`` and ``P- = -P+`` (``o = peak_offset``, ``w = peak_width``, integers) satisfy ``w >= 1``,
    ``o - w // 2 >= 1`` and ``o - w // 2 + w - 1 <= flank``; returns the shape ``(n_sets, 2, 2 * flank + 1)`` of
    the end-count matrix."""
    shape = _ocf_shape(flank, n_sets)
    for name, v in (("peak_offset", peak_offset), ("peak_width", peak_width)):
        if isinstance(v, bool) or not isinstance(v, (int, np.integer)):
            raise ValueError(f"{name} must be an integer, got {v!r}")
    o, w, f = int(peak_offset), int(peak_width), int(flank)
    if w < 1 or o - w // 2 < 1 or o - w // 2 + w - 1 > f:
        raise ValueError(f"the peak window [{o - w // 2}, {o - w // 2 + w - 1}] (peak_offset {o}, peak_width {w}) "
                         f"must have a width >= 1 and lie within [1, flank = {f}]")
    return shape


def ocf_length_check(min_length, max_length) -> None:
    """ValueError unless each bound is None (unbounded) or an integer in [0, 2**31 - 1] and min <= max."""
    for name, v in (("min_length", min_length), ("max_length", max_length)):
        if v is not None and (isinstance(v, bool) or int(v) != v or not 0 <= int(v) <= 2 ** 31 - 1):
            raise ValueError(f"{name} must be None or an integer in [0, 2**31 - 1], got {v!r}")
    if min_length is not None and max_length is not None and int(max_length) < int(min_length):
        raise ValueError(f"need min_length <= max_length, got {min_length} and {max_length}")


def _ocf_cta_bounds(site_set: np.ndarray, n_sets: int, splits: int) -> np.ndarray:
    """Unit boundaries of the OCF kernel's CTAs over sites sorted by set (unit = site * splits + slice): each set's
    units are split into about ``_TARGET_CTAS`` * (its share of the units) CTAs of at least 8 units (one per warp)
    where it has that many; no CTA crosses a set."""
    per_set = np.bincount(site_set, minlength=n_sets).astype(np.int64) * splits
    total = int(per_set.sum())
    bounds, first = [0], 0
    for u in per_set.tolist():
        if u == 0:
            continue
        n_cta = max(1, min(-(-u // 8), -(-u * _TARGET_CTAS // total)))
        bounds += [first + u * j // n_cta for j in range(1, n_cta + 1)]
        first += u
    return np.asarray(bounds, dtype=np.int32)


def ocf_sites(frags: ContigFragments, site_center, site_flip, site_set, n_sets, flank, min_length=None,
              max_length=None, quality_threshold=30, out=None):
    """Upstream- and downstream-end offset counts around the sites of one contig, summed per site set
    (``ftk_ocf_u64``).

    Site k is centred on ``site_center[k]``, mirrored when ``site_flip[k]`` is true and belongs to set
    ``site_set[k]`` (``0 <= site_set[k] < n_sets``).  A fragment ``[s, e)`` passes when mapq >=
    ``quality_threshold`` and ``max(1, min_length) <= e - s <= max_length`` (None = unbounded).  Its upstream end
    offset is ``s - c`` and its downstream one ``e - 1 - c`` (mirrored: ``c - (e - 1)`` and ``c - s``); each end
    within ``flank`` of the centre adds 1 at ``[set, 0, x + flank]`` (upstream) or ``[set, 1, x + flank]``
    (downstream).  Returns the device int64 tensor of shape ``(n_sets, 2, 2 * flank + 1)``; ``out`` (such a tensor)
    is accumulated into."""
    t = torch()
    shape = _ocf_shape(flank, n_sets)
    ocf_length_check(min_length, max_length)
    dev = frags.device
    if out is None:
        out = t.zeros(shape, dtype=t.int64, device=dev)
    elif out.dtype != t.int64 or tuple(out.shape) != shape or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous int64 tensor of shape {shape}")
    c = np.asarray(site_center, dtype=np.int64).reshape(-1)
    n = c.size
    s = np.asarray(site_set, dtype=np.int64).reshape(-1)
    f = np.asarray(site_flip, dtype=bool).reshape(-1)
    if s.size != n or f.size != n:
        raise ValueError(f"site_center, site_flip and site_set must have the same length, got {n}, {f.size}, {s.size}")
    if n == 0:
        return out
    if int(s.min()) < 0 or int(s.max()) >= shape[0]:
        raise ValueError(f"site sets must lie in [0, {shape[0]})")
    flank = int(flank)
    # a CTA counts one set; 16-bit keys take numpy's linear-time radix sort
    order = np.argsort(s.astype(np.uint16) if shape[0] <= 1 << 16 else s, kind="stable")
    c, f, s = c[order], f[order], s[order]
    sites, flip = _site_windows(c, f, flank, dev)
    splits = _splits_for(n, frags.n)
    bounds = _ocf_cta_bounds(s, shape[0], splits)
    tab = _to_device(np.concatenate([s.astype(np.int32), bounds]), dev, np.int32)
    fs, fe, mq = frags.ptrs()
    _launch(dev, "ftk_ocf_u64",
        fs, fe, mq, frags.n, frags.max_len, sites.start.data_ptr(), sites.stop.data_ptr(), flip.data_ptr(),
        tab.data_ptr(), n, shape[0], flank, none_to_ftk(min_length), none_to_ftk(max_length), int(quality_threshold),
        splits, tab[n:].data_ptr(), bounds.size - 1, int(OCF_FLUSH_CANDIDATES), sites.scratch.data_ptr(),
        out.data_ptr())
    return out


GC_MAX_LENGTH = 1024   # FTK_GC_MAX_LENGTH
GC_MAX_TILE = 16384    # FTK_GC_MAX_TILE


def gc_check(min_length, max_length):
    """ValueError unless ``1 <= min_length <= max_length <= 1024`` (integers); returns the shape of the GC-bias
    matrices ``(max_length - min_length + 1, max_length + 1)``."""
    if min_length is None or max_length is None or isinstance(min_length, bool) or isinstance(max_length, bool) \
            or int(min_length) != min_length or int(max_length) != max_length:
        raise ValueError(f"min_length and max_length must be integers, got {min_length!r} and {max_length!r}")
    min_length, max_length = int(min_length), int(max_length)
    if not 1 <= min_length <= max_length <= GC_MAX_LENGTH:
        raise ValueError(f"need 1 <= min_length <= max_length <= {GC_MAX_LENGTH}, got {min_length} and {max_length}")
    return (max_length - min_length + 1, max_length + 1)


def _gc_out(shape, out, dev):
    t = torch()
    if out is None:
        return t.zeros(shape, dtype=t.int64, device=dev)
    if out.dtype != t.int64 or tuple(out.shape) != shape or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous int64 tensor of shape {shape}")
    return out


def _gc_regions(reg_start, reg_stop):
    s = np.asarray(reg_start, dtype=np.int64).reshape(-1)
    e = np.asarray(reg_stop, dtype=np.int64).reshape(-1)
    if s.shape != e.shape:
        raise ValueError("reg_start and reg_stop must have the same length")
    return s, e


def gc_observed(frags: ContigFragments, ref: PackedContig, reg_start, reg_stop, min_length, max_length,
                quality_threshold=30, out=None):
    """Fragment counts by (length, G+C bases) of one contig (``ftk_gc_observed_u64``).

    A fragment ``[s, e)`` with ``mapq >= quality_threshold`` and ``min_length <= L <= max_length`` adds 1 at
    ``[L - min_length, g]`` (g = C/G bases of ``[s, e)``) when its midpoint ``(s + e) // 2`` lies in one of the regions
    (sorted, disjoint, clipped to ``[0, ref.length]``), ``0 <= s``, ``e <= ref.length`` and no base of it is N.
    Returns the device int64 matrix of shape ``(max_length - min_length + 1, max_length + 1)``; ``out`` (such a
    matrix) is accumulated into."""
    shape = gc_check(min_length, max_length)
    _same_device(frags.device, ref)
    out = _gc_out(shape, out, frags.device)
    s, e = _gc_regions(reg_start, reg_stop)
    n = s.size
    if n == 0:
        return out
    regs = IntervalSet(s, e, frags.device)
    fs, fe, mq = frags.ptrs()
    _launch(frags.device, "ftk_gc_observed_u64",
        fs, fe, mq, frags.n, frags.max_len, ref.seq.data_ptr(), ref.nmask.data_ptr(), ref.length,
        regs.start.data_ptr(), regs.stop.data_ptr(), n, int(min_length), int(max_length), int(quality_threshold),
        _splits_for(n, frags.n), regs.scratch.data_ptr(), out.data_ptr())
    return out


def _gc_tile_for(max_length: int) -> int:
    """Midpoints per ``gc_expected_kernel`` CTA: long enough that the flush of its ``32 x (max_length + 1)`` bins is
    small next to its ``32 x tile`` placements, short enough that two CTAs of lengths <= 500 share an SM."""
    return 8192


def gc_tiles(reg_start, reg_stop, tile: int):
    """The regions cut into consecutive midpoint tiles of at most ``tile`` positions: ``(lo, hi)`` int64 arrays."""
    s, e = _gc_regions(reg_start, reg_stop)
    n = np.maximum(-(-(e - s) // tile), 0)
    first = np.repeat(s, n)
    k = np.arange(int(n.sum()), dtype=np.int64) - np.repeat(np.cumsum(n) - n, n)
    lo = first + k * tile
    return lo, np.minimum(lo + tile, np.repeat(e, n))


def gc_expected(ref: PackedContig, reg_start, reg_stop, min_length, max_length, out=None):
    """Counts by (length, G+C bases) of every placement of one contig (``ftk_gc_expected_u64``).

    Every ``[p, p + L)`` with ``min_length <= L <= max_length``, ``p >= 0``, ``p + L <= ref.length``, its midpoint
    ``p + L // 2`` in one of the regions (sorted, disjoint, clipped) and no N base adds 1 at ``[L - min_length, g]``.
    Returns the device int64 matrix of shape ``(max_length - min_length + 1, max_length + 1)``; ``out`` is
    accumulated into."""
    shape = gc_check(min_length, max_length)
    out = _gc_out(shape, out, ref.device)
    tile = int(_gc_tile_for(int(max_length)))
    if not 1 <= tile <= GC_MAX_TILE:
        raise ValueError(f"the midpoint tile must lie in [1, {GC_MAX_TILE}], got {tile}")
    lo, hi = gc_tiles(reg_start, reg_stop, tile)
    if lo.size == 0:
        return out
    d_lo, d_hi = _to_device(lo, ref.device, np.int32), _to_device(hi, ref.device, np.int32)
    _launch(ref.device, "ftk_gc_expected_u64",
        ref.seq.data_ptr(), ref.nmask.data_ptr(), ref.length, d_lo.data_ptr(), d_hi.data_ptr(), lo.size, tile,
        int(min_length), int(max_length), out.data_ptr())
    return out


def gc_weights_to_device(weights, shape, dev):
    """The weight table as a contiguous float64 device tensor; ValueError unless it has ``shape`` and every entry is
    finite and ``>= 0``."""
    t = torch()
    w = weights if t.is_tensor(weights) else t.from_numpy(np.asarray(weights, dtype=np.float64))
    if tuple(w.shape) != tuple(shape):
        raise ValueError(f"the weight table must have shape {tuple(shape)}, got {tuple(w.shape)}")
    w = w.to(dev, t.float64).contiguous()
    if not bool((t.isfinite(w) & (w >= 0)).all()):
        raise ValueError("the weight table must hold finite, non-negative values")
    return w


def _gc_weighted_out(n, out, dev):
    t = torch()
    if out is None:
        return t.zeros(n, dtype=t.int64, device=dev), t.zeros(n, dtype=t.float64, device=dev)
    count, corrected = out
    for x, dt in ((count, t.int64), (corrected, t.float64)):
        if x.dtype != dt or tuple(x.shape) != (n,) or not x.is_contiguous():
            raise ValueError(f"out must be contiguous (int64, float64) tensors of shape ({n},)")
    return count, corrected


def gc_weighted_intervals(frags: ContigFragments, ref: PackedContig, ivl_start, ivl_stop, weights, min_length,
                          max_length, quality_threshold=30, out=None):
    """Plain and GC-weighted fragment counts of each interval of one contig (``ftk_gc_weighted_intervals_f64``).

    A fragment ``[s, e)`` with ``mapq >= quality_threshold``, ``min_length <= L <= max_length`` and its midpoint
    ``(s + e) // 2`` in ``[ivl_start[k], ivl_stop[k])`` (None = unbounded) adds 1 to ``count[k]``, and
    ``weights[L - min_length, g]`` to ``corrected[k]`` when ``0 <= s``, ``e <= ref.length`` and no base of it is N
    (g = its C/G bases).  ``weights``: float64 of the GC-bias matrices' shape, finite and non-negative.  Returns
    device tensors ``(count int64[n], corrected float64[n])``; ``out`` (such a pair) is accumulated into.  The
    corrected sums are bit-identical between runs with the same slice count."""
    shape = gc_check(min_length, max_length)
    dev = frags.device
    _same_device(dev, ref)
    n = len(ivl_start)
    if len(ivl_stop) != n:
        raise ValueError("ivl_start and ivl_stop must have the same length")
    w = gc_weights_to_device(weights, shape, dev)
    count, corrected = _gc_weighted_out(n, out, dev)
    if n == 0:
        return count, corrected
    ivl = IntervalSet(ivl_start, ivl_stop, dev)
    splits = _splits_for(n, frags.n)
    scratch = torch().empty(2 * n + 2 * n * splits, dtype=torch().int64, device=dev)
    fs, fe, mq = frags.ptrs()
    _launch(dev, "ftk_gc_weighted_intervals_f64",
        fs, fe, mq, frags.n, frags.max_len, ref.seq.data_ptr(), ref.nmask.data_ptr(), ref.length,
        ivl.start.data_ptr(), ivl.stop.data_ptr(), n, int(min_length), int(max_length), int(quality_threshold), splits,
        scratch.data_ptr(), w.data_ptr(), count.data_ptr(), corrected.data_ptr())
    return count, corrected


def gc_weighted_sites(frags: ContigFragments, ref: PackedContig, site_center, site_flip, flank, weights, min_length,
                      max_length, quality_threshold=30, out=None):
    """Plain and GC-weighted fragment-midpoint profiles around the sites of one contig (``ftk_gc_weighted_sites_f64``).

    Site k is centred on ``site_center[k]`` and mirrored when ``site_flip[k]`` is true; a fragment selected as in
    ``gc_weighted_intervals`` whose midpoint lies within ``flank`` of the centre adds 1 to ``count[offset + flank]``
    and its weight to ``corrected[offset + flank]``.  Returns device tensors ``(count int64[2 * flank + 1],
    corrected float64[2 * flank + 1])`` summed over the sites; ``out`` is accumulated into.  The corrected sums are
    fp64 atomics, so their last bits may vary between runs."""
    shape = gc_check(min_length, max_length)
    flank = int(flank)
    if not 0 <= flank <= VPLOT_MAX_FLANK:
        raise ValueError(f"flank must lie in [0, {VPLOT_MAX_FLANK}], got {flank}")
    dev = frags.device
    _same_device(dev, ref)
    w = gc_weights_to_device(weights, shape, dev)
    count, corrected = _gc_weighted_out(2 * flank + 1, out, dev)
    c = np.asarray(site_center, dtype=np.int64).reshape(-1)
    n = c.size
    if n == 0:
        return count, corrected
    sites, flip = _site_windows(c, site_flip, flank, dev)
    fs, fe, mq = frags.ptrs()
    _launch(dev, "ftk_gc_weighted_sites_f64",
        fs, fe, mq, frags.n, frags.max_len, ref.seq.data_ptr(), ref.nmask.data_ptr(), ref.length,
        sites.start.data_ptr(), sites.stop.data_ptr(), flip.data_ptr(), n, flank, int(min_length), int(max_length),
        int(quality_threshold), _splits_for(n, frags.n), sites.scratch.data_ptr(), w.data_ptr(), count.data_ptr(),
        corrected.data_ptr())
    return count, corrected


SPECTRUM_MAX_PERIOD = 1024   # FTK_SPECTRUM_MAX_PERIOD


def spectrum_check(min_period, max_period) -> int:
    """ValueError unless ``2 <= min_period <= max_period <= 1024`` (integers); returns the number of periods."""
    if min_period is None or max_period is None or isinstance(min_period, bool) or isinstance(max_period, bool) \
            or int(min_period) != min_period or int(max_period) != max_period:
        raise ValueError(f"min_period and max_period must be integers, got {min_period!r} and {max_period!r}")
    if not 2 <= int(min_period) <= int(max_period) <= SPECTRUM_MAX_PERIOD:
        raise ValueError(f"need 2 <= min_period <= max_period <= {SPECTRUM_MAX_PERIOD}, got {min_period} and "
                         f"{max_period}")
    return int(max_period) - int(min_period) + 1


def spectrum_segments(x, offsets, min_period=120, max_period=280, out=None):
    """Periodogram of every segment at the integer periods ``min_period .. max_period`` (``ftk_spectrum_*_f64``).

    ``x``: an int32 or float64 CUDA tensor holding the segments back to back; segment s is
    ``x[offsets[s]:offsets[s + 1]]`` (host int64 offsets, non-decreasing).  With N values of mean mu,
    ``I(P) = |sum_n (x[n] - mu) exp(-2 pi i (n mod P) / P)|^2 / N``; an empty segment gives a row of NaN.  Returns the
    device float64 matrix ``[n_seg, n_periods]`` (``out``, such a matrix, is written).  Bit-identical from run to
    run; a segment's row does not depend on the other segments."""
    t = torch()
    n_p = spectrum_check(min_period, max_period)
    if not (t.is_tensor(x) and x.is_cuda and x.dtype in (t.int32, t.float64)):
        raise ValueError("x must be an int32 or float64 CUDA tensor")
    dev = x.device
    off = np.asarray(offsets, dtype=np.int64).reshape(-1)
    if off.size == 0 or off[0] < 0 or (np.diff(off) < 0).any() or off[-1] > x.numel():
        raise ValueError("offsets must be non-decreasing, start at >= 0 and end within x")
    shape = (off.size - 1, n_p)
    if out is None:
        out = t.empty(shape, dtype=t.float64, device=dev)
    elif out.dtype != t.float64 or tuple(out.shape) != shape or not out.is_contiguous() or out.device != dev:
        raise ValueError(f"out must be a contiguous float64 tensor of shape {shape} on {dev}")
    if shape[0] == 0:
        return out
    xd = x.contiguous() if x.numel() else t.zeros(1, dtype=x.dtype, device=dev)
    d_off = _to_device(off, dev, np.int64)
    name = "ftk_spectrum_i32_f64" if xd.dtype == t.int32 else "ftk_spectrum_f64_f64"
    _launch(dev, name, xd.data_ptr(), d_off.data_ptr(), shape[0], int(min_period), int(max_period), out.data_ptr())
    return out


def frag_lengths(frags: ContigFragments, start=None, stop=None, intersect_policy="midpoint",
                 min_length=0, max_length=1000000000, quality_threshold=30):
    """int32 lengths of the stream of one region, in stream order (device tensor)."""
    t = torch()
    dev = frags.device
    nb = (frags.n + 1023) // 1024 + 1
    scratch = t.empty(2 + nb + (nb + 1) // 2, dtype=t.int64, device=dev)
    out = t.empty(max(frags.n, 1), dtype=t.int32, device=dev)
    n_out = t.zeros(1, dtype=t.int64, device=dev)
    fs, fe, mq = frags.ptrs()
    _launch(dev, "ftk_frag_lengths_i32",
        fs, fe, mq, frags.n, frags.max_len, none_to_ftk(start), none_to_ftk(stop),
        policy_code(intersect_policy), none_to_ftk(min_length), none_to_ftk(max_length),
        int(quality_threshold), scratch.data_ptr(), scratch.numel(), out.data_ptr(),
        n_out.data_ptr())
    return out[: int(n_out.item())]


class PackedContig:
    """2-bit packed reference contig + N mask in HBM (layout: synth.pack_twobit)."""

    def __init__(self, seq_words: np.ndarray, nmask_words: np.ndarray, length: int, device=None):
        self.device = require_cuda(device)
        self.length = int(length)
        self.seq = _to_device(seq_words, self.device, np.uint32)
        self.nmask = _to_device(nmask_words, self.device, np.uint32)

    @classmethod
    def from_codes(cls, codes: np.ndarray, n_mask: np.ndarray, device=None):
        from .synth import pack_twobit
        sw, nw = pack_twobit(codes, n_mask)
        return cls(sw, nw, codes.shape[0], device)


def end_motif_hist(frags: ContigFragments, ref: PackedContig, ivl_start, ivl_stop, k=4,
                   strand_mode=0, quality_threshold=20, pooled=False, counts=None, breakpoint=False):
    """k-mer counts int64[rows, 4**k] (device); raises RuntimeError like the reference.

    ``breakpoint=True`` counts k-mers centred on the breakpoints (frag/_breakpoint_motifs.py)
    instead of 5' end motifs; that variant has no error path."""
    t = torch()
    dev = frags.device
    _same_device(dev, ref)
    n_ivl = len(ivl_start)
    rows = 1 if pooled else n_ivl
    if counts is None:
        counts = t.zeros((max(rows, 1), 4 ** k), dtype=t.int64, device=dev)
    if n_ivl == 0:
        return counts[:rows]
    ivl = IntervalSet(ivl_start, ivl_stop, dev)
    err = t.zeros(1, dtype=t.int32, device=dev)
    fs, fe, mq = frags.ptrs()
    sd = 0 if frags.strand is None else frags.strand.data_ptr()
    # a CTA's fixed latency chain (ranges -> slice bounds -> N pre-scan -> first fragments -> windows) is
    # paid once per slice: 16 K fragments amortise it (and the zero + flush of a 4^k-bin histogram)
    splits = _splits_for(n_ivl, frags.n, unit_frags=max(16384, 16 * 4 ** min(int(k), 6)))
    if breakpoint:
        _launch(dev, "ftk_breakpoint_motif_hist_u64",
            fs, fe, mq, sd, frags.n, frags.max_len, ref.seq.data_ptr(), ref.nmask.data_ptr(), ref.length,
            ivl.start.data_ptr(), ivl.stop.data_ptr(), n_ivl, int(k), int(strand_mode), int(quality_threshold),
            int(bool(pooled)), splits, ivl.scratch.data_ptr(), counts.data_ptr())
        return counts[:rows]
    _launch(dev, "ftk_end_motif_hist_u64",
        fs, fe, mq, sd, frags.n, frags.max_len, ref.seq.data_ptr(), ref.nmask.data_ptr(), ref.length,
        ivl.start.data_ptr(), ivl.stop.data_ptr(), n_ivl, int(k), int(strand_mode), int(quality_threshold),
        int(bool(pooled)), splits, ivl.scratch.data_ptr(), counts.data_ptr(),
        err.data_ptr())
    if int(err.item()):
        raise RuntimeError(
            "Error querying sequence: reverse k-mer window out of contig bounds. Please verify "
            "that the reference file matches the fragment file.")
    return counts[:rows]


def blacklist_in_windows(bl_start, bl_stop, win_start, win_stop):
    """Blacklist regions contained in each window (frag/_delfi.py:110-127), as CSR (host).

    ``bl_start``/``bl_stop``: the contig's regions sorted by (start, stop).  A region belongs to a
    window when ``start >= window_start`` and ``stop <= window_stop``.  Returns
    ``(off int32[n_win+1], starts int32, stops int32)``."""
    bs = np.asarray(bl_start, dtype=np.int64); be = np.asarray(bl_stop, dtype=np.int64)
    ws = np.asarray(win_start, dtype=np.int64); we = np.asarray(win_stop, dtype=np.int64)
    off = np.zeros(len(ws) + 1, dtype=np.int64)
    if not bs.size or not ws.size:
        return off.astype(np.int32), np.zeros(0, np.int32), np.zeros(0, np.int32)
    lo = np.searchsorted(bs, ws, side="left")
    # a contained region starts before the window stops: bound the scan with a second search
    cnt = np.maximum(np.searchsorted(bs, we, side="right") - lo, 0)
    win = np.repeat(np.arange(len(ws)), cnt)                          # candidate (window, region) pairs
    reg = lo[win] + (np.arange(win.size) - np.repeat(np.cumsum(cnt) - cnt, cnt))
    keep = be[reg] <= we[win]
    win, reg = win[keep], reg[keep]
    np.cumsum(np.bincount(win, minlength=len(ws)), out=off[1:])
    return off.astype(np.int32), bs[reg].astype(np.int32), be[reg].astype(np.int32)


def delfi_windows(frags: ContigFragments, ref: PackedContig | None, win_start, win_stop, blacklist=None,
                  gaps=None, quality_threshold=30):
    """DELFI bin counts of one contig: int64[n_win, 4] = short, long, num_frags, G+C bases (device).

    ``blacklist`` = (starts, stops) of the contig sorted by (start, stop); ``gaps`` = (centromere
    (start, stop), [telomere (start, stop), ...]) or None (frag/_delfi.py:404-511)."""
    t = torch()
    dev = frags.device
    _same_device(dev, *([] if ref is None else [ref]))
    n_win = len(win_start)
    counts = t.zeros((max(n_win, 1), 4), dtype=t.int64, device=dev)
    if n_win == 0:
        return counts[:0]
    win = IntervalSet(win_start, win_stop, dev)
    fs, fe, mq = frags.ptrs()
    bl = (0, 0, 0)
    keep = []
    if blacklist is not None and len(blacklist[0]):
        off, rs, re = blacklist_in_windows(blacklist[0], blacklist[1], win_start, win_stop)
        if rs.size:
            keep = [_to_device(off, dev, np.int32), _to_device(rs, dev, np.int32), _to_device(re, dev, np.int32)]
            bl = tuple(x.data_ptr() for x in keep)
    g5 = None
    if gaps is not None:
        (c0, c1), telomeres = gaps[0], list(gaps[1])
        lim = 2 ** 31 - 1
        g5 = np.array([c0, c1, len(telomeres), max((a for a, _ in telomeres), default=0),
                       min((b for _, b in telomeres), default=0)], dtype=np.int64).clip(-lim, lim).astype(np.int32)
    _launch(dev, "ftk_delfi_windows_u64",
        fs, fe, mq, frags.n, frags.max_len, 0 if ref is None else ref.seq.data_ptr(),
        0 if ref is None else ref.nmask.data_ptr(), 0 if ref is None else ref.length,
        win.start.data_ptr(), win.stop.data_ptr(), n_win, *bl, None if g5 is None else _np_ptr(g5, c_int32),
        int(quality_threshold), _splits_for(n_win, frags.n), win.scratch.data_ptr(), counts.data_ptr())
    return counts


def agg_signal(rows, strand, trim_lo: int, out_len: int, device=None):
    """Strand-aware fp64 sum of equal-length signal rows (utils/_agg_bw.py:84-123) -> float64[out_len] (device).

    ``rows``: float32 [n_seg, row_len] (numpy or CUDA tensor); ``strand``: int8 per row (+1, -1, 0 = skip).
    ``device`` defaults to the device of a CUDA ``rows``, else the current device."""
    t = torch()
    dev = require_cuda(rows.device if device is None and t.is_tensor(rows) and rows.is_cuda else device)
    x = rows if t.is_tensor(rows) else _to_device(np.ascontiguousarray(rows, np.float32), dev, np.float32)
    x = x.to(dev, t.float32).contiguous()
    sd = _to_device(np.ascontiguousarray(strand, np.int8), dev, np.int8)
    n_seg, row_len = (int(x.shape[0]), int(x.shape[1])) if x.dim() == 2 else (0, 0)
    out = t.zeros(int(out_len), dtype=t.float64, device=dev)
    _launch(dev, "ftk_agg_signal_f64", x.data_ptr(), n_seg, row_len, int(trim_lo), int(out_len), sd.data_ptr(),
            out.data_ptr())
    return out


_ADJ_SLOTS = 148 * 3 * 128


def savgol_tables(window: int, degree: int):
    """Savitzky-Golay interior coefficients and mode='interp' edge-fit matrices (host, fp64); cached."""
    coef, first, last = _savgol_tables_cached(int(window), int(degree))
    return coef.copy(), first.copy(), last.copy()


@functools.lru_cache(maxsize=32)
def _savgol_tables_cached(window: int, degree: int):
    """The tables of ``savgol_tables``.

    The filter of scipy.signal.savgol_filter (reference call site frag/_adjust_wps.py:135-138;
    scipy/signal/_savitzky_golay.py): interior = the centre row of the hat matrix of a
    degree-``degree`` least-squares polynomial fit over ``window`` points; the first/last
    ``window//2`` outputs evaluate the fit of the first/last ``window`` samples at their own
    positions.

    The hat matrix is ``Q Q^T`` with ``Q`` an orthonormal basis of the polynomials of degree
    <= ``degree`` on the window positions, built by the Arnoldi (Stieltjes) process: column
    k+1 = position * column k, orthogonalised twice against every earlier column.  A
    Vandermonde matrix and its pseudo-inverse lose digits with the degree (wrong filters
    from degree ~10 on a 93-point window); this stays within a few ulp of the exact rational
    hat matrix at every degree.
    """
    if window % 2 != 1 or window < 1:
        raise ValueError("window_length must be odd.")
    if degree >= window:
        raise ValueError("polyorder must be less than window_length.")
    half = window // 2
    pos = np.arange(-half, half + 1, dtype=np.float64) / max(half, 1)
    Q = np.empty((window, degree + 1))
    Q[:, 0] = 1.0 / np.sqrt(window)
    for k in range(degree):
        v = pos * Q[:, k]
        for _ in range(2):
            v -= Q[:, : k + 1] @ (Q[:, : k + 1].T @ v)
        Q[:, k + 1] = v / np.linalg.norm(v)
    hat = Q @ Q.T                            # hat[i, j]: weight of sample j in the fit at i
    coef = np.ascontiguousarray(hat[half])   # symmetric: correlation == convolution
    edge_first = np.ascontiguousarray(hat[:half])
    edge_last = np.ascontiguousarray(hat[half + 1:])
    return coef, edge_first, edge_last


def savgol_rational(window: int, degree: int):
    """Interior Savitzky-Golay coefficients as exact rationals ``c_i = (a + b * i**2) / den`` (degree <= 3;
    the least-squares fit on symmetric points: degree 0/1 is the moving average, degree 2/3 gives
    ``a = S4, b = -S2, den = m * S4 - S2**2`` with ``Sk = sum i**k``), reduced by their gcd and checked
    against the fp64 table ``savgol_tables`` returns.  ``(0, 0, 0)`` when the coefficients have no such form."""
    import math
    m, h = int(window), int(window) // 2
    if degree <= 1:
        a, b, den = 1, 0, m
    elif degree <= 3:
        s2 = sum(i * i for i in range(-h, h + 1))
        s4 = sum(i ** 4 for i in range(-h, h + 1))
        a, b, den = s4, -s2, m * s4 - s2 * s2
    else:
        return 0, 0, 0
    if den <= 0:
        return 0, 0, 0
    g = math.gcd(math.gcd(abs(a), abs(b)), den)
    a, b, den = a // g, b // g, den // g
    coef = _savgol_tables_cached(m, int(degree))[0]
    exact = np.array([(a + b * i * i) / den for i in range(-h, h + 1)])
    if coef.shape != exact.shape or float(np.abs(coef - exact).max()) > 1e-12:
        return 0, 0, 0
    return a, b, den


import os as _os
_RANK_T_MAX = int(_os.environ.get("FTK_RANK_T_MAX", 4096))          # outputs per tile of the rank-bitmap kernel
_RANK_SMEM_MAX = 227 * 1024


def rank_tiles(seg_lengths, w: int, sg_w: int, t_max: int = _RANK_T_MAX, n_out=None):
    """Tile plan of ``ftk_adjust_rank_f64``: every segment's ``n - w`` outputs split evenly into
    pieces of at most ``t_max``.  Returns ``(tile_seg, tile_t0, tile_n, a_cap, s_cap)`` (int32 arrays;
    caps = most adjusted values / samples a tile stages, same arithmetic as the kernel)."""
    seg_lengths = np.asarray(seg_lengths, dtype=np.int64)
    n_out = (seg_lengths - int(w)) if n_out is None else np.asarray(n_out, dtype=np.int64)
    pieces = np.maximum(-(-n_out // int(t_max)), 0)
    piece = np.where(pieces > 0, -(-n_out // np.maximum(pieces, 1)), 0)
    tile_seg = np.repeat(np.arange(len(seg_lengths), dtype=np.int64), pieces)
    first = np.cumsum(pieces) - pieces
    k = np.arange(int(pieces.sum()), dtype=np.int64) - np.repeat(first, pieces)
    t0 = k * piece[tile_seg]
    n_t = np.minimum(piece[tile_seg], n_out[tile_seg] - t0)
    half = int(sg_w) >> 1
    no = n_out[tile_seg]
    a0 = np.maximum(t0 - half, 0)
    a1 = np.minimum(t0 + n_t + half, no)
    if sg_w:
        a1 = np.where(t0 < half, np.maximum(a1, np.minimum(int(sg_w), no)), a1)
        a0 = np.where(t0 + n_t > no - half, np.minimum(a0, np.maximum(no - int(sg_w), 0)), a0)
    A = a1 - a0
    a_cap = int(A.max()) if A.size else 1
    return (tile_seg.astype(np.int32), t0.astype(np.int32), n_t.astype(np.int32), a_cap, a_cap + int(w))


def _rank_smem(a_cap: int, s_cap: int, shifted: bool = True) -> int:
    """Shared memory of one ``adjust_rank_kernel`` CTA (rank_smem_bytes in csrc/ftk_adjust.cu)."""
    a_slots = a_cap + (a_cap >> 4) + 2
    nword = (s_cap + 31) // 32
    nwp = max((nword + 1) | 1, 69)
    b = (a_slots * (8 if shifted else 4) + 15) & ~15
    b += 32 * nwp * 8
    b = (b + 15) & ~15
    return b + (nword * 32 + 32) * 2


class AdjustPlan:
    """Everything ``adjust_segments`` needs that depends only on the segment layout and the filter
    parameters - segment / output offsets, the rank kernel's tile table, the Savitzky-Golay tables -
    built once, resident in HBM, reusable for any number of inputs with the same layout
    (``distributed.multi_wps_genome`` keeps one per contig)."""

    def __init__(self, seg_lengths, median_window_size=1000, savgol=True, savgol_window_size=21,
                 savgol_poly_deg=2, device=None, skip_short=False):
        t = torch()
        self.device = dev = require_cuda(device)
        self.w = w = int(median_window_size)
        self.seg_lengths = seg_lengths = np.asarray(seg_lengths, dtype=np.int64)
        if w % 2 or w < 2:
            raise ValueError("operands could not be broadcast together: median_window_size must be even "
                             "(frag/_adjust_wps.py:43 slices w//2 from both ends)")
        n_out = seg_lengths - w
        if skip_short:
            n_out = self.output_lengths(seg_lengths, w, savgol, savgol_window_size)
        else:
            if (seg_lengths < w).any():
                bad = int(seg_lengths[seg_lengths < w][0])
                raise ValueError(f"median_window_size ({w}) cannot be greater than the length of interval ({bad}).")
            if savgol and (n_out < savgol_window_size).any():
                raise ValueError("If mode is 'interp', window_length must be less than or equal to the size of x.")
        self.n_out = n_out
        self.n_seg = len(seg_lengths)
        self.seg_off = np.zeros(self.n_seg + 1, np.int64); np.cumsum(seg_lengths, out=self.seg_off[1:])
        self.out_off = np.zeros(self.n_seg + 1, np.int64); np.cumsum(n_out, out=self.out_off[1:])
        self.n_total = int(self.out_off[-1])
        self.d_seg = _to_device(self.seg_off, dev, np.int64)
        self.d_out = _to_device(self.out_off, dev, np.int64)
        self.sg_w = int(savgol_window_size) if savgol else 0
        self.tables = None
        self.sg_rational = (0, 0, 0)
        if savgol:
            self.sg_rational = savgol_rational(self.sg_w, int(savgol_poly_deg))
            coef, ef, el = savgol_tables(self.sg_w, int(savgol_poly_deg))
            self.tables = (_to_device(coef, dev, np.float64),
                           _to_device(ef.reshape(-1) if ef.size else np.zeros(1), dev, np.float64),
                           _to_device(el.reshape(-1) if el.size else np.zeros(1), dev, np.float64))
        # tile table of the rank kernel (None when the window / tile does not fit its shared memory)
        self.rank = None
        if self.n_total and w <= 32766 and self.sg_w <= 127:
            tile_seg, tile_t0, tile_n, a_cap, s_cap = rank_tiles(seg_lengths, w, self.sg_w, n_out=n_out)
            if s_cap <= 65535 - 64 and _rank_smem(a_cap, s_cap) <= _RANK_SMEM_MAX:
                self.rank = (tuple(_to_device(a, dev, np.int32) for a in (tile_seg, tile_t0, tile_n)),
                             len(tile_seg), a_cap, s_cap)

    @staticmethod
    def output_lengths(seg_lengths, median_window_size=1000, savgol=True, savgol_window_size=21):
        """Outputs per segment with ``skip_short``: ``n - median_window_size``, or 0 for a segment too short for the
        filters (the reference's driver skips it: frag/_adjust_wps.py:125-129 raises per interval, :145-153 skips
        it); such segments stay in the sample layout."""
        n_out = np.asarray(seg_lengths, dtype=np.int64) - int(median_window_size)
        return np.where((n_out >= (int(savgol_window_size) if savgol else 0)) & (n_out > 0), n_out, 0)

    def run_rank(self, xd, shift_ptr=0, out=None):
        """Launch the fused median + Savitzky-Golay kernel; returns ``(out, tile_flag)`` (no sync:
        the caller decides when to look at the flags)."""
        t = torch()
        (d_ts, d_t0, d_tn), n_tiles, a_cap, s_cap = self.rank
        if out is None:
            out = t.empty(max(self.n_total, 1), dtype=t.float64, device=self.device)
        flag = t.empty(n_tiles, dtype=t.uint8, device=self.device)
        tb = self.tables
        _launch(self.device, "ftk_adjust_rank_f64",
            xd.data_ptr(), 1 if xd.dtype == t.int32 else 0, self.d_seg.data_ptr(), self.d_out.data_ptr(), shift_ptr,
            self.n_seg, d_ts.data_ptr(), d_t0.data_ptr(), d_tn.data_ptr(), n_tiles, self.w, self.sg_w,
            tb[0].data_ptr() if tb else 0, tb[1].data_ptr() if tb else 0, tb[2].data_ptr() if tb else 0,
            *(self.sg_rational if not shift_ptr else (0, 0, 0)),
            a_cap, s_cap, out.data_ptr(), flag.data_ptr())
        return out, flag


def adjust_segments(x, seg_lengths, median_window_size=1000, use_mean=False, savgol=True,
                    savgol_window_size=21, savgol_poly_deg=2, subtract_edges=False, edge_size=500,
                    run_len=None, impl=None, plan: AdjustPlan | None = None, defer_check: bool = False):
    """Median/mean-adjust + Savitzky-Golay smooth contiguous raw-WPS segments on the GPU.

    ``x``: samples of all segments back to back - float32 (numpy or CUDA tensor; bigWig values) or an
    int32 CUDA tensor (device-resident WPS, no conversion pass); ``seg_lengths``: samples per segment.
    Returns ``(out float64 CUDA tensor, out_off)`` with segment s's ``n_s - w`` outputs at
    ``out[out_off[s]:out_off[s+1]]``.  Raises ValueError exactly where the reference does
    (frag/_adjust_wps.py:125-129 and numpy/scipy shape errors for odd windows / too-short segments).

    The median path runs the fused rank-bitmap kernel (``ftk_adjust_rank_f64``: median + Savitzky-Golay in
    one pass, 12 B of HBM traffic per position); tiles it flags (non-integer samples, huge values) and the
    mean path go through the sliding-histogram / generic kernels + the separate Savitzky-Golay kernel.
    ``impl="hist"`` forces that older path (``run_len`` only applies to it).  ``plan``: a prebuilt
    ``AdjustPlan`` for this layout and these parameters (skips all host-side planning and uploads), on the device
    of ``x`` when ``x`` is a CUDA tensor (ValueError otherwise).
    ``defer_check=True`` (median path with a rank plan only): no host synchronisation - returns
    ``(out, out_off, tile_flag)`` and the caller looks at ``tile_flag.any()`` later (and calls again
    with ``impl="hist"`` if it is set).
    """
    t = torch()
    on_device = t.is_tensor(x) and x.is_cuda
    dev = require_cuda(x.device if on_device else None if plan is None else plan.device)
    if plan is None:
        plan = AdjustPlan(seg_lengths, median_window_size, savgol, savgol_window_size, savgol_poly_deg, dev)
    _same_device(dev, plan)
    w, n_seg, n_out, n_total = plan.w, plan.n_seg, plan.n_out, plan.n_total
    out_off = plan.out_off
    if on_device and x.dtype == t.int32:
        xd = x.contiguous()
    else:
        xd = x if t.is_tensor(x) else _to_device(np.asarray(x), dev, np.float32)
        xd = xd.to(dev, t.float32).contiguous()
    out = t.empty(max(n_total, 1), dtype=t.float64, device=dev)
    if n_total == 0:
        return out[:0], out_off
    d_seg, d_out = plan.d_seg, plan.d_out
    shift_ptr = 0
    if subtract_edges:
        xf = xd if xd.dtype == t.float32 else xd.to(t.float32)
        shift = t.empty(n_seg, dtype=t.float64, device=dev)
        _launch(dev, "ftk_adjust_edge_shift_f64", xf.data_ptr(), d_seg.data_ptr(), n_seg, int(edge_size),
                shift.data_ptr())
        shift_ptr = shift.data_ptr()
    sg_w, tables = plan.sg_w, plan.tables

    # ---- fused rank-bitmap kernel (median path)
    if not use_mean and impl != "hist" and plan.rank is not None:
        _, flag = plan.run_rank(xd, shift_ptr, out)
        if defer_check:
            return out[:n_total], out_off, flag
        if not bool(flag.any().item()):
            return out[:n_total], out_off
        # some tile could not be handled: redo the call on the general path (rare: non-integer input)

    # ---- sliding-histogram / generic kernels + separate Savitzky-Golay
    if xd.dtype != t.float32:
        xd = xd.to(t.float32)
    if run_len is None:
        # one thread slides one run: aim for a single full wave of the 148 SMs x 3 CTAs x 128 threads,
        # keep the w-sample window fill amortised (>= 1024 outputs) and split short segments evenly
        slots = _ADJ_SLOTS
        run_len = int(min(max(-(-int(n_out.sum()) // slots), 1024), 16384))
        nmax = int(n_out.max()) if n_seg else 0
        if 0 < nmax <= 4 * run_len:
            run_len = -(-nmax // max(1, round(nmax / run_len)))
    run_len = max(int(run_len), 1)
    runs = -(-n_out // run_len)
    run_off = np.zeros(n_seg + 1, np.int64); np.cumsum(runs, out=run_off[1:])
    n_runs = int(run_off[-1])
    if n_runs == 0:
        return out[:0], out_off
    d_run = _to_device(run_off, dev, np.int64)
    adj = t.empty(max(n_total, 1), dtype=t.float64, device=dev) if savgol else out
    fb = t.empty(n_runs, dtype=t.uint8, device=dev)
    _launch(dev, "ftk_adjust_wps_f64", xd.data_ptr(), d_seg.data_ptr(), d_out.data_ptr(), d_run.data_ptr(), shift_ptr,
            n_seg, n_runs, int(w), int(bool(use_mean)), int(run_len), adj.data_ptr(), fb.data_ptr())
    flagged = t.nonzero(fb).flatten().to(t.int64)   # plumbing: compact the flagged run ids
    if flagged.numel():
        scratch = t.empty(flagged.numel() * w, dtype=t.float32, device=dev)
        _launch(dev, "ftk_adjust_wps_generic_f64", xd.data_ptr(), d_seg.data_ptr(), d_out.data_ptr(),
                d_run.data_ptr(), shift_ptr, n_seg, flagged.data_ptr(), flagged.numel(), int(w), int(bool(use_mean)),
                int(run_len), adj.data_ptr(), scratch.data_ptr())
    if savgol:
        _launch(dev, "ftk_savgol_f64", adj.data_ptr(), d_out.data_ptr(), n_seg, n_total, sg_w, tables[0].data_ptr(),
                tables[1].data_ptr(), tables[2].data_ptr(), out.data_ptr())
    if defer_check:
        return out[:n_total], out_off, None
    return out[:n_total], out_off


def cleavage_intervals(frags: ContigFragments, ivl_start, ivl_stop, chrom_size, min_length=None,
                       max_length=None, quality_threshold=30):
    """Cleavage proportion (float64, percent) of every interval back to back + host offsets.

    ``ivl_start/ivl_stop`` are the already padded/clamped bounds (frag/_cleavage_profile.py:188-189).
    """
    t = torch()
    plan = WpsPlan(ivl_start, ivl_stop, int(chrom_size), 0, frags.device)   # max_len 0: mid_lo/hi = [start, stop)
    out = t.empty(max(plan.n_positions, 1), dtype=t.float64, device=frags.device)
    if plan.n_tiles:
        fs, fe, mq = frags.ptrs()
        sd = 0 if frags.strand is None else frags.strand.data_ptr()
        _launch(frags.device, "ftk_cleavage_tiles_f64",
            fs, fe, mq, sd, frags.n, frags.max_len, plan.tile_p0.data_ptr(), plan.tile_len.data_ptr(),
            plan.tile_mid_lo.data_ptr(), plan.tile_mid_hi.data_ptr(), plan.tile_out_off.data_ptr(), plan.n_tiles,
            none_to_ftk(min_length), none_to_ftk(max_length), int(quality_threshold),
            plan.scratch.data_ptr(), out.data_ptr())
    return out[: plan.n_positions], plan.offsets


def depth_intervals(frags: ContigFragments, ivl_start, ivl_stop, chrom_size, min_length=None, max_length=None,
                    quality_threshold=30, midpoint=False):
    """Per-base fragment depth (int32) of every interval back to back + host offsets.

    Span depth (the coverage of _coverage_and_ends, frag/_cleavage_profile.py:33-90) counts the passing
    fragments with start <= p < stop; ``midpoint=True`` counts those with (start + stop) // 2 == p.
    ``ivl_start/ivl_stop`` are already padded/clamped bounds; one launch for all of them.
    """
    t = torch()
    plan = WpsPlan(ivl_start, ivl_stop, int(chrom_size), 0, frags.device)   # the tile table of cleavage_intervals
    out = t.empty(max(plan.n_positions, 1), dtype=t.int32, device=frags.device)
    if plan.n_tiles:
        fs, fe, mq = frags.ptrs()
        _launch(frags.device, "ftk_depth_tiles_i32",
            fs, fe, mq, frags.n, frags.max_len, plan.tile_p0.data_ptr(), plan.tile_len.data_ptr(),
            plan.tile_mid_lo.data_ptr(), plan.tile_mid_hi.data_ptr(), plan.tile_out_off.data_ptr(), plan.n_tiles,
            none_to_ftk(min_length), none_to_ftk(max_length), int(quality_threshold), int(bool(midpoint)),
            plan.scratch.data_ptr(), out.data_ptr())
    return out[: plan.n_positions], plan.offsets


GC_DEPTH_MAX_WEIGHT = 2 ** 62   # FTK_GC_DEPTH_MAX_WEIGHT: quantised weights stay below it


def gc_quantise_weights(weights, shape) -> np.ndarray:
    """The weight table in units of 2^-32: ``rint(W * 2^32)`` as int64 (fp64 on the host; the scaling is exact and
    ``rint`` rounds half to even).  ValueError unless ``weights`` has ``shape`` and every entry is finite and ``>= 0``,
    or when a quantised weight reaches 2^62."""
    t = torch()
    w = weights.detach().cpu().numpy() if t.is_tensor(weights) else np.asarray(weights)
    if tuple(w.shape) != tuple(shape):
        raise ValueError(f"the weight table must have shape {tuple(shape)}, got {tuple(w.shape)}")
    w = w.astype(np.float64)
    if not bool((np.isfinite(w) & (w >= 0)).all()):
        raise ValueError("the weight table must hold finite, non-negative values")
    q = np.rint(w * 2.0 ** 32)
    if q.size and float(q.max()) >= GC_DEPTH_MAX_WEIGHT:
        raise ValueError(f"a GC weight of {float(w.max())!r} is too large for the depth tracks (below 2^30 needed)")
    return q.astype(np.int64)


def gc_depth_intervals(frags: ContigFragments, ref: PackedContig, ivl_start, ivl_stop, chrom_size, weights,
                       min_length, max_length, quality_threshold=30, midpoint=False):
    """GC-weighted per-base fragment depth (float64) of every interval back to back + host offsets
    (``ftk_gc_depth_tiles_f64``).

    A fragment ``[s, e)`` with ``mapq >= quality_threshold`` and ``min_length <= L <= max_length`` weighs
    ``Q[L - min_length, g] * 2^-32`` with ``Q = gc_quantise_weights(weights)`` when ``0 <= s``, ``e <= ref.length`` and
    no base of it is N (g = its C/G bases), else 0.  Span depth sums the weights of the fragments with
    ``s <= p < e``, ``midpoint=True`` those with ``(s + e) // 2 == p``.  The sums are int64, so the result is exact
    (``fp64(S) * 2^-32``), 0.0 where no weighted fragment counts and bit-identical between runs and batchings.
    ``ivl_start/ivl_stop`` are already padded/clamped bounds; one launch for all of them.  OverflowError when a tile's
    sums could pass 2^63 (a pile-up of huge weights); nothing is returned then."""
    t = torch()
    shape = gc_check(min_length, max_length)
    dev = frags.device
    _same_device(dev, ref)
    q = gc_quantise_weights(weights, shape)
    plan = WpsPlan(ivl_start, ivl_stop, int(chrom_size), 0, dev)   # the tile table of depth_intervals
    out = t.empty(max(plan.n_positions, 1), dtype=t.float64, device=dev)
    if plan.n_tiles:
        qd = _to_device(q, dev, np.int64)
        flag = t.zeros(1, dtype=t.int32, device=dev)
        fs, fe, mq = frags.ptrs()
        _launch(dev, "ftk_gc_depth_tiles_f64",
            fs, fe, mq, frags.n, frags.max_len, ref.seq.data_ptr(), ref.nmask.data_ptr(), ref.length,
            plan.tile_p0.data_ptr(), plan.tile_len.data_ptr(), plan.tile_mid_lo.data_ptr(), plan.tile_mid_hi.data_ptr(),
            plan.tile_out_off.data_ptr(), plan.n_tiles, int(min_length), int(max_length), int(quality_threshold),
            int(bool(midpoint)), qd.data_ptr(), int(q.max()), plan.scratch.data_ptr(), flag.data_ptr(), out.data_ptr())
        if int(flag.item()):
            raise OverflowError(f"GC-weighted depth of contig {frags.contig!r}: a pile-up of large GC weights could "
                                "overflow the int64 sums of a tile")
    return out[: plan.n_positions], plan.offsets
