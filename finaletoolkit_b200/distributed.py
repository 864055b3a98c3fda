"""Genome-wide features across the GPUs of one box: one process per GPU, contigs sharded by LPT.

Launch with ``python -m torch.distributed.run --nproc-per-node N ...`` (NCCL).  Per-position /
per-interval outputs (WPS, adjust_wps, interval coverage, interval statistics) stay on the rank
that owns the contig - no collective.  Genome-wide reductions use exactly one packed
``all_reduce(SUM)`` (+ one ``MIN`` for first-seen order), see ``sharding.py``.

Reference semantics reproduced: ``coverage(normalize=True)`` total = ``single_coverage`` over the
whole file (frag/_coverage.py:215-227, 254); ``frag_length_bins`` genome-wide dict in stream order
(frag/_frag_length.py:408-421); ``end_motifs`` 4^k counts summed over contigs' 1 Mb windows
(frag/_motif_common.py:599-609); DELFI bins are independent per contig (frag/_delfi.py:283-294).
"""
from __future__ import annotations

import numpy as np

from .sharding import DistContext, genome_length_dict, lpt_pack, reduce_length_dict

__all__ = ["owned_contigs", "genome_total_coverage", "genome_length_distribution", "genome_end_motif_counts",
           "genome_delfi_windows", "genome_bin_counts", "table_shard", "ContigWps", "GenomeShard", "multi_wps_genome", "adjust_wps_genome", "tile_genome",
           "wps_spectrum_genome", "gather_to_writer"]


def owned_contigs(table, ctx: DistContext | None = None):
    """Contigs of ``table`` this rank owns (LPT by ``shard_weight``: fragment count, or compressed byte
    span for a lazy tabix-backed table; deterministic and cheap on every rank)."""
    ctx = ctx or DistContext()
    weight = getattr(table, "shard_weight", None) or table.n_fragments
    weights = {c: weight(c) for c in table.contigs}
    return lpt_pack(weights, ctx.world)[ctx.rank]


def genome_total_coverage(table, min_length=None, max_length=None, intersect_policy="midpoint",
                          quality_threshold=30, ctx: DistContext | None = None, device=None) -> int:
    """Whole-file fragment count (the ``normalize=True`` denominator) with one all-reduce."""
    from .device import interval_hist, require_cuda, torch
    ctx = ctx or DistContext()
    dev = require_cuda(device)
    t = torch()
    total = t.zeros(1, dtype=t.int64, device=dev)
    for c in owned_contigs(table, ctx):
        if table.n_fragments(c):
            cnt, _, _ = interval_hist(table.device(c, dev), [0], [None], intersect_policy, min_length, max_length,
                                      quality_threshold)
            total += cnt[:1]
    ctx.all_reduce_sum(total)
    return int(total.item())


def genome_length_distribution(table, min_length=0, max_length=None, intersect_policy="midpoint",
                               quality_threshold=30, ctx: DistContext | None = None, device=None,
                               region=(None, None)) -> dict:
    """The reference's genome-wide ``length -> count`` dict (first-seen order) on every rank."""
    from .device import interval_hist, require_cuda, torch
    ctx = ctx or DistContext()
    dev = require_cuda(device)
    t = torch()
    order = {c: i for i, c in enumerate(table.contigs)}
    mine = owned_contigs(table, ctx)
    # a common histogram width: the longest fragment over ALL contigs = MAX over the ranks' own contigs
    gmax_t = t.tensor([max([table.device(c, dev).max_len for c in mine if table.n_fragments(c)] + [0])],
                      dtype=t.int64, device=dev)
    ctx.all_reduce_max(gmax_t)
    gmax = int(gmax_t.item())
    n_bins = (gmax if max_length is None else min(gmax, int(max_length))) + 1
    if region == (None, None):
        # every contig whole: one launch per shard group over the rank's contigs laid end to end
        shard = table_shard(table, ctx, dev, mine)
        _, hist, keys = shard.interval_counts(None, order, intersect_policy, min_length, max_length, quality_threshold,
                                              n_bins=n_bins, first_seen=True)
        return reduce_length_dict(ctx, hist, keys)
    parts = []
    for c in mine:
        if not table.n_fragments(c):
            continue
        _, h, f = interval_hist(table.device(c, dev), [region[0]], [region[1]], intersect_policy, min_length,
                                max_length, quality_threshold, n_bins=n_bins, pooled=True, first_seen=True)
        parts.append((order[c], h[0], f[0]))
    if not parts:  # rank without fragments still takes part in the collectives
        parts = [(0, t.zeros(n_bins, dtype=t.int64, device=dev), t.full((n_bins,), 2 ** 31 - 1, dtype=t.int32, device=dev))]
    return genome_length_dict(ctx, parts, n_bins)


def genome_end_motif_counts(table, ref, k=4, strand_mode=0, quality_threshold=30,
                            ctx: DistContext | None = None, device=None, breakpoint=False) -> np.ndarray:
    """int64[4**k] genome-wide end-motif (or, with ``breakpoint``, breakpoint-motif) counts over every
    contig's 1 Mb windows, one all-reduce."""
    from .device import require_cuda, torch
    from .frag._motif_common import genome_windows, pooled_window_counts
    ctx = ctx or DistContext()
    dev = require_cuda(device)
    t = torch()
    total = t.zeros((1, 4 ** k), dtype=t.int64, device=dev)
    mine = set(owned_contigs(table, ctx))
    for chrom, chrom_length in ref.chroms.items():
        if chrom not in mine or not table.n_fragments(chrom):
            continue
        pooled_window_counts(table, ref, chrom, genome_windows(chrom_length), k, strand_mode, quality_threshold,
                             breakpoint=breakpoint, total=total, device=dev)
    ctx.all_reduce_sum(total)
    return total[0].cpu().numpy()


def genome_delfi_windows(table, ref, bins_by_contig, blacklist_by_contig=None, gaps_by_contig=None,
                         quality_threshold=30, ctx: DistContext | None = None, device=None) -> dict:
    """DELFI bin counts of a whole genome: contigs are LPT-sharded over the ranks (bins of different
    contigs are independent, frag/_delfi.py:283-294 hands them to a process pool), each rank runs
    ``ftk_delfi_windows_u64`` on the contigs it owns and ONE all-reduce merges the packed table.

    ``bins_by_contig``: {contig: (starts, stops)}; ``blacklist_by_contig``: {contig: (starts, stops)}
    sorted by (start, stop); ``gaps_by_contig``: {contig: (centromere, telomeres)}.
    Returns {contig: int64[n_bins, 4]} = short, long, num_frags, G+C bases, identical on every rank."""
    from .device import require_cuda, torch
    from .frag._delfi import delfi_rows
    ctx = ctx or DistContext()
    dev = require_cuda(device)
    t = torch()
    names = [c for c in bins_by_contig if len(bins_by_contig[c][0])]
    sizes = [len(bins_by_contig[c][0]) for c in names]
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    packed = t.zeros((int(offs[-1]), 4), dtype=t.int64, device=dev)
    mine = set(owned_contigs(table, ctx))
    for i, chrom in enumerate(names):
        # a contig the fragment table does not know is owned by nobody: rank 0 counts its G+C bases
        owner_here = chrom in mine or (chrom not in table.contigs and ctx.rank == 0)
        if not owner_here:
            continue
        ws, we = bins_by_contig[chrom]
        got = delfi_rows(table, ref, chrom, np.asarray(ws, np.int64).tolist(), np.asarray(we, np.int64).tolist(),
                         (blacklist_by_contig or {}).get(chrom), (gaps_by_contig or {}).get(chrom), quality_threshold, dev)
        packed[int(offs[i]): int(offs[i + 1])] = t.from_numpy(got).to(dev)
    ctx.all_reduce_sum(packed)
    host = packed.cpu().numpy()
    return {c: host[int(offs[i]): int(offs[i + 1])] for i, c in enumerate(names)}


# ----------------------------------------------------------------------------------------------
# Genome-wide WPS (+ coverage + length histogram) and the device-resident WPS -> adjust_wps chain
# ----------------------------------------------------------------------------------------------
class ContigWps:
    """Per-contig result of ``multi_wps_genome`` on the rank that owns the contig (device tensors)."""

    __slots__ = ("contig", "starts", "stops", "offsets", "wps", "cov", "adjusted", "adj_offsets", "adj_segments", "flags")

    def __init__(self, contig, starts, stops, offsets, wps, cov=None):
        self.contig, self.starts, self.stops, self.offsets = contig, starts, stops, offsets
        self.wps, self.cov = wps, cov
        self.adjusted = self.adj_offsets = self.adj_segments = self.flags = None


def tile_genome(chrom_sizes, interval_size: int = 5000) -> dict:
    """{contig: (starts, stops)}: every contig tiled by ``interval_size`` windows (the genome-wide
    site set of SURVEY.md §8d config 3)."""
    out = {}
    for contig, size in chrom_sizes:
        edges = np.arange(0, int(size) + int(interval_size), int(interval_size), dtype=np.int64).clip(max=int(size))
        out[contig] = (edges[:-1].copy(), edges[1:].copy())
    return out


_SHARD_SPAN = (1 << 31) - (1 << 22)     # the virtual coordinates of a group stay well inside int32
empty_i64 = np.zeros(0, np.int64)


class _ShardGroup:
    __slots__ = ("frags", "plan", "wps", "cov", "seg_lengths", "aplans", "adjusted", "n_ivl", "ivl_base")


class GenomeShard:
    """The contigs ONE rank owns, laid end to end in one virtual coordinate space, so that a genome
    pass is one range prepass + ONE persistent-kernel launch per rank instead of one pair per contig.

    Contig ``c`` is shifted by ``base[c]``: its fragments (``start + base``, ``stop + base``), its tiles
    (``p0``, the midpoint window ``[mid_lo, mid_hi)`` clamped to the contig as frag/_wps.py:156-157 asks)
    and nothing else - the kernels are the per-contig ones, unchanged, they simply see one longer
    start-sorted column and one longer tile table.  Neighbouring contigs are separated by a guard band
    wider than anything a fragment can reach (window + the longest fragment + max_length, twice), so no
    fragment of one contig lies in the staged range of, or leaves an event in, a tile of another.  A
    group ends before the virtual coordinate would leave int32 (the 3.1 Gb genome on one rank: two
    groups).  Outputs live in buffers the shard owns and reuses from pass to pass: one int32 WPS buffer
    (every contig's part starts on a 16-byte boundary so the 128-bit stores stay aligned), one int64
    coverage vector indexed by (contig, interval), one float64 buffer for the adjusted series.
    """

    def __init__(self, table, sizes: dict, sites: dict, contigs, max_length: int, window_size: int = 120,
                 device=None):
        from .device import ContigFragments, WpsPlan, require_cuda, torch
        t = torch()
        self.device = dev = require_cuda(device)
        self.max_length, self.window_size = int(max_length), int(window_size)
        self.contigs = list(contigs)
        self.groups: list = []
        self.layout: dict = {}
        self._packed = None
        pend = None                      # the group being filled

        def close():
            nonlocal pend
            if pend is None:
                return
            g = _ShardGroup()
            tiles = {k: (np.concatenate(v) if v else np.zeros(0, np.int64 if k in ("out_off", "offsets") else np.int32))
                     for k, v in pend["tiles"].items()}
            tiles["offsets"] = np.concatenate([tiles["offsets"], [pend["pos"]]]).astype(np.int64)
            g.plan = WpsPlan.from_tiles(tiles, self.max_length, dev, n_positions=pend["pos"])
            cols = pend["cols"]
            if cols:
                start = t.cat([c_[0] for c_ in cols]); stop = t.cat([c_[1] for c_ in cols])
                mapq = None if all(c_[2] is None for c_ in cols) else t.cat(
                    [c_[2] if c_[2] is not None else t.full((c_[0].numel(),), 255, dtype=t.uint8, device=dev) for c_ in cols])
            else:
                start = t.zeros(0, dtype=t.int32, device=dev); stop = start.clone(); mapq = None
            g.frags = ContigFragments(start, stop, mapq, None, device=dev, max_len=pend["flen"])
            g.wps = None
            g.cov = None
            g.seg_lengths = np.concatenate(pend["segs"]) if pend["segs"] else np.zeros(0, np.int64)
            g.aplans, g.adjusted = {}, None
            g.n_ivl, g.ivl_base = pend["ivl"], pend["ivl_base"]
            self.groups.append(g)
            pend = None

        ivl_total = 0
        empty = np.zeros(0, np.int64)
        for c in self.contigs:
            starts, stops = (np.ascontiguousarray(a, dtype=np.int64) for a in (sites[c] if sites is not None else (empty, empty)))
            clen = int(sizes[c])
            frags = table.device(c, dev) if table.n_fragments(c) else None
            n = frags.n if frags is not None else 0
            flen = frags.max_len if n else 0
            lo = min([0] + ([int(starts.min())] if len(starts) else []) + ([int(frags.start[0].item())] if n else []))
            hi = max([clen] + ([int(stops.max())] if len(stops) else []) + ([int(frags.stop.max().item())] if n else []))
            guard = 2 * (flen + self.max_length + self.window_size) + 4096
            if hi - lo + 2 * guard > _SHARD_SPAN:
                raise ValueError(f"contig {c} does not fit the int32 coordinate space of a shard group")
            if pend is not None and pend["end"] + guard - lo + hi + guard > _SHARD_SPAN:
                close()
            if pend is None:
                pend = {"end": 0, "pos": 0, "ivl": 0, "ivl_base": ivl_total, "flen": 0, "nfrag": 0, "cols": [], "segs": [],
                        "tiles": {k: [] for k in ("p0", "len", "mid_lo", "mid_hi", "out_off", "ivl", "offsets")}}
            base = (pend["end"] + guard - lo + 63) & ~63
            tl = WpsPlan.host_tiles(starts, stops, clen, self.max_length)
            obase, ibase = pend["pos"], pend["ivl"]
            first = tl["ivl"] < 0
            idx = (tl["ivl"].astype(np.int64) & 0x7fffffff) + ibase
            pend["tiles"]["p0"].append((tl["p0"].astype(np.int64) + base).astype(np.int32))
            pend["tiles"]["len"].append(tl["len"])
            pend["tiles"]["mid_lo"].append((tl["mid_lo"].astype(np.int64) + base).astype(np.int32))
            pend["tiles"]["mid_hi"].append((tl["mid_hi"].astype(np.int64) + base).astype(np.int32))
            pend["tiles"]["out_off"].append(tl["out_off"] + obase)
            pend["tiles"]["ivl"].append(np.where(first, idx - (1 << 31), idx).astype(np.int32))
            pend["tiles"]["offsets"].append(tl["offsets"][:-1] + obase)
            npos = int(tl["offsets"][-1])
            pad = (-npos) & 3
            seg_lo = sum(len(a) for a in pend["segs"])
            pend["segs"].append(np.diff(tl["offsets"]))
            pend["segs"].append(np.array([pad], dtype=np.int64))     # alignment gap: a segment without output
            self.layout[c] = {"group": len(self.groups), "base": int(base), "wps": (obase, obase + npos),
                              "ivl": (ivl_total, ivl_total + len(starts)), "starts": starts, "stops": stops,
                              "offsets": tl["offsets"], "seg": (seg_lo, seg_lo + len(starts)),
                              "span": (int(lo), int(hi)), "frag": (pend["nfrag"], pend["nfrag"] + n)}
            if n:
                pend["cols"].append((frags.start + int(base), frags.stop + int(base), frags.mapq))
                pend["nfrag"] += n
            pend["flen"] = max(pend["flen"], flen)
            pend["end"] = base + hi
            pend["pos"] += npos + pad
            pend["ivl"] += len(starts)
            ivl_total += len(starts)
        close()
        self.n_intervals = ivl_total
        self._bin_sets: dict = {}
        self.cov = t.zeros(max(ivl_total, 1), dtype=t.int64, device=dev)
        for g in self.groups:
            g.wps = t.empty(max(g.plan.n_positions, 1), dtype=t.int32, device=dev)
            g.cov = self.cov[g.ivl_base: g.ivl_base + g.n_ivl] if g.n_ivl else self.cov[:1]

    def interval_counts(self, bins: dict | None, order: dict, intersect_policy="midpoint", min_length=None,
                        max_length=None, quality_threshold=30, n_bins: int = 0, first_seen: bool = False,
                        cache_key=None):
        """Fragment counts of ``bins`` {contig: (starts, stops)} (``None``: one whole-contig interval per
        contig, the reference's region ``(None, None)``) + the pooled length histogram of the counted
        fragments (+ first-seen keys), ONE ``ftk_interval_hist_u64`` launch per shard group instead of one
        per contig.  ``order``: {contig: position in the file header} - the first-seen key of a length is
        ``(order << 32) | row index within the contig``, comparable across ranks (``sharding.first_seen_keys``).
        Returns ``({contig: int64 counts view}, hist int64[n_bins] | None, keys int64[n_bins] | None)``."""
        from .device import IntervalSet, interval_hist, torch
        from .sharding import FIRST_SEEN_NONE
        t = torch()
        dev = self.device
        key = cache_key if cache_key is not None else ("whole" if bins is None else id(bins))
        hit = self._bin_sets.get(key)
        # an id()-keyed entry keeps its dict alive, so the id cannot be handed to another object while cached
        sets = hit[1] if (hit is not None and (cache_key is not None or bins is None or hit[0] is bins)) else None
        if sets is None:
            sets = []
            for gi, g in enumerate(self.groups):
                ss, ee, where, f_off, f_ord = [], [], {}, [0], []
                n_b = 0
                for c in self.contigs:
                    lay = self.layout[c]
                    if lay["group"] != gi:
                        continue
                    if bins is None:
                        # one below the lowest coordinate: tabix's `stop > start` test must keep zero-length rows
                        a, b = np.array([lay["span"][0] - 1], np.int64), np.array([lay["span"][1] + 1], np.int64)
                    else:
                        # clipped to the contig's own extent (no fragment lies outside it, so membership is
                        # unchanged): a bin must not reach into the neighbouring contig's coordinates
                        a, b = (np.clip(np.asarray(x, dtype=np.int64), lay["span"][0] - 1, lay["span"][1] + 1)
                                for x in bins.get(c, (empty_i64, empty_i64)))
                    ss.append(a + lay["base"]); ee.append(b + lay["base"])
                    where[c] = (n_b, n_b + len(a)); n_b += len(a)
                    f_off.append(lay["frag"][1]); f_ord.append(int(order[c]))
                ivl = IntervalSet(np.concatenate(ss) if ss else empty_i64, np.concatenate(ee) if ee else empty_i64, dev)
                sets.append((ivl, where, t.tensor(f_off, dtype=t.int64, device=dev),
                             t.tensor(f_ord or [0], dtype=t.int64, device=dev),
                             t.zeros(max(ivl.n, 1), dtype=t.int64, device=dev)))
            self._bin_sets[key] = (bins, sets)
        hist = t.zeros((1, n_bins), dtype=t.int64, device=dev) if n_bins else None
        keys = t.full((n_bins,), FIRST_SEEN_NONE, dtype=t.int64, device=dev) if (n_bins and first_seen) else None
        counts = {}
        for g, (ivl, where, f_off, f_ord, cnt) in zip(self.groups, sets):
            cnt.zero_()
            first = t.full((1, n_bins), 2 ** 31 - 1, dtype=t.int32, device=dev) if keys is not None else None
            if ivl.n and g.frags.n:
                interval_hist(g.frags, intersect_policy=intersect_policy, min_length=min_length, max_length=max_length,
                              quality_threshold=quality_threshold, n_bins=n_bins, pooled="hist" if n_bins else False,
                              ivl_set=ivl, out=(cnt, hist, first))
            if keys is not None:
                f = first[0].to(t.int64)
                ci = t.bucketize(f, f_off[1:], right=True).clamp_(max=max(f_ord.numel() - 1, 0))
                k = (f_ord[ci] << 32) + (f - f_off[ci])
                keys = t.minimum(keys, t.where(first[0] == 2 ** 31 - 1, t.full_like(k, FIRST_SEEN_NONE), k))
            for c, (a, b) in where.items():
                counts[c] = cnt[a:b]
        return counts, (hist[0] if hist is not None else None), keys

    def packed(self, n_bins: int):
        """[coverage total, length histogram...]: the one buffer that is all-reduced."""
        from .device import torch
        t = torch()
        if self._packed is None or self._packed.numel() != 1 + int(n_bins):
            self._packed = t.zeros(1 + int(n_bins), dtype=t.int64, device=self.device)
        return self._packed

    def adjust_plan(self, g: _ShardGroup, adjust: dict):
        from .device import AdjustPlan
        key = (int(adjust.get("median_window_size", 1000)), bool(adjust.get("savgol", True)),
               int(adjust.get("savgol_window_size", 21)), int(adjust.get("savgol_poly_deg", 2)))
        if key not in g.aplans:
            g.aplans[key] = AdjustPlan(g.seg_lengths, key[0], key[1], key[2], key[3], self.device, skip_short=True)
        return g.aplans[key]

    def results(self, fused: bool, adjust: dict | None, keep_adjusted: bool = True) -> dict:
        """{contig: ContigWps} - views into the shard's buffers (valid until the shard's next pass)."""
        out = {}
        for c in self.contigs:
            lay = self.layout[c]
            g = self.groups[lay["group"]]
            res = ContigWps(c, lay["starts"], lay["stops"], lay["offsets"], g.wps[lay["wps"][0]: lay["wps"][1]],
                            self.cov[lay["ivl"][0]: lay["ivl"][1]] if fused else None)
            if adjust is not None:
                ap = self.adjust_plan(g, adjust)
                s0, s1 = lay["seg"]
                res.adj_offsets = ap.out_off[s0: s1 + 1] - ap.out_off[s0]
                res.adj_segments = np.flatnonzero(ap.n_out[s0: s1] > 0)
                if keep_adjusted and g.adjusted is not None:
                    res.adjusted = g.adjusted[int(ap.out_off[s0]): int(ap.out_off[s1])]
            out[c] = res
        return out


def multi_wps_genome(table, chrom_sizes, sites: dict | None = None, interval_size=5000, window_size=120,
                     min_length=120, max_length=180, quality_threshold=30, coverage=False, length_hist=False,
                     adjust: dict | None = None, ctx: DistContext | None = None, device=None,
                     contigs: list | None = None, reduce: bool = True, plans: dict | None = None,
                     keep_adjusted: bool = True, n_bins: int | None = None, sync: bool = True):
    """Genome-wide L-WPS over the ranks of one box (reference drivers frag/_multi_wps.py:152-198 +,
    with ``adjust``, frag/_adjust_wps.py:229-291) - contigs LPT-sharded, every rank sweeps the contigs
    it owns, results stay on the owning rank's GPU, no data-path collective.

    The rank's contigs are laid end to end in one virtual coordinate space (``GenomeShard``): a pass is
    ONE range prepass + ONE launch of the persistent WPS kernel per rank (two of each when a single rank
    holds more than 2^31 bp), into buffers the shard owns.

    ``sites``: {contig: (starts, stops)} sorted by start (``tile_genome`` when None).  With
    ``coverage`` / ``length_hist`` the sweep is the fused pass (WPS + per-interval midpoint coverage +
    pooled length histogram, one read of the fragments); the histogram and the coverage total are the
    only things combined across ranks (ONE packed all_reduce).  ``adjust`` = kwargs of
    ``device.adjust_segments`` (median_window_size, savgol, ...): each interval of at least
    ``median_window_size`` positions is adjusted straight from the int32 WPS in HBM - no bigWig
    round trip, no float32 copy.

    BAM input: the genome pass selects FRAGMENTS per interval, not reads (a device-resident sweep has no
    per-interval index query, DESIGN §7.1); a table that carries read-1 spans gets a ``UserWarning`` - use
    ``multi_wps`` where the reference's read-level selection matters.

    ``n_bins``: histogram width when the caller knows it (longest fragment of the job + 1) - saves the
    MAX all-reduce and its host synchronisation; ``plans``: a dict the shard is cached in (built on the
    first call, reused afterwards: same table, sites, contigs and max_length) - the returned tensors
    are then VIEWS into the shard's buffers, valid until the next call with the same ``plans``;
    ``contigs``: override the LPT assignment; ``reduce=False`` skips the collectives (single-rank
    checks inside a multi-rank job); ``keep_adjusted=False`` returns no adjusted series (timing runs);
    ``sync=False``: the coverage total comes back as a one-element device tensor instead of an ``int`` and the
    rank kernel's tile flags are not looked at (``results[c].flags`` holds them) - nothing in the call waits
    for the GPU, so back-to-back passes overlap their host work with the previous pass' kernels.

    Returns ``(results {contig: ContigWps} of this rank, hist int64[n_bins] | None, total | None)``.
    """
    from .device import adjust_segments, require_cuda, torch
    ctx = ctx or DistContext()
    dev = require_cuda(device)
    t = torch()
    sizes = dict(chrom_sizes)
    if sites is None:
        sites = tile_genome(chrom_sizes, interval_size)
    mine = contigs if contigs is not None else [c for c in owned_contigs(table, ctx) if c in sites]
    fused = bool(coverage or length_hist)
    key = ("shard", tuple(mine), int(max_length), int(window_size))
    shard = plans.get(key) if plans is not None else None
    if shard is None:
        if getattr(table, "has_read1", None) is not None and any(table.has_read1(c) for c in mine):
            import warnings
            warnings.warn("multi_wps_genome selects fragments, not reads, per interval: on BAM input its values can "
                          "differ from multi_wps at interval edges (DESIGN 7.1)", UserWarning, stacklevel=2)
        shard = GenomeShard(table, sizes, sites, mine, int(max_length), int(window_size), dev)
        if plans is not None:
            plans[key] = shard
    if not length_hist:
        n_bins = 0
    elif n_bins is None:   # one histogram width for the whole job: MAX over the ranks' own contigs
        m = t.tensor([max([g.frags.max_len for g in shard.groups if g.frags.n] + [0])], dtype=t.int64, device=dev)
        if reduce:
            ctx.all_reduce_max(m)
        n_bins = int(m.item()) + 1
    n_bins = int(n_bins)
    packed = shard.packed(n_bins)            # [coverage total, histogram...]
    cleared = False
    flags = []
    general = adjust is not None and (adjust.get("use_mean") or adjust.get("subtract_edges"))
    for g in shard.groups:
        if fused:
            # the range prepass clears the group's coverage counts and (first group) the packed buffer
            g.plan.ranges_fused(g.frags, window_size, None, zero_counts=g.cov, zero_hist=None if cleared else packed)
            cleared = True
            g.plan.run_fused(g.frags, window_size, min_length, max_length, quality_threshold, None, None,
                             quality_threshold, n_bins=n_bins, out=g.wps, counts=g.cov,
                             hist=packed[1:] if n_bins else None, ranges_ready=True)
        else:
            g.plan.run(g.frags, window_size, min_length, max_length, quality_threshold, out=g.wps)
        if adjust is not None:
            # every interval is a segment of the int32 WPS buffer as it lies in HBM (no gather, no float
            # copy); intervals shorter than the filters need produce no output, like the reference's driver
            ap = shard.adjust_plan(g, adjust)
            if ap.n_total:
                if g.adjusted is None or g.adjusted.numel() < ap.n_total:
                    g.adjusted = t.empty(ap.n_total, dtype=t.float64, device=dev)
                if ap.rank is not None and not general:
                    _, flag = ap.run_rank(g.wps, 0, g.adjusted)
                    flags.append((g, ap, flag.any()))
                else:
                    g.adjusted[: ap.n_total] = adjust_segments(g.wps, None, plan=ap, **adjust)[0]
    if flags and sync and bool(t.stack([f for _, _, f in flags]).any().item()):
        # a tile the rank kernel could not take (cannot happen for integer WPS of ordinary depth):
        # redo those groups on the general path
        for g, ap, f in flags:
            if bool(f.item()):
                g.adjusted[: ap.n_total] = adjust_segments(g.wps, None, plan=ap, impl="hist", **adjust)[0]
    if fused:
        if not cleared:
            packed.zero_()
        if shard.n_intervals:
            t.sum(shard.cov[: shard.n_intervals], dim=0, keepdim=True, out=packed[:1])
        if reduce:
            ctx.all_reduce_sum(packed)
    hist = packed[1:] if n_bins else None
    res = shard.results(fused, adjust, keep_adjusted)
    if not sync:
        for r in res.values():
            r.flags = [f for _, _, f in flags]
        return res, hist, (packed[:1] if fused else None)
    return res, hist, (int(packed[0].item()) if fused else None)


def table_shard(table, ctx: DistContext | None = None, device=None, contigs=None) -> "GenomeShard":
    """The count-only shard (no WPS tiles) of the contigs this rank owns, cached on the table."""
    from .device import require_cuda
    ctx = ctx or DistContext()
    dev = require_cuda(device)
    mine = list(contigs) if contigs is not None else owned_contigs(table, ctx)
    cache = table.__dict__.setdefault("_ftk_shards", {})
    key = (tuple(mine), str(dev))
    if key not in cache:
        sizes = {c: 0 for c in mine}
        sizes.update({c: n for c, n in (getattr(table, "contig_lengths", None) or {}).items() if c in sizes})
        cache[key] = GenomeShard(table, sizes, None, mine, 0, 1, dev)
    return cache[key]


def genome_bin_counts(table, bins: dict, n_bins: int = 0, intersect_policy="midpoint", min_length=None,
                      max_length=None, quality_threshold=30, ctx: DistContext | None = None, device=None,
                      contigs=None, cache_key=None):
    """Fragment counts of genome-wide bins {contig: (starts, stops)} (DELFI-style coverage,
    frag/_delfi.py:283-300 / frag/_coverage.py:215-254) and, with ``n_bins``, the genome-wide fragment-length
    dict of the counted fragments in first-seen order (frag/_frag_length.py:408-421) - contigs LPT-sharded,
    ONE kernel launch per rank, one ``all_reduce(SUM)`` of the packed counts (+ SUM / MIN for the dict).
    Returns ``({contig: int64[n] counts (host)}, dict | None)``, identical on every rank."""
    from .device import require_cuda, torch
    ctx = ctx or DistContext()
    dev = require_cuda(device)
    t = torch()
    shard = table_shard(table, ctx, dev, contigs)
    names = [c for c in table.contigs if c in bins]
    order = {c: i for i, c in enumerate(table.contigs)}
    offs = np.concatenate([[0], np.cumsum([len(bins[c][0]) for c in names])]).astype(np.int64)
    n_cnt = int(offs[-1])
    packed = t.zeros(max(n_cnt + int(n_bins), 1), dtype=t.int64, device=dev)      # [bin counts..., length histogram...]
    counts, hist, keys = shard.interval_counts(bins, order, intersect_policy, min_length, max_length, quality_threshold,
                                               n_bins=n_bins, first_seen=bool(n_bins), cache_key=cache_key)
    for i, c in enumerate(names):
        if c in counts:
            packed[int(offs[i]): int(offs[i + 1])] = counts[c]
    if n_bins and hist is not None:
        packed[n_cnt: n_cnt + n_bins] = hist
    ctx.all_reduce_sum(packed)                   # ONE SUM for counts and histogram
    host = packed.cpu().numpy()
    ldict = None
    if n_bins:
        if keys is None:
            from .sharding import FIRST_SEEN_NONE
            keys = t.full((n_bins,), FIRST_SEEN_NONE, dtype=t.int64, device=dev)
        ctx.all_reduce_min(keys)                 # + ONE MIN for the first-seen order
        h, k = host[n_cnt: n_cnt + n_bins], keys.cpu().numpy()
        nz = np.flatnonzero(h)
        nz = nz[np.argsort(k[nz], kind="stable")]
        ldict = {int(L): int(h[L]) for L in nz}
    return {c: host[int(offs[i]): int(offs[i + 1])] for i, c in enumerate(names)}, ldict


def adjust_wps_genome(results: dict, **adjust):
    """Adjust already computed device-resident WPS (``multi_wps_genome`` results) in place of the
    reference's bigWig -> adjust_wps -> bigWig pass (frag/_adjust_wps.py:59-111).  Interval i's adjusted
    series is ``res.adjusted[res.adj_offsets[i]: res.adj_offsets[i + 1]]`` (empty for intervals shorter
    than the filters need)."""
    from .device import AdjustPlan, adjust_segments
    for res in results.values():
        aplan = AdjustPlan(np.diff(res.offsets), int(adjust.get("median_window_size", 1000)),
                           adjust.get("savgol", True), adjust.get("savgol_window_size", 21),
                           adjust.get("savgol_poly_deg", 2), res.wps.device, skip_short=True)
        res.adj_offsets, res.adj_segments = aplan.out_off, np.flatnonzero(aplan.n_out > 0)
        if aplan.n_total:
            res.adjusted, _ = adjust_segments(res.wps, None, plan=aplan, **adjust)
    return results


def wps_spectrum_genome(results: dict, min_period=120, max_period=280) -> dict:
    """Periodograms (``device.spectrum_segments``) of every interval of ``multi_wps_genome`` results, from the
    adjusted series when the results hold them (``adjust=`` or ``adjust_wps_genome``), otherwise from the raw WPS -
    all in HBM.  Returns {contig: float64[n_intervals, n_periods] device tensor}; an interval with an empty series
    (too short for the filters) gives a row of NaN."""
    from .device import spectrum_check, spectrum_segments, torch
    spectrum_check(min_period, max_period)
    out = {}
    for c, res in results.items():
        if res.adj_offsets is None:
            x, off = res.wps, res.offsets
        else:
            if res.adjusted is None and res.adj_offsets[-1] > 0:
                raise ValueError(f"the results of {c} hold no adjusted series (keep_adjusted=False)")
            x = res.adjusted if res.adjusted is not None else torch().zeros(0, dtype=torch().float64,
                                                                              device=res.wps.device)
            off = res.adj_offsets
        out[c] = spectrum_segments(x, off, min_period, max_period)
    return out


def gather_to_writer(obj, ctx: DistContext | None = None):
    """Collect a picklable per-rank object on rank 0 (list in rank order; None elsewhere) - used by the
    file-writing API mirrors, whose single output file is written by rank 0 only."""
    ctx = ctx or DistContext()
    if not (ctx.on and ctx.world > 1):
        return [obj]
    out = [None] * ctx.world if ctx.rank == 0 else None
    ctx.dist.gather_object(obj, out, dst=0)
    return out
