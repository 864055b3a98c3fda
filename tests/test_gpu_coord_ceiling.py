"""Every fragment kernel at the top of the int32 coordinate space.

A contig may be up to 2^31 - 1 bases long, and ``distributed.GenomeShard`` lays a rank's contigs end to end in
one virtual int32 space of up to ``_SHARD_SPAN`` bases, so real runs put fragments, tiles and intervals near 2^31.
A sum such as ``start + stop`` wraps there.  The tests below translate a seeded contig (with pile-ups, zero-length
rows, long outliers and hand-placed rows ending at 2^31 - 1) up by ``B`` and require every kernel to give, bit for
bit, what the oracle gives for the untranslated contig.  Positions within reach of coordinate 0 (where the
reference clamps windows) are left out: the translation moves them away from that clamp."""
import numpy as np
import pytest

import depth_oracle as DO
import vplot_oracle as VO
from oracle import oracle as O

pytestmark = pytest.mark.gpu

TOP = 2 ** 31 - 1
CLEN = 200_000


def _np(x):
    return None if x is None else x.cpu().numpy()


def _sh(v, B):
    return None if v is None else int(v) + B


@pytest.fixture(scope="module")
def top():
    from finaletoolkit_b200 import device as D
    from finaletoolkit_b200.synth import synth_fragments, synth_twobit
    dev = D.require_cuda("cuda:0")
    rng = np.random.default_rng(2031)
    st, sp, mq, sd = (a.astype(np.int64) for a in synth_fragments(CLEN, 50_000, 0, seed_base=7731))
    st[1000:3000] = st[1000]; sp[1000:3000] = st[1000] + rng.integers(120, 181, 2000)   # a 2000-fold pile-up
    z = rng.choice(np.flatnonzero(st < CLEN - 3000), 40, replace=False)
    sp[z[:20]] = st[z[:20]]                                                          # zero-length rows
    sp[z[20:]] = st[z[20:]] + rng.integers(700, 2500, 20)                            # long outliers
    sp[-30:] = np.maximum(sp[-30:], CLEN + rng.integers(1, 400, 30))                 # past the synthetic contig end
    B = (TOP - (CLEN + 400)) & ~31            # a multiple of 32: the packed reference lines up with its words
    T = TOP - B                               # local coordinate that lands on 2^31 - 1
    hand_st = np.array([T - 170, T, T - 1, T - 2500] + [T - 167] * 300, np.int64)    # + a 300-fold pile-up at the top
    hand_sp = np.array([T, T, T, T] + [T] * 300, np.int64)
    st = np.concatenate([st, hand_st]); sp = np.concatenate([sp, hand_sp])
    mq = np.concatenate([mq, np.full(hand_st.size, 60, np.uint8)])
    sd = np.concatenate([sd, (np.arange(hand_st.size) & 1).astype(np.uint8)])
    order = np.argsort(st, kind="stable")
    st, sp, mq, sd = st[order], sp[order], mq[order], sd[order]
    assert int(sp.max()) + B == TOP and int(st.max()) + B == TOP
    st32, sp32 = st.astype(np.int32), sp.astype(np.int32)
    frB = D.ContigFragments((st + B).astype(np.int32), (sp + B).astype(np.int32), mq, sd, device=dev)
    # motifs / DELFI: a reference of length T (ending at 2^31 - 1 once translated) and rows long enough for a k-mer
    codes, nm = synth_twobit(T, 0, seed_base=5151, telomere=600, block_len=2500)
    seq = np.frombuffer(b"ACGT", np.uint8)[codes].copy(); seq[nm] = ord("N")
    km = (sp - st) >= 8
    frM = D.ContigFragments((st[km] + B).astype(np.int32), (sp[km] + B).astype(np.int32), mq[km], sd[km], device=dev)
    return dict(D=D, dev=dev, B=B, T=T, st=st32, sp=sp32, mq=mq, sd=sd, frB=frB, ofr=O.Frags(st32, sp32, mq, sd),
                frM=frM, ofrM=O.Frags(st32[km], sp32[km], mq[km], sd[km]), codes=codes, nm=nm, seq=seq.tobytes())


def _ivs(T, cs):
    """Intervals away from coordinate 0, clipped to a contig of size ``cs``; several end at ``T``."""
    ivs = [(5000, 10_000), (10_000, 15_119), (12_345, 12_346), (100_000, 111_111), (CLEN - 5000, CLEN),
           (CLEN - 3, CLEN + 200), (T - 5000, T), (T - 1, T), (T - 2 * 5119 - 3, T - 7), (T - 300, T)]
    return [(a, min(b, cs)) for a, b in ivs if min(b, cs) > a]


@pytest.mark.parametrize("cs_top", [False, True])
@pytest.mark.parametrize("W,lo,hi", [(120, 120, 180), (121, 0, 2600), (1, 0, 180)])
def test_wps_plain_and_fused(top, cs_top, W, lo, hi):
    """``WpsPlan.run`` and ``run_fused`` (int32 / int16 / int8 with the overflow flag, coverage, length histogram)."""
    import torch
    D, B, T, fr, ofr = top["D"], top["B"], top["T"], top["frB"], top["ofr"]
    cs = T if cs_top else CLEN
    ivs = _ivs(T, cs)
    s, e = [a for a, _ in ivs], [b for _, b in ivs]
    plan = D.WpsPlan([a + B for a in s], [b + B for b in e], cs + B, hi, top["dev"])
    exp, off = O.wps_intervals(ofr, s, e, cs, W, lo, hi, 30, threads=4)
    assert np.array_equal(off, plan.offsets)
    got = _np(plan.run(fr, W, lo, hi, 30)).astype(np.int64)
    assert np.array_equal(got, exp), (W, lo, hi, cs_top)
    n_bins = fr.max_len + 1
    exp_cov = O.interval_coverage(ofr, s, e, None, None, "midpoint", 30)
    exp_hist = np.zeros(n_bins, np.int64)
    for a, b in ivs:
        for L, c in O.length_dist(ofr, a, b, None, None, "midpoint", 30).items():
            exp_hist[L] += c
    peak = int(np.abs(exp).max())
    for dtype, lim in ((torch.int32, None), (torch.int16, 32767), (torch.int8, 127)):
        out = torch.empty(plan.n_positions, dtype=dtype, device=top["dev"])
        flag = torch.zeros(1, dtype=torch.int32, device=top["dev"])
        w, cov, h = plan.run_fused(fr, W, lo, hi, 30, None, None, 30, n_bins=n_bins, out=out, overflow=flag)
        assert np.array_equal(_np(cov), exp_cov) and np.array_equal(_np(h), exp_hist), (dtype, W)
        if lim is None or peak <= lim:
            assert int(flag.item()) == 0 and np.array_equal(_np(w).astype(np.int64), exp), (dtype, W, lo, hi)
        else:
            assert int(flag.item()) == 1, (dtype, W, peak)


def test_interval_hist_and_frag_lengths(top):
    """Counts, per-interval / pooled / pooled="hist" length histograms with first-seen order, ``None`` bounds,
    and the raw-length stream - including a zero-length row at 2^31 - 1 under an unbounded stop."""
    D, B, T, fr, ofr = top["D"], top["B"], top["T"], top["frB"], top["ofr"]
    ivs = _ivs(T, T) + [(None, 50_000), (T - 10, None), (None, None), (5000, T), (T, None)]
    s, e = [_sh(a, B) for a, _ in ivs], [_sh(b, B) for _, b in ivs]
    nb = fr.max_len + 1
    for pol, lo, hi, q in [("midpoint", None, None, 30), ("any", 0, None, 0), ("any", 100, 220, 30),
                           ("midpoint", 0, 600, 0)]:
        cnt = _np(D.interval_hist(fr, s, e, pol, lo, hi, q)[0])
        assert cnt.tolist() == [O.single_coverage(ofr, a, b, lo, hi, pol, q) for a, b in ivs], (pol, lo, hi, q)
        c1, h1, f1 = map(_np, D.interval_hist(fr, s, e, pol, lo, hi, q, n_bins=nb, first_seen=True))
        assert np.array_equal(c1, cnt)
        for j, (a, b) in enumerate(ivs):
            exp = O.length_dist(ofr, a, b, lo, hi, pol, q)
            nz = np.flatnonzero(h1[j])
            got = {int(nz[i]): int(h1[j][nz[i]]) for i in np.argsort(f1[j][nz], kind="stable")}
            assert got == exp and list(got) == list(exp), (pol, a, b)
        c2, h2, f2 = map(_np, D.interval_hist(fr, s, e, pol, lo, hi, q, n_bins=nb, pooled="hist", first_seen=True))
        assert np.array_equal(c2, cnt) and np.array_equal(h2[0], h1.sum(0)) and np.array_equal(f2[0], f1.min(0))
        c3, h3, f3 = map(_np, D.interval_hist(fr, s, e, pol, lo, hi, q, n_bins=nb, pooled=True, first_seen=True))
        assert int(c3[0]) == int(cnt.sum()) and np.array_equal(h3[0], h1.sum(0)) and np.array_equal(f3[0], f1.min(0))
    for a, b in [(5000, 20_000), (T - 3000, None), (None, None), (None, 7000), (T - 1, T), (T, None)]:
        for pol in ("midpoint", "any"):
            got = _np(D.frag_lengths(fr, _sh(a, B), _sh(b, B), pol, quality_threshold=30))
            assert np.array_equal(got, O.frag_lengths(ofr, a, b, pol, 30)), (a, b, pol)


@pytest.mark.parametrize("cs_top", [False, True])
def test_cleavage_and_depth(top, cs_top):
    D, B, T, fr, ofr = top["D"], top["B"], top["T"], top["frB"], top["ofr"]
    cs = T if cs_top else CLEN
    ivs = _ivs(T, cs)
    s, e = [a for a, _ in ivs], [b for _, b in ivs]
    for lo, hi, q in [(None, None, 30), (0, 2600, 0), (100, 200, 30)]:
        out, off = D.cleavage_intervals(fr, [a + B for a in s], [b + B for b in e], cs + B, lo, hi, q)
        out = _np(out)
        for k, (a, b) in enumerate(ivs):
            _, exp = O.cleavage_profile(ofr, cs, a, b, 0, 0, lo, hi, q)
            assert np.array_equal(out[off[k]:off[k + 1]], exp), (a, b, lo, hi, q)
        for midpoint in (False, True):
            got, goff = D.depth_intervals(fr, [a + B for a in s], [b + B for b in e], cs + B, lo, hi, q, midpoint)
            exp, eoff = DO.depth_intervals(top["st"], top["sp"], top["mq"], s, e, lo, hi, q, midpoint)
            assert np.array_equal(goff, eoff) and np.array_equal(_np(got).astype(np.int64), exp), (lo, hi, q, midpoint)


@pytest.mark.parametrize("flank,lo,hi", [(0, 0, 600), (37, 0, 2600), (1000, 100, 400)])
def test_vplot_windows_reaching_the_ceiling(top, flank, lo, hi):
    D, B, T = top["D"], top["B"], top["T"]
    c = np.array([T, T - 3, T - flank, T - max(flank - 1, 0), T - 2 * flank - 1, 100_000, CLEN, T - 500], np.int64)
    flip = (np.arange(c.size) % 2).astype(bool)
    exp = VO.vplot(top["st"], top["sp"], top["mq"], c, flip, flank, lo, hi, 30)
    got = _np(D.vplot_sites(top["frB"], c + B, flip, flank, lo, hi, 30))
    assert np.array_equal(got, exp), (flank, lo, hi)
    assert exp.sum() > 0
    with pytest.raises(ValueError, match="int32"):
        D.vplot_sites(top["frB"], np.array([TOP + 1]), [False], flank, lo, hi, 30)


@pytest.fixture(scope="module")
def big_ref(top):
    """The reference translated by B: zero words below B, the small contig's words above (~800 MB of HBM)."""
    from finaletoolkit_b200.synth import pack_twobit
    B, T = top["B"], top["T"]
    sw, nw = pack_twobit(top["codes"], top["nm"])
    big_s = np.zeros(B // 16 + sw.size, np.uint32); big_s[B // 16:] = sw
    big_n = np.zeros(B // 32 + nw.size, np.uint32); big_n[B // 32:] = nw
    ref = top["D"].PackedContig(big_s, big_n, B + T, top["dev"])
    del big_s, big_n
    yield ref
    del ref
    import torch
    torch.cuda.empty_cache()


@pytest.mark.parametrize("breakpoint", [False, True])
def test_end_and_breakpoint_motifs(top, big_ref, breakpoint):
    D, B, T = top["D"], top["B"], top["T"]
    ivs = _ivs(T, T)
    k = 6 if breakpoint else 4
    ref_fn = O.region_breakpoint_motifs if breakpoint else O.region_end_motifs
    for mode, (both, neg) in enumerate([(True, False), (False, False), (False, True)]):
        got = _np(D.end_motif_hist(top["frM"], big_ref, [a + B for a, _ in ivs], [b + B for _, b in ivs], k=k,
                                   strand_mode=mode, quality_threshold=30, breakpoint=breakpoint))
        for j, (a, b) in enumerate(ivs):
            exp = ref_fn(top["ofrM"], top["seq"], a, b, k, both, neg, 30)
            assert np.array_equal(got[j], exp), (breakpoint, mode, a, b)
        pooled = _np(D.end_motif_hist(top["frM"], big_ref, [a + B for a, _ in ivs], [b + B for _, b in ivs], k=k,
                                      strand_mode=mode, quality_threshold=30, breakpoint=breakpoint, pooled=True))
        assert np.array_equal(pooled[0], got.sum(0))


def test_delfi_windows(top, big_ref):
    D, B, T = top["D"], top["B"], top["T"]
    wins = [(5000, 55_000), (50_000, 100_000), (100_000, 150_000), (150_000, T), (T - 20_000, T), (T - 1, T)]
    rng = np.random.default_rng(3)
    r0 = np.sort(rng.integers(5000, T, 60)); r1 = np.minimum(r0 + rng.integers(1, 8000, 60), T)
    r0 = np.append(r0, T - 400); r1 = np.append(r1, T)
    order = np.lexsort((r1, r0)); blk = (r0[order], r1[order])
    gaps = ((80_000, 90_000), [(0, 3000), (T - 3000, T)])
    for g in (None, gaps):
        gB = None if g is None else ((g[0][0] + B, g[0][1] + B), [(a + B, b + B) for a, b in g[1]])
        got = _np(D.delfi_windows(top["frM"], big_ref, [a + B for a, _ in wins], [b + B for _, b in wins],
                                  blacklist=(blk[0] + B, blk[1] + B), gaps=gB, quality_threshold=30))
        for j, (a, b) in enumerate(wins):
            assert np.array_equal(got[j], O.delfi_counts(top["ofrM"], top["seq"], a, b, blk, g, 30)), (a, b, g is None)


# ---------------------------------------------------------------------------------------------------------------
# A genome shard whose working contig ends right below _SHARD_SPAN, with the real span (not patched down)
# ---------------------------------------------------------------------------------------------------------------
def test_shard_at_the_top_of_its_span():
    import torch
    from finaletoolkit_b200 import distributed as FD
    from finaletoolkit_b200.device import AdjustPlan, WpsPlan, adjust_segments, require_cuda
    from finaletoolkit_b200.io.fragments import FragmentTable
    from finaletoolkit_b200.synth import synth_fragments
    dev = require_cuda("cuda:0")
    rng = np.random.default_rng(77)
    work = 61_003
    pad1 = 1_070_000_000
    pad2 = FD._SHARD_SPAN - 80_000 - pad1 - work       # the guards add 14-30 kb: the working contig ends 50-66 kb short
    sizes = {"pad1": pad1, "pad2": pad2, "work": work}
    cols, sites = {}, {}
    for i, (c, n) in enumerate(sizes.items()):
        span = min(n, 200_000)
        st, sp, mq, sd = synth_fragments(span, 3000 if c != "work" else 20_000, i, seed_base=990)
        st = st.astype(np.int64) + (n - span); sp = sp.astype(np.int64) + (n - span)     # near the contig's own end
        z = rng.choice(st.size, 5, replace=False); sp[z] = st[z]
        j = rng.choice(st.size, 5, replace=False); sp[j] = st[j] + rng.integers(700, 2500, 5)
        sp[-3:] = n + np.array([5, 40, 300])
        order = np.argsort(st, kind="stable")
        cols[c] = (st[order].astype(np.int32), sp[order].astype(np.int32), mq[order], sd[order])
        if c == "work":
            edges = np.arange(0, n + 5000, 5000, dtype=np.int64).clip(max=n)
            sites[c] = (edges[:-1].copy(), edges[1:].copy())
        else:
            s0 = np.array([n - 150_000, n - 60_000, n - 9000], np.int64)
            sites[c] = (s0, s0 + np.array([5000, 7001, 9000]))
    table = FragmentTable(cols)
    adj = dict(median_window_size=1000, savgol=True, savgol_window_size=21, savgol_poly_deg=2)
    plans = {}
    res, hist, tot = FD.multi_wps_genome(table, list(sizes.items()), sites, 5000, 120, 120, 180, 30, coverage=True,
                                         length_hist=True, adjust=adj, device=dev, contigs=list(sizes), plans=plans)
    shard = next(iter(plans.values()))
    assert len(shard.groups) == 1
    lay = shard.layout["work"]
    end = lay["base"] + lay["span"][1]
    assert FD._SHARD_SPAN - 100_000 <= end <= FD._SHARD_SPAN, (end, FD._SHARD_SPAN)
    exp_hist = np.zeros(hist.numel(), np.int64)
    for c, n in sizes.items():
        fr = table.device(c, dev)
        s, e = sites[c]
        plan = WpsPlan(s, e, n, 180, dev)
        wps, cov, h = plan.run_fused(fr, 120, 120, 180, 30, None, None, 30, n_bins=hist.numel())
        r = res[c]
        assert torch.equal(r.wps, wps[: plan.n_positions]) and torch.equal(r.cov, cov), c
        exp_hist += _np(h)
        ap = AdjustPlan(np.diff(plan.offsets), 1000, True, 21, 2, dev, skip_short=True)
        assert np.array_equal(r.adj_offsets, ap.out_off) and ap.n_total
        a, _ = adjust_segments(wps, None, plan=ap, **adj)
        assert torch.equal(r.adjusted, a), c
        ofr = O.Frags(*cols[c])
        exp, _ = O.wps_intervals(ofr, s, e, n, 120, 120, 180, 30, threads=4)
        assert np.array_equal(_np(r.wps).astype(np.int64), exp), c
        assert np.array_equal(_np(r.cov), O.interval_coverage(ofr, s, e, None, None, "midpoint", 30)), c
    assert np.array_equal(_np(hist), exp_hist) and tot == sum(int(r.cov.sum()) for r in res.values())

    # the count-only shard (bins, whole-contig length dict) over the same contigs
    frs = {c: O.Frags(*cols[c]) for c in sizes}
    bins = {c: (np.arange(n - 200_000, n, 10_000, dtype=np.int64),
                np.minimum(np.arange(n - 200_000, n, 10_000, dtype=np.int64) + 10_000, n)) for c, n in sizes.items()
            if c != "work"}
    bins["work"] = (np.arange(0, work, 10_000, dtype=np.int64), np.minimum(np.arange(0, work, 10_000) + 10_000, work))
    got, ldict = FD.genome_bin_counts(table, bins, n_bins=2600, quality_threshold=30, device=dev, contigs=list(sizes))
    cshard = FD.table_shard(table, device=dev, contigs=list(sizes))
    assert len(cshard.groups) == 1
    assert cshard.layout["work"]["base"] + cshard.layout["work"]["span"][1] > 2 * 1_000_000_000
    for c in sizes:
        assert np.array_equal(got[c], O.interval_coverage(frs[c], bins[c][0], bins[c][1], None, None, "midpoint", 30)), c
    exp_dict = O.merge_dists(O.length_dist(frs[c], int(a), int(b), None, None, "midpoint", 30)
                             for c in sizes for a, b in zip(*bins[c]))
    assert {k: v for k, v in exp_dict.items() if k < 2600} == ldict
    d = FD.genome_length_distribution(table, min_length=0, max_length=None, quality_threshold=30, device=dev)
    exp = O.merge_dists(O.length_dist(frs[c], None, None, 0, None, "midpoint", 30) for c in sizes)
    assert d == exp and list(d) == list(exp)
