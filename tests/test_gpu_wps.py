"""CUDA WPS (through the C ABI) vs the reference goldens and the CPU oracle."""
import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    import torch
    from finaletoolkit_b200.device import require_cuda
    return require_cuda("cuda:0")


def _run(frags_dev, ivs, chrom_size, **kw):
    """ivs: list of (start, stop). Returns list of int64 arrays (one per interval)."""
    import torch
    from finaletoolkit_b200.device import WpsPlan
    kw = {"window_size": 120, "min_length": 120, "max_length": 180, "quality_threshold": 30, **kw}
    plan = WpsPlan([s for s, _ in ivs], [e for _, e in ivs], chrom_size, kw["max_length"], frags_dev.device)
    out = plan.run(frags_dev, **kw)
    torch.cuda.synchronize()
    host = out.cpu().numpy().astype(np.int64)
    return [host[plan.offsets[i]:plan.offsets[i + 1]] for i in range(len(ivs))]


def _dev_frags(g, prefix, dev):
    from finaletoolkit_b200.device import ContigFragments
    return ContigFragments(g[prefix + "start"], g[prefix + "stop"], g[prefix + "mapq"], g[prefix + "strand"], device=dev)


def test_fixture17_known_answers(manifest, golden, dev):
    g = golden("fixture17")
    m = manifest["fixture17"]
    fr = _dev_frags(g, "", dev)
    for i, c in enumerate(m["wps_cases"]):
        got = _run(fr, [(c["start"], c["stop"])], m["chrom_size"], **c["kwargs"])[0]
        assert np.array_equal(got, g[f"wps_{i}"]), c
    got = _run(fr, [(34444145, 34444155)], 133851895, quality_threshold=0)[0]
    assert got.tolist() == [-1] * 5 + [1] * 5  # reference tests/test_wps.py:18-26
    # config 1: the two truncated windows of intervals.bed in ONE launch
    got = _run(fr, [(34440828, 34443041), (34443041, 34448041)], m["chrom_size"])
    assert np.array_equal(np.concatenate(got), g["mwps_cfg1_score"])


def test_synth_small_golden(manifest, golden, dev):
    g = golden("synth_small")
    m = manifest["synth_small"]
    sizes = dict(m["contigs"])
    frs = {c: _dev_frags(g, c + "_", dev) for c in sizes}
    for c in m["wps_cases"]:
        got = _run(frs[c["contig"]], [(c["start"], c["stop"])], sizes[c["contig"]], **c["kwargs"])[0]
        assert np.array_equal(got, g[c["key"]]), c


@pytest.mark.parametrize("seed", range(6))
def test_random_vs_oracle(seed, dev):
    """Randomised parameters / interval shapes; oracle = literal brute force."""
    from finaletoolkit_b200.device import ContigFragments
    from finaletoolkit_b200.synth import synth_fragments
    rng = np.random.default_rng(seed)
    clen = int(rng.integers(20_000, 120_000))
    n = int(rng.integers(0, 40_000)) if seed else 0
    st, sp, mq, sd = synth_fragments(clen, n, seed, seed_base=555)
    if n:  # push some fragments past the contig end and make heavy pile-ups
        k = min(50, n)
        sp[-k:] = np.minimum(sp[-k:] + 300, np.iinfo(np.int32).max)
        st[: n // 10] = st[0]
        order = np.argsort(st, kind="stable"); st, sp, mq, sd = st[order], sp[order], mq[order], sd[order]
    ofr = O.Frags(st, sp, mq, sd)
    dfr = ContigFragments(st, sp, mq, sd, device=dev)
    W = int(rng.choice([1, 2, 3, 20, 59, 60, 119, 120, 121, 200, 333]))
    lo = int(rng.choice([0, 1, 30, 120, 150])); hi = int(lo + rng.choice([0, 1, 30, 60, 450]))
    q = int(rng.choice([0, 1, 30, 60, 61]))
    ivs = []
    for _ in range(12):
        s = int(rng.integers(-50, clen)); e = s + int(rng.integers(0, 12_000))
        ivs.append((max(s, 0), min(e, clen + 100)))
    ivs += [(0, 1), (clen - 1, clen), (0, 5119), (0, 5120), (0, 5121), (7, 10_243), (clen - 3000, clen)]
    got = _run(dfr, ivs, clen, window_size=W, min_length=lo, max_length=hi, quality_threshold=q)
    for (s, e), gv in zip(ivs, got):
        exp = O.wps_interval(ofr, s, e, clen, W, lo, hi, q)
        assert np.array_equal(gv, exp), (seed, W, lo, hi, q, s, e)


@pytest.mark.parametrize("W,lo,hi", [(120, 120, 180), (16, 35, 80), (121, 121, 300), (59, 60, 450), (2, 2, 600),
                                      (1, 1, 200), (250, 250, 600), (253, 253, 400), (120, 119, 180)])
def test_window_and_length_grid_vs_oracle(W, lo, hi, dev):
    """Even / odd / tiny / wide windows with lengths straddling both bounds (many L == W),
    a pile-up on one start and fragments past the contig end."""
    from finaletoolkit_b200.device import ContigFragments
    from finaletoolkit_b200.synth import synth_fragments
    rng = np.random.default_rng(W * 1000 + lo)
    clen = 61_000
    st, sp, mq, sd = synth_fragments(clen, 30_000, W, seed_base=31)
    ln = rng.integers(max(lo - 3, 1), hi + 4, st.size)
    ln[rng.random(st.size) < 0.2] = max(W, lo)
    sp = (st + ln).astype(np.int32)
    st[:3000] = st[0]; sp[:3000] = st[0] + ln[:3000]
    st[-40:] = clen - 5; sp[-40:] = clen + ln[-40:]
    order = np.argsort(st, kind="stable"); st, sp, mq, sd = st[order], sp[order], mq[order], sd[order]
    ofr = O.Frags(st, sp, mq, sd); dfr = ContigFragments(st, sp, mq, sd, device=dev)
    ivs = [(0, 5000), (5000, 10_000), (clen - 700, clen), (12_345, 12_346), (3, 5122)]
    got = _run(dfr, ivs, clen, window_size=W, min_length=lo, max_length=hi, quality_threshold=30)
    for (s, e), a in zip(ivs, got):
        assert np.array_equal(a, O.wps_interval(ofr, s, e, clen, W, lo, hi, 30)), (W, lo, hi, s, e)


def test_deep_pile_up_exact(dev):
    """70 000 fragments starting on one base (|WPS| > 65535): int32 scores stay exact and the
    range scratch is reusable with ``ranges_ready``."""
    import torch
    from finaletoolkit_b200.device import ContigFragments, WpsPlan
    rng = np.random.default_rng(4)
    clen, n = 20_000, 150_000
    st = rng.integers(4_000, 9_000, n).astype(np.int32)
    st[:70_000] = 6_000
    st = np.sort(st)
    sp = (st + rng.integers(120, 181, n)).astype(np.int32)
    mq = np.full(n, 60, np.uint8)
    ofr = O.Frags(st, sp, mq, np.ones(n, np.uint8)); dfr = ContigFragments(st, sp, mq, None, device=dev)
    ivs = [(0, 5000), (5000, 10_000), (10_000, 15_000)]
    got = _run(dfr, ivs, clen)
    for (s, e), a in zip(ivs, got):
        assert np.array_equal(a, O.wps_interval(ofr, s, e, clen)), (s, e)
    assert min(int(a.min()) for a in got) < -65535
    plan = WpsPlan([s for s, _ in ivs], [e for _, e in ivs], clen, 180, dev)
    plan.ranges(dfr); torch.cuda.synchronize()
    before = plan.scratch.clone()
    out = plan.run(dfr, ranges_ready=True); torch.cuda.synchronize()
    assert torch.equal(plan.scratch, before)
    assert np.array_equal(out.cpu().numpy().astype(np.int64), np.concatenate(got))


def test_no_mapq_column_and_empty(dev):
    from finaletoolkit_b200.device import ContigFragments
    st = np.array([100, 150, 150, 400], np.int32); sp = st + np.array([167, 121, 180, 130], np.int32)
    dfr = ContigFragments(st, sp, None, None, device=dev)
    ofr = O.Frags(st, sp, np.full(4, 255, np.uint8))
    got = _run(dfr, [(0, 1000), (5, 5)], 1000)
    assert np.array_equal(got[0], O.wps_interval(ofr, 0, 1000, 1000))
    assert got[1].size == 0
    empty = ContigFragments(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.uint8), None, device=dev)
    assert not _run(empty, [(0, 6000)], 10_000)[0].any()


def wps_total_closed_form(st, sp, mq, clen, W, lo, hi, q):
    """Sum over c in [0, clen) of WPS(c) from per-fragment range lengths (even W)."""
    a_, b_ = W // 2, W // 2 - 1
    fs = st.astype(np.int64); fe = sp.astype(np.int64); L = fe - fs
    ok = (mq >= q) & (L >= lo) & (L <= hi)
    fs, fe, L = fs[ok], fe[ok], L[ok]

    def clipped(x0, x1):
        return np.maximum(np.minimum(x1, clen - 1) - np.maximum(x0, 0) + 1, 0)

    short = L <= W
    tot = -clipped(fs - b_, fe + a_)[short].sum()
    lg = ~short
    tot += (-clipped(fs - b_, fs + a_) + clipped(fs + a_ + 1, fe - b_ - 1) - clipped(fe - b_, fe + a_))[lg].sum()
    return int(tot)


def test_full_size_properties(dev):
    """Size-independent checks at chr-scale: tiling invariance and a checksum identity.

    The sum over all positions of WPS equals the sum over passing fragments of
    the (contig-clipped) lengths of their -1/+1/-1 ranges: an oracle-free identity.
    """
    import torch
    from finaletoolkit_b200.device import ContigFragments, WpsPlan
    from finaletoolkit_b200.synth import synth_fragments
    clen, n = 20_000_000, 6_000_000
    st, sp, mq, sd = synth_fragments(clen, n, 3)
    dfr = ContigFragments(st, sp, mq, sd, device=dev)
    W, lo, hi, q = 120, 120, 180, 30
    # (1) 5 kb tiling == one long interval == 1237-bp tiling
    edges = np.arange(0, clen + 5000, 5000).clip(max=clen)
    a = WpsPlan(edges[:-1], edges[1:], clen, hi, dev).run(dfr, W, lo, hi, q)
    b = WpsPlan([0], [clen], clen, hi, dev).run(dfr, W, lo, hi, q)
    e2 = np.arange(0, clen + 1237, 1237).clip(max=clen)
    c = WpsPlan(e2[:-1], e2[1:], clen, hi, dev).run(dfr, W, lo, hi, q)
    assert torch.equal(a, b) and torch.equal(a, c)
    # (2) checksum of checksums: closed-form total of every passing fragment's clipped ranges
    ofr = O.Frags(st, sp, mq, sd)
    ah = a.cpu().numpy()
    assert int(ah.sum(dtype=np.int64)) == wps_total_closed_form(st, sp, mq, clen, W, lo, hi, q)
    # (3) random 5 kb intervals against the oracle
    rng = np.random.default_rng(0)
    for s in rng.integers(0, clen - 5000, 40).tolist():
        assert np.array_equal(ah[s:s + 5000], O.wps_interval(ofr, s, s + 5000, clen, W, lo, hi, q))


def test_streamed_pipeline_matches_resident(dev):
    """Chunked host->device->host pipeline (int16 WPS on the wire) == the resident int32 path."""
    import torch
    from finaletoolkit_b200 import device as D
    from finaletoolkit_b200.pipeline import StreamedContig
    from finaletoolkit_b200.synth import synth_fragments
    clen, n = 3_000_000, 900_000
    st, sp, mq, sd = synth_fragments(clen, n, 5)
    edges = np.arange(0, clen + 5000, 5000).clip(max=clen)
    fr = D.ContigFragments(st, sp, mq, sd, device=dev)
    ref = D.WpsPlan(edges[:-1], edges[1:], clen, 180, dev).run(fr).cpu().numpy()
    cov, _, _ = D.interval_hist(fr, edges[:-1].tolist(), edges[1:].tolist())
    tot, hist, _ = D.interval_hist(fr, [0], [None], n_bins=fr.max_len + 1, pooled=True)
    for chunks in (1, 3, 7):
        pipe = StreamedContig(torch.from_numpy(st).pin_memory(), torch.from_numpy(sp).pin_memory(),
                              torch.from_numpy(mq).pin_memory(), edges[:-1], edges[1:], clen, n_chunks=chunks, device=dev)
        for _ in range(2):   # twice: buffers and events are reused across runs
            w, c, h, t = pipe.run()
        assert np.array_equal(w.numpy()[: pipe.n_positions].astype(np.int32), ref)
        assert np.array_equal(c.numpy(), cov.cpu().numpy()) and int(t[0]) == int(tot[0])
        assert np.array_equal(h.numpy(), hist.cpu().numpy())
    # int8 on the wire: exact while |WPS| <= 127 (this 50x-like shard stays below), flagged otherwise
    assert np.abs(ref).max() <= 127
    pipe8 = StreamedContig(torch.from_numpy(st).pin_memory(), torch.from_numpy(sp).pin_memory(),
                           torch.from_numpy(mq).pin_memory(), edges[:-1], edges[1:], clen, n_chunks=4, device=dev,
                           wps_dtype="int8")
    w8, c8, h8, t8 = pipe8.run()
    assert w8.dtype == torch.int8 and np.array_equal(w8.numpy()[: pipe8.n_positions].astype(np.int32), ref)
    assert np.array_equal(c8.numpy(), cov.cpu().numpy()) and pipe8.d2h_bytes < pipe.d2h_bytes
    # WPS alone (no coverage, no histogram) runs the plain kernel with narrow outputs: even and odd window
    ref121 = D.WpsPlan(edges[:-1], edges[1:], clen, 180, dev).run(fr, 121).cpu().numpy()
    assert np.abs(ref121).max() <= 127
    for W, exp in ((120, ref), (121, ref121)):
        for dtype in ("int16", "int8"):
            plain = StreamedContig(torch.from_numpy(st).pin_memory(), torch.from_numpy(sp).pin_memory(),
                                   torch.from_numpy(mq).pin_memory(), edges[:-1], edges[1:], clen, window_size=W,
                                   n_chunks=3, device=dev, coverage=False, length_hist=False, wps_dtype=dtype)
            wp, _, _, _ = plain.run()
            assert np.array_equal(wp.numpy()[: plain.n_positions].astype(np.int32), exp), (W, dtype)
    deep_s = np.sort(np.random.default_rng(2).integers(1000, 1400, 30_000)).astype(np.int32)
    deep = StreamedContig(torch.from_numpy(deep_s).pin_memory(), torch.from_numpy(deep_s + 150).pin_memory(),
                          torch.full((30_000,), 60, dtype=torch.uint8).pin_memory(), [0], [5000], 10_000, device=dev,
                          wps_dtype="int8")
    with pytest.raises(OverflowError, match="int16"):
        deep.run()
    # int16 overflow is detected, not silently wrapped: 40000 identical fragments
    big_s = np.full(40_000, 1000, np.int32); big_e = big_s + 150
    pipe = StreamedContig(torch.from_numpy(big_s).pin_memory(), torch.from_numpy(big_e).pin_memory(),
                          torch.full((40_000,), 60, dtype=torch.uint8).pin_memory(), [0], [5000], 10_000, device=dev)
    with pytest.raises(OverflowError):
        pipe.run()
