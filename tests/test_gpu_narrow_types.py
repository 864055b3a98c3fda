"""The kernels' narrow internal types at their exact limits, and the fallback each one has.

- int16 / int8 WPS outputs raise an overflow flag (``store4`` / ``store1`` in ftk_wps.cu): +32767 and -32768 fit,
  +32768 and -32769 do not (127 / -128 for int8), in the vector stores and in the scalar head / tail alike.
- ``multi_wps`` streams large contigs with int16 scores and falls back to the int32 path on overflow.
- The adjust rank kernel stages samples as int16 and takes |x| <= 32000 (``kRankMaxAbs``); larger tiles are flagged
  and redone on the histogram path, by ``adjust_segments`` and by ``multi_wps_genome``.  Its exact sliding-moment
  Savitzky-Golay keeps moments in int32 while |2 adj| < 2^17.  The smoothed output is checked against exact
  rational arithmetic, to the rounding error of an fp64 dot product.
- Length histograms are privatised in shared memory below 1024 (fused WPS) / 2048 (interval kernels) bins and go
  through global atomics above, up to ``n_bins``."""
from fractions import Fraction

import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps


@pytest.fixture(scope="module")
def dev():
    from finaletoolkit_b200.device import require_cuda
    return require_cuda("cuda:0")


def _np(x):
    return None if x is None else x.cpu().numpy()


# ------------------------------------------------------------------------------------------------------ B1
S0 = 5000


def _plans():
    """(name, intervals): aligned int4 stores only / an output offset of 1 (scalar stores only) / 3-position tiles
    (the scalar tail) on the plateau of long fragments and on the trough."""
    return [("vec", [(S0 - 400, S0 + 600)]),
            ("unaligned", [(S0 - 401, S0 - 400), (S0 - 400, S0 + 600)]),
            ("tail_plateau", [(S0 + 78, S0 + 81)]),
            ("tail_trough", [(S0, S0 + 3)])]


@pytest.mark.parametrize("dtype,N", [("int8", 127), ("int8", 128), ("int8", 129),
                                     ("int16", 32767), ("int16", 32768), ("int16", 32769)])
@pytest.mark.parametrize("long", [True, False])
def test_wps_overflow_flag_at_the_exact_boundary(dev, dtype, N, long):
    """N identical fragments: L > W gives a plateau of +N and troughs of -N; L <= W gives -N only."""
    import torch
    from finaletoolkit_b200.device import ContigFragments, WpsPlan
    from finaletoolkit_b200.pipeline import StreamedContig
    L, lo = (160, 120) if long else (100, 0)
    st = np.full(N, S0, np.int32); sp = st + L; mq = np.full(N, 60, np.uint8)
    fr = ContigFragments(st, sp, mq, None, device=dev)
    tdt = getattr(torch, dtype)
    hi_ok, lo_ok = (127, -128) if dtype == "int8" else (32767, -32768)
    for name, ivs in _plans():
        s, e = [a for a, _ in ivs], [b for _, b in ivs]
        plan = WpsPlan(s, e, 20_000, 180, dev)
        ref = _np(plan.run(fr, 120, lo, 180, 30)).astype(np.int64)
        assert np.array_equal(ref, np.concatenate([O.wps_interval(O.Frags(st, sp, mq), a, b, 20_000, 120, lo, 180, 30)
                                                   for a, b in ivs]))
        if name.startswith("tail"):     # the boundary value itself sits in the scalar tail
            assert (ref == (N if long and name == "tail_plateau" else -N)).all(), (name, long)
        else:                            # ... and in full int4 groups / unaligned scalar stores
            assert int(ref.min()) == -N and int(ref.max()) == (N if long else 0), (name, long)
        bad = bool((ref > hi_ok).any() or (ref < lo_ok).any())
        # the fused kernel shape
        out = torch.empty(plan.n_positions, dtype=tdt, device=dev)
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        plan.run_fused(fr, 120, lo, 180, 30, None, None, 30, out=out, overflow=flag)
        assert int(flag.item()) == int(bad), (name, dtype, N, long)
        if not bad:
            assert np.array_equal(_np(out).astype(np.int64), ref), (name, dtype, N, long)
        # the plain kernel shape (WPS alone, through the streamed pipeline)
        pipe = StreamedContig(torch.from_numpy(st).pin_memory(), torch.from_numpy(sp).pin_memory(),
                              torch.from_numpy(mq).pin_memory(), s, e, 20_000, 120, lo, 180, 30, n_chunks=1,
                              device=dev, coverage=False, length_hist=False, wps_dtype=dtype)
        if bad:
            with pytest.raises(OverflowError):
                pipe.run()
        else:
            w, _, _, _ = pipe.run()
            assert np.array_equal(w.numpy()[: pipe.n_positions].astype(np.int64), ref), (name, dtype, N, long)


# ------------------------------------------------------------------------------------------------------ B2
def test_multi_wps_falls_back_from_int16_streaming(dev, tmp_path, monkeypatch):
    import gzip

    import finaletoolkit_b200 as F
    from finaletoolkit_b200.frag import _multi_wps, _wps
    from finaletoolkit_b200.io.fragments import FragmentTable
    from finaletoolkit_b200.io.textout import bedgraph_text
    from finaletoolkit_b200.synth import synth_fragments
    clen = 300_000
    st, sp, mq, sd = synth_fragments(clen, 60_000, 0, seed_base=6060)
    pile = 147_000                  # a site of its own: no neighbour truncates its window
    st = np.concatenate([st, np.full(40_000, pile, np.int32)]); sp = np.concatenate([sp, np.full(40_000, pile + 160, np.int32)])
    mq = np.concatenate([mq, np.full(40_000, 60, np.uint8)]); sd = np.concatenate([sd, np.ones(40_000, np.uint8)])
    order = np.argsort(st, kind="stable"); st, sp, mq, sd = st[order], sp[order], mq[order], sd[order]
    cs = tmp_path / "chrom.sizes"; cs.write_text(f"chrA\t{clen}\n")
    centres = np.arange(10_000, clen - 10_000, 12_000).tolist() + [pile]
    bed = tmp_path / "sites.bed"; bed.write_text("".join(f"chrA\t{c}\t{c + 1}\n" for c in sorted(centres)))
    assert len(centres) >= 16
    monkeypatch.setattr(_wps, "_STREAM_MIN_FRAGMENTS", 1000)

    def run(name, cols):
        out = str(tmp_path / name)
        F.multi_wps(FragmentTable({"chrA": cols}), str(bed), chrom_sizes=str(cs), output_file=out)
        with gzip.open(out, "rt") as fh:
            return fh.read(), _multi_wps.LAST_TIMINGS["streamed_contigs"]

    # control: without the pile-up the contig streams
    keep = ~((st == pile) & (sp == pile + 160))
    _, n_streamed = run("plain.bed.gz", (st[keep], sp[keep], mq[keep], sd[keep]))
    assert n_streamed == 1
    txt, n_streamed = run("pile.bed.gz", (st, sp, mq, sd))
    assert n_streamed == 0                               # int16 overflowed: the contig went the resident int32 way
    monkeypatch.setattr(_wps, "_STREAM_MIN_FRAGMENTS", 1 << 40)
    txt_resident, n_streamed = run("resident.bed.gz", (st, sp, mq, sd))
    assert n_streamed == 0 and txt == txt_resident
    exp = O.wps_interval(O.Frags(st, sp, mq, sd), pile - 2500, pile + 2500, clen)
    assert int(np.abs(exp).max()) > 32767
    assert bedgraph_text("chrA", pile - 2500, exp).tobytes().decode() in txt


# ------------------------------------------------------------------------------------------------------ B3
def exact_check(got, x, w, sg, tag=""):
    """``got``: adjusted series of the integer samples ``x``.  Without smoothing it must equal ``O.local_filter``
    bit for bit.  With smoothing ``sg = (window, degree)``, each output is compared with exact rational arithmetic:
    interior outputs with the rational coefficients of ``savgol_rational``, the edge rows with the fp64 hat matrix
    of ``savgol_tables`` taken as exact doubles.  The bound is window * eps * sum |c_i x_i| (the error of an fp64
    dot product of that many terms; the exact sliding moments do better) plus, in the interior, sum |dc_i x_i|
    with dc_i the difference between the fp64 stencil and the exact coefficient."""
    from finaletoolkit_b200.device import savgol_rational, savgol_tables
    pre = O.local_filter(np.asarray(x, np.float64), w)
    if sg is None:
        assert np.array_equal(got, pre), tag
        return
    m, deg = sg
    h = m // 2
    adj2 = np.rint(2 * pre).astype(np.int64)                  # 2 * adjusted: an integer
    assert np.array_equal(adj2 / 2, pre)
    n = adj2.size
    coef, first, last = savgol_tables(m, deg)
    a, b, den = savgol_rational(m, deg)
    assert den > 0
    k = np.array([a + b * i * i for i in range(-h, h + 1)], np.int64)
    num = np.convolve(adj2, k[::-1], "valid")                  # interior: y = num / (2 den), exactly
    dc = np.array([float(abs(Fraction(float(c)) - Fraction(int(kk), den))) for c, kk in zip(coef, k)])
    mag = np.convolve(np.abs(adj2), np.abs(coef)[::-1], "valid") / 2
    dmag = np.convolve(np.abs(adj2), dc[::-1], "valid") / 2
    for j in range(h, n - h):
        err = abs(Fraction(float(got[j])) - Fraction(int(num[j - h]), 2 * den))
        lim = m * EPS * float(mag[j - h]) * (1 + 1e-9) + float(dmag[j - h]) * (1 + 1e-9)
        assert err <= Fraction(lim), (tag, j, float(err), lim)
    for rows, base, js in ((first, 0, range(h)), (last, n - m, range(n - h, n))):
        for r, j in enumerate(js):
            c = rows[r]
            exact = sum(Fraction(float(ci)) * Fraction(int(v), 2) for ci, v in zip(c, adj2[base: base + m]))
            lim = m * EPS * float(np.sum(np.abs(c) * np.abs(adj2[base: base + m]) / 2)) * (1 + 1e-9)
            assert abs(Fraction(float(got[j])) - exact) <= Fraction(lim), (tag, "edge", j)


def _series(rng, n, kind):
    if kind == "walk32000":          # a random walk with spikes to exactly +-32000
        v = np.cumsum(rng.integers(-3, 4, n)); v[rng.choice(n, 40, replace=False)] = 32000
        v[rng.choice(n, 40, replace=False)] = -32000
        return v
    if kind in ("low", "high"):      # a +-32000 plateau with spikes to the other extreme: |2 adj| reaches 128 000
        sgn = -1 if kind == "low" else 1
        v = np.full(n, sgn * 32000); v[rng.choice(n, n // 50, replace=False)] = -sgn * 32000
        return v
    v = np.cumsum(rng.integers(-3, 4, n))
    spike = {"32001": 32001, "-32001": -32001, "65535": 65535, "-70000": -70000}[kind]
    v[rng.choice(n, 3, replace=False)] = spike
    return v


SG = [None, (21, 2), (5, 2), (51, 3)]


@pytest.mark.parametrize("w", [2, 1000])
@pytest.mark.parametrize("sg", SG, ids=["nosg", "sg21", "sg5", "sg51"])
def test_adjust_rank_kernel_at_kRankMaxAbs(dev, w, sg):
    import torch
    from finaletoolkit_b200.device import adjust_segments
    rng = np.random.default_rng(w + (0 if sg is None else sg[0]))
    kw = dict(median_window_size=w, savgol=sg is not None)
    if sg is not None:
        kw.update(savgol_window_size=sg[0], savgol_poly_deg=sg[1])
    for kinds, fits in ((["walk32000", "low", "high"], True), (["32001", "-32001", "65535", "-70000"], False)):
        xs = [_series(rng, w + 3000 + 7 * i, kd) for i, kd in enumerate(kinds)]
        lens = [x.size for x in xs]
        x = np.concatenate(xs)
        assert int(np.abs(x).max()) == 32000 if fits else int(np.abs(x).max()) > 32000
        for xin in (x.astype(np.float32), torch.from_numpy(x.astype(np.int32)).to(dev)):
            _, _, flag = adjust_segments(xin, lens, **kw, defer_check=True)
            # staging refuses |x| > 32000 whatever the window; with w = 1000 the median of these series stays on one
            # level band, so the rank kernel must take them (with w = 2 a spike moves the median by 32 000 levels,
            # past the kernel's band search: a flag there is by design, and the output is checked either way)
            assert flag is not None
            if not fits or w == 1000:
                assert bool(flag.any().item()) != fits, (kinds, w, sg)
            got, off = adjust_segments(xin, lens, **kw)
            got = _np(got)
            for i, xi in enumerate(xs):
                exact_check(got[off[i]: off[i + 1]], xi, w, sg, (kinds[i], w, sg))
    if w == 1000:   # the alternating blocks do reach the bound of the exact moments
        pre = O.local_filter(np.asarray(_series(rng, w + 3000, "low"), np.float64), w)
        assert float(np.abs(2 * pre).max()) == 128_000.0


@pytest.mark.parametrize("seed", range(3))
def test_adjust_random_series_to_fp64_rounding(seed):
    """The random integer series of the existing rank-kernel test, held to the exact bound instead of 1e-5."""
    from finaletoolkit_b200.device import adjust_segments
    from test_gpu_adjust import _int_series
    rng = np.random.default_rng(50 + seed)
    w = int(rng.choice([2, 100, 250, 1000]))
    lens = [int(v) for v in rng.integers(w + 51, w + 9000, 5)] + [w + 51, w + 4096, 13_000 + w]
    xs = [_int_series(rng, l, (seed + i) % 5) for i, l in enumerate(lens)]
    x = np.concatenate(xs).astype(np.float32)
    for sg in SG:
        kw = dict(median_window_size=w, savgol=sg is not None)
        if sg is not None:
            kw.update(savgol_window_size=sg[0], savgol_poly_deg=sg[1])
        for impl in (None, "hist"):
            got, off = adjust_segments(x, lens, impl=impl, **kw)
            got = _np(got)
            for i, xi in enumerate(xs):
                exact_check(got[off[i]: off[i + 1]], xi, w, sg, (seed, i, sg, impl))


# ------------------------------------------------------------------------------------------------------ B4
def test_shard_redoes_flagged_adjust_tiles(dev):
    import torch
    from finaletoolkit_b200 import distributed as FD
    from finaletoolkit_b200.device import AdjustPlan, WpsPlan, adjust_segments
    from finaletoolkit_b200.io.fragments import FragmentTable
    from finaletoolkit_b200.synth import synth_fragments
    sizes = {"a": 61_003, "b": 40_000}
    cols = {}
    for i, (c, n) in enumerate(sizes.items()):
        st, sp, mq, sd = synth_fragments(n, 15_000, i, seed_base=4242)
        if c == "a":   # a 40 000-fold pile-up: |WPS| = 40 000 > kRankMaxAbs
            st = np.concatenate([st, np.full(40_000, 30_000, np.int32)]); sp = np.concatenate([sp, np.full(40_000, 30_160, np.int32)])
            mq = np.concatenate([mq, np.full(40_000, 60, np.uint8)]); sd = np.concatenate([sd, np.ones(40_000, np.uint8)])
            o = np.argsort(st, kind="stable"); st, sp, mq, sd = st[o], sp[o], mq[o], sd[o]
        cols[c] = (st, sp, mq, sd)
    table = FragmentTable(cols)
    sites = FD.tile_genome(list(sizes.items()), 5000)
    adj = dict(median_window_size=1000, savgol=True, savgol_window_size=21, savgol_poly_deg=2)
    res, _, _ = FD.multi_wps_genome(table, list(sizes.items()), sites, 5000, 120, 120, 180, 30, adjust=adj, device=dev,
                                    contigs=list(sizes), sync=False)
    assert any(bool(f.item()) for f in res["a"].flags)              # the rank kernel flagged a tile ...
    res, _, _ = FD.multi_wps_genome(table, list(sizes.items()), sites, 5000, 120, 120, 180, 30, adjust=adj, device=dev,
                                    contigs=list(sizes))
    for c, n in sizes.items():
        s, e = sites[c]
        r = res[c]
        plan = WpsPlan(s, e, n, 180, dev)
        wps = plan.run(table.device(c, dev))
        assert torch.equal(r.wps, wps)
        ap = AdjustPlan(np.diff(plan.offsets), 1000, True, 21, 2, dev, skip_short=True)
        hist, _ = adjust_segments(wps, None, plan=ap, impl="hist", **adj)     # ... and the shard redid it there
        assert torch.equal(r.adjusted, hist), c
        wh, got = _np(wps), _np(r.adjusted)
        if c == "a":
            assert int(np.abs(wh).max()) > 32000
        for i in np.flatnonzero(ap.n_out > 0):
            exact_check(got[ap.out_off[i]: ap.out_off[i + 1]], wh[plan.offsets[i]: plan.offsets[i + 1]], 1000, (21, 2),
                        (c, int(i)))


# ------------------------------------------------------------------------------------------------------ B5
@pytest.mark.parametrize("n_bins", [1024, 2048, 2500])
def test_length_histogram_privatisation_edges(dev, n_bins):
    from finaletoolkit_b200 import device as D
    from finaletoolkit_b200.synth import synth_fragments
    rng = np.random.default_rng(n_bins)
    clen = 200_000
    st, sp, mq, sd = synth_fragments(clen, 40_000, 1, seed_base=8080)
    edges = [1023, 1024, 2047, 2048, n_bins - 1, n_bins, n_bins + 1]
    idx = rng.choice(st.size - 100, 7 * 30, replace=False)
    for k, L in enumerate(edges):
        sel = idx[k * 30: (k + 1) * 30]
        sp[sel] = st[sel] + L
        mq[sel] = 60
    ofr = O.Frags(st, sp, mq, sd)
    fr = D.ContigFragments(st, sp, mq, sd, device=dev)
    starts = np.arange(5000, clen - 10_000, 9000, dtype=np.int64)
    ivs = [(int(a), int(a + 9000)) for a in starts] + [(0, clen), (None, 60_000)]
    s, e = [a for a, _ in ivs], [b for _, b in ivs]
    for pol in ("midpoint", "any"):
        dists = [O.length_dist(ofr, a, b, None, None, pol, 30) for a, b in ivs]
        assert all(any(L in d for d in dists) for L in edges)
        c1, h1, f1 = map(_np, D.interval_hist(fr, s, e, pol, None, None, 30, n_bins=n_bins, first_seen=True))
        for j, d in enumerate(dists):
            exp = {L: v for L, v in d.items() if L < n_bins}
            nz = np.flatnonzero(h1[j])
            got = {int(nz[i]): int(h1[j][nz[i]]) for i in np.argsort(f1[j][nz], kind="stable")}
            assert got == exp and list(got) == list(exp), (pol, ivs[j], n_bins)
            assert int(c1[j]) == sum(d.values())
        c2, h2, f2 = map(_np, D.interval_hist(fr, s, e, pol, None, None, 30, n_bins=n_bins, pooled="hist", first_seen=True))
        assert np.array_equal(c2, c1) and np.array_equal(h2[0], h1.sum(0)) and np.array_equal(f2[0], f1.min(0))
        c3, h3, f3 = map(_np, D.interval_hist(fr, s, e, pol, None, None, 30, n_bins=n_bins, pooled=True, first_seen=True))
        assert int(c3[0]) == int(c1.sum()) and np.array_equal(h3[0], h1.sum(0)) and np.array_equal(f3[0], f1.min(0))
        pooled = O.merge_dists(dists)
        nz = np.flatnonzero(h3[0])
        got = {int(nz[i]): int(h3[0][nz[i]]) for i in np.argsort(f3[0][nz], kind="stable")}
        assert got == {L: v for L, v in pooled.items() if L < n_bins}
    # the fused WPS pass: coverage + pooled histogram of the counted fragments over 5 kb tiles
    tiles = np.arange(0, clen + 5000, 5000).clip(max=clen)
    plan = D.WpsPlan(tiles[:-1], tiles[1:], clen, 180, dev)
    _, cov, h = plan.run_fused(fr, 120, 120, 180, 30, None, None, 30, n_bins=n_bins)
    exp_h = np.zeros(n_bins, np.int64)
    for L, v in O.length_dist(ofr, 0, clen, None, None, "midpoint", 30).items():
        if L < n_bins:
            exp_h[L] += v
    assert np.array_equal(_np(h), exp_h)
    assert all(exp_h[L] for L in edges if L < n_bins)
    assert np.array_equal(_np(cov), O.interval_coverage(ofr, tiles[:-1], tiles[1:], None, None, "midpoint", 30))
