"""GC-corrected counts (gc_corrected_coverage / gc_corrected_profile, device.gc_weighted_intervals /
gc_weighted_sites, ftk_gc_weighted_intervals_f64 / ftk_gc_weighted_sites_f64) against the numpy definition in
tests/gc_correct_oracle.py, cross-pinned to interval_hist, vplot and gc_observed, the model identity, slices and
accumulation, the coordinate ceiling, the public API, the CLI and the BAM fetch semantics."""
import gzip
import math
import warnings

import numpy as np
import pytest

import gc_correct_oracle as CO
import gc_oracle as GO
import test_gpu_gc_bias as G
import vplot_oracle as VO
from test_gpu_coord_ceiling import big_ref, top  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

_FLANKS = [1000, 0, 37, 1, 300]


def _intervals(seed, clen):
    """Overlapping, unsorted and 1-bp intervals, some before 0, past the contig end or unbounded."""
    rng = np.random.default_rng(1200 + seed)
    a = rng.integers(-500, clen, 40)
    b = a + rng.integers(1, 8000, 40)
    s, e = a.tolist(), b.tolist()
    s += [-700, 0, 5, clen - 700, clen + 10, clen - 1, None, clen - 2000, None, s[0], s[1] + 3]
    e += [300, 1, 6, clen + 500, clen + 900, clen, 1000, None, None, e[0], s[1] + 4]
    return s, e


def _sites(seed, clen):
    """Random sites of both strands, several near 0 and near the contig end (and one past it)."""
    rng = np.random.default_rng(1300 + seed)
    c = rng.integers(0, clen, 30).tolist() + [0, 3, 600, clen - 1, clen - 4, clen + 200, 777, 777]
    return c, (rng.random(len(c)) < 0.5).tolist()


def _weights(seed, shape, integer):
    """Small-integer weights (fp64 sums of them are exact in any order) or real ones, both with zeros."""
    rng = np.random.default_rng(1400 + seed)
    w = rng.integers(0, 5, shape).astype(np.float64) if integer else rng.random(shape) * 3.0
    w[rng.random(shape) < 0.1] = 0.0
    return w


def _dev(codes, nm, st, sp, mq):
    from finaletoolkit_b200 import device as D
    return D, D.PackedContig.from_codes(codes, nm, device="cuda:0"), D.ContigFragments(st, sp, mq, device="cuda:0")


def _np(pair):
    return pair[0].cpu().numpy(), pair[1].cpu().numpy()


def _check(got, exp, integer):
    assert got[0].dtype == np.int64 and got[1].dtype == np.float64
    assert np.array_equal(got[0], exp[0])
    if integer:
        assert np.array_equal(got[1], exp[1])
    else:
        assert np.allclose(got[1], exp[1], rtol=1e-12, atol=0)


@pytest.mark.parametrize("seed", range(5))
def test_random_vs_numpy(seed):
    clen, codes, nm, (st, sp, mq), _ = G._case(seed)
    lo, hi, q = G._FILTERS[seed]
    D, ref, fr = _dev(codes, nm, st, sp, mq)
    s, e = _intervals(seed, clen)
    c, f = _sites(seed, clen)
    flank = _FLANKS[seed]
    shape = (hi - lo + 1, hi + 1)
    for integer in (False, True):
        W = _weights(seed, shape, integer)
        exp = CO.intervals(st, sp, mq, codes, nm, clen, s, e, W, lo, hi, q)
        _check(_np(D.gc_weighted_intervals(fr, ref, s, e, W, lo, hi, q)), exp, integer)
        assert exp[0].sum() > 0 and exp[1].sum() > 0
        exp = CO.sites(st, sp, mq, codes, nm, clen, c, f, flank, W, lo, hi, q)
        _check(_np(D.gc_weighted_sites(fr, ref, c, f, flank, W, lo, hi, q)), exp, integer)
        assert exp[0].sum() > 0 and exp[1].sum() > 0


def test_cross_pins():
    """count == interval_hist (midpoint) and == vplot summed over lengths; one-hot weights == gc_observed of that key;
    all-ones weights == the N-free, in-contig selected fragments."""
    clen, codes, nm, (st, sp, mq), _ = G._case(0)
    lo, hi, q = 50, 500, 30
    D, ref, fr = _dev(codes, nm, st, sp, mq)
    s, e = _intervals(0, clen)
    c, f = _sites(0, clen)
    W = _weights(0, (hi - lo + 1, hi + 1), False)
    cnt, _ = _np(D.gc_weighted_intervals(fr, ref, s, e, W, lo, hi, q))
    assert np.array_equal(cnt, D.interval_hist(fr, s, e, "midpoint", lo, hi, q)[0].cpu().numpy())
    pc, _ = _np(D.gc_weighted_sites(fr, ref, c, f, 1000, W, lo, hi, q))
    assert np.array_equal(pc, D.vplot_sites(fr, c, f, 1000, lo, hi, q).sum(dim=0).cpu().numpy())
    # one-hot at the most frequent (L, g) of the contig
    O = D.gc_observed(fr, ref, [0], [clen], lo, hi, q).cpu().numpy()
    i, g = np.unravel_index(int(np.argmax(O)), O.shape)
    one = np.zeros_like(W); one[i, g] = 1.0
    clipped = [(max(a, 0), min(b, clen)) for a, b in zip(s, e) if a is not None and b is not None and min(b, clen) > max(a, 0)]
    _, got = _np(D.gc_weighted_intervals(fr, ref, [a for a, _ in clipped], [b for _, b in clipped], one, lo, hi, q))
    exp = [int(D.gc_observed(fr, ref, [a], [b], lo, hi, q)[i, g]) for a, b in clipped]
    assert np.array_equal(got, np.array(exp, np.float64)) and sum(exp) > 0
    # all ones
    _, got = _np(D.gc_weighted_intervals(fr, ref, s, e, np.ones_like(W), lo, hi, q))
    sel, m, _, defined = CO.fragment_weights(st, sp, mq, codes, nm, clen, W, lo, hi, q)
    exp = [int((sel & defined & (m >= (-2 ** 62 if a is None else a)) & (m < (2 ** 62 if b is None else b))).sum())
           for a, b in zip(s, e)]
    assert np.array_equal(got, np.array(exp, np.float64)) and sum(exp) > 0


@pytest.mark.parametrize("lo,hi,q", [(50, 500, 30), (1, 64, 0)])
def test_model_identity(lo, hi, q):
    """Corrected total of the region the model was fitted on == sum_L sum(O_L) * sum_{g: O > 0} E[L, g] / sum(E_L)."""
    clen, codes, nm, (st, sp, mq), _ = G._case(3)
    D, ref, fr = _dev(codes, nm, st, sp, mq)
    a, b = 1000, clen - 1000
    O = D.gc_observed(fr, ref, [a], [b], lo, hi, q).cpu().numpy()
    E = D.gc_expected(ref, [a], [b], lo, hi).cpu().numpy()
    _, got = _np(D.gc_weighted_intervals(fr, ref, [a], [b], CO.weights(GO.ratio(O, E)), lo, hi, q))
    so, se = O.sum(axis=1), E.sum(axis=1)
    exp = math.fsum(so[i] * math.fsum(E[i, O[i] > 0].tolist()) / se[i] for i in range(O.shape[0]) if so[i] > 0)
    assert exp > 0 and abs(float(got[0]) - exp) <= 1e-12 * exp


@pytest.mark.parametrize("splits", [1, 2, 7, 1000])
def test_splits_accumulation_and_mirror(splits, monkeypatch):
    import torch
    clen, codes, nm, (st, sp, mq), _ = G._case(1)
    lo, hi, q = 20, 300, 30
    D, ref, fr = _dev(codes, nm, st, sp, mq)
    monkeypatch.setattr(D, "_splits_for", lambda *a, **k: splits)
    s, e = _intervals(1, clen)
    c, f = _sites(1, clen)
    shape = (hi - lo + 1, hi + 1)
    Wr, Wi = _weights(1, shape, False), _weights(1, shape, True)
    a = D.gc_weighted_intervals(fr, ref, s, e, Wr, lo, hi, q)
    _check(_np(a), CO.intervals(st, sp, mq, codes, nm, clen, s, e, Wr, lo, hi, q), False)
    b = D.gc_weighted_intervals(fr, ref, s, e, Wr, lo, hi, q)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1].view(torch.int64), b[1].view(torch.int64))   # bit-identical
    _check(_np(D.gc_weighted_sites(fr, ref, c, f, 300, Wr, lo, hi, q)),
           CO.sites(st, sp, mq, codes, nm, clen, c, f, 300, Wr, lo, hi, q), False)
    # out=: the two halves of the fragment table into one pair of outputs
    k = st.size // 2
    h1 = D.ContigFragments(st[:k], sp[:k], mq[:k], device="cuda:0")
    h2 = D.ContigFragments(st[k:], sp[k:], mq[k:], device="cuda:0")
    acc = D.gc_weighted_intervals(h1, ref, s, e, Wi, lo, hi, q)
    r = D.gc_weighted_intervals(h2, ref, s, e, Wi, lo, hi, q, out=acc)
    assert r[0] is acc[0] and r[1] is acc[1]
    _check(_np(acc), CO.intervals(st, sp, mq, codes, nm, clen, s, e, Wi, lo, hi, q), True)
    acc = D.gc_weighted_sites(h1, ref, c, f, 300, Wi, lo, hi, q)
    D.gc_weighted_sites(h2, ref, c, f, 300, Wi, lo, hi, q, out=acc)
    _check(_np(acc), CO.sites(st, sp, mq, codes, nm, clen, c, f, 300, Wi, lo, hi, q), True)
    # a '-' site is the '+' profile reversed
    plus = _np(D.gc_weighted_sites(fr, ref, c, [False] * len(c), 300, Wi, lo, hi, q))
    minus = _np(D.gc_weighted_sites(fr, ref, c, [True] * len(c), 300, Wi, lo, hi, q))
    assert np.array_equal(minus[0], plus[0][::-1]) and np.array_equal(minus[1], plus[1][::-1]) and plus[1].sum() > 0
    if splits == 1:
        for bad in (np.zeros((3, 3)), np.full(shape, np.nan), np.full(shape, -1.0), np.full(shape, np.inf)):
            with pytest.raises(ValueError):
                D.gc_weighted_intervals(fr, ref, s, e, bad, lo, hi, q)
            with pytest.raises(ValueError):
                D.gc_weighted_sites(fr, ref, c, f, 300, bad, lo, hi, q)
        for bad in [(0, 10), (10, 9), (1, 1025)]:
            with pytest.raises(ValueError):
                D.gc_weighted_intervals(fr, ref, s, e, np.zeros((2, 2)), *bad)
        with pytest.raises(ValueError):
            D.gc_weighted_sites(fr, ref, c, f, 2 ** 20 + 1, Wi, lo, hi, q)

        def no_call():
            raise AssertionError("a launch without units")
        monkeypatch.setattr(D, "lib", no_call)
        assert [x.numel() for x in D.gc_weighted_intervals(fr, ref, [], [], Wi, lo, hi, q)] == [0, 0]
        got = _np(D.gc_weighted_sites(fr, ref, [], [], 5, Wi, lo, hi, q))
        assert got[0].shape == (11,) and not got[0].any() and not got[1].any()


def test_coordinate_ceiling(top, big_ref):
    """Intervals and sites reaching 2^31 - 1 on the translated reference: the oracle of the untranslated contig."""
    D, B, T = top["D"], top["B"], top["T"]
    s = [5000, 100_000, T - 5000, T - 2, T - 300, T - 1]
    e = [60_000, 150_000, T, T, None, None]
    c = [50_000, T - 1000, T - 10, T - 1]
    f = [False, True, False, True]
    sh = lambda v: None if v is None else v + B   # noqa: E731
    for lo, hi, q in [(50, 500, 30), (1, 1024, 0)]:
        W = _weights(7, (hi - lo + 1, hi + 1), True)
        got = _np(D.gc_weighted_intervals(top["frB"], big_ref, [sh(v) for v in s], [sh(v) for v in e], W, lo, hi, q))
        exp = CO.intervals(top["st"], top["sp"], top["mq"], top["codes"], top["nm"], T, s, e, W, lo, hi, q)
        _check(got, exp, True)
        assert exp[0][2:].sum() > 0 and exp[1][2:].sum() > 0
        got = _np(D.gc_weighted_sites(top["frB"], big_ref, [v + B for v in c], f, 1000, W, lo, hi, q))
        exp = CO.sites(top["st"], top["sp"], top["mq"], top["codes"], top["nm"], T, c, f, 1000, W, lo, hi, q)
        _check(got, exp, True)
        assert exp[1].sum() > 0


# ------------------------------------------------------------------------------------------ public API
_IVL_BED = ("# intervals\ntrack name=i\n\nchrM1\t100\t5000\tfirst\nchrM1\t4000\t9000\nchrM1\t9000\t9001\tone\n"
            "chrZ\t5\t10\tmissing\nchrM2\t0\t1\nchrM2\t30\t200000\twide\nchrM1\t2500\t2600\nchrQ\t1\t2\n")
_SITE_BED = ("chrM1\t5000\t5001\t.\t0\t+\nchrM1\t9000\t9100\t.\t0\t-\nchrZ\t5\t10\nchrM2\t0\t1\t.\t0\t-\n"
             "chrM2\t150000\t150000\nchrM1\t20\t30\t.\t0\t+\n")


def _api_expected(cols, seqs, model, q, flank):
    """Oracle coverage rows and profile of the two BEDs under ``model``."""
    W = CO.weights(model.ratio)
    lo, hi = model.min_length, model.max_length
    rows = []
    for ln in _IVL_BED.splitlines():
        if not ln.strip() or ln.startswith(("#", "track", "browser")):
            continue
        p = ln.split("\t")
        c, a, b, name = p[0], int(p[1]), int(p[2]), p[3] if len(p) > 3 else "."
        if c in seqs:
            codes, nm = seqs[c]
            k, w = CO.intervals(*cols[c][:3], codes, nm, len(codes), [a], [b], W, lo, hi, q)
            rows.append((c, a, b, name, int(k[0]), float(w[0])))
        else:
            rows.append((c, a, b, name, 0, 0.0))
    count, corr = np.zeros(2 * flank + 1, np.int64), np.zeros(2 * flank + 1)
    sites = VO.read_sites(_SITE_BED.splitlines(keepends=True))
    for c in seqs:
        sel = [x for x in sites if x[0] == c]
        codes, nm = seqs[c]
        k, w = CO.sites(*cols[c][:3], codes, nm, len(codes), [x[1] for x in sel], [x[2] for x in sel], flank, W,
                        lo, hi, q)
        count += k; corr += w
    return rows, count, corr, sum(1 for x in sites if x[0] in seqs)


def _rows(res):
    return [tuple(r) for r in res]


def test_api_models_text_and_cli(tmp_path, manifest, golden):
    import finaletoolkit_b200 as F
    from click.testing import CliRunner
    from finaletoolkit_b200.cli.main_cli import main_cli
    frag, tb, seqs, cols = G.motif_files(tmp_path, manifest, golden)
    ivl, sb = tmp_path / "i.bed", tmp_path / "s.bed"
    ivl.write_text(_IVL_BED); sb.write_text(_SITE_BED)
    lo, hi, q, flank = 100, 220, 20, 300
    model = F.gc_bias(frag, tb, min_length=lo, max_length=hi, quality_threshold=q)
    model_tsv = str(tmp_path / "model.tsv")
    F.gc_bias(frag, tb, output_file=model_tsv, min_length=lo, max_length=hi, quality_threshold=q)
    rows, count, corr, n_sites = _api_expected(cols, seqs, model, q, flank)
    assert sum(r[4] for r in rows) > 0 and corr.sum() > 0
    results = []
    for gcb, extra in ((model, {}), (model_tsv, {}), (None, dict(min_length=lo, max_length=hi))):
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            r = F.gc_corrected_coverage(frag, tb, str(ivl), gc_bias=gcb, quality_threshold=q, **extra)
            p = F.gc_corrected_profile(frag, tb, str(sb), flank=flank, gc_bias=gcb, quality_threshold=q, **extra)
        assert [str(x.message) for x in w if issubclass(x.category, UserWarning)] == [
            "gc_corrected_coverage: intervals on contigs that the input or the reference lacks count 0: chrZ, chrQ",
            "gc_corrected_profile: sites on contigs that the input or the reference lacks count 0: chrZ"]
        assert all(isinstance(x, F.GCCoverageResult) for x in r)
        got = _rows(r)
        assert [x[:5] for x in got] == [x[:5] for x in rows]
        assert np.allclose([x[5] for x in got], [x[5] for x in rows], rtol=1e-12, atol=0)
        assert isinstance(p, F.GCSiteProfile) and (p.flank, p.n_sites) == (flank, n_sites)
        assert np.array_equal(p.count, count) and np.allclose(p.corrected, corr, rtol=1e-12, atol=0)
        results.append(got)
    assert results[0] == results[1] == results[2]   # the same model three ways: identical output
    # text: .tsv, .tsv.gz and the CLI on stdout
    text = CO.coverage_text(results[0])
    tsv, tgz = str(tmp_path / "c.tsv"), str(tmp_path / "c.tsv.gz")
    F.gc_corrected_coverage(frag, tb, str(ivl), output_file=tsv, gc_bias=model, quality_threshold=q)
    assert open(tsv).read() == text
    F.gc_corrected_coverage(frag, tb, str(ivl), output_file=tgz, gc_bias=model, quality_threshold=q)
    with gzip.open(tgz, "rt") as fh:
        assert fh.read() == text
    res = CliRunner().invoke(main_cli, ["gc-corrected-coverage", frag, tb, str(ivl), "--gc-bias", model_tsv, "-q", "20"])
    assert res.exit_code == 0, res.output
    assert res.output == text
    p = F.gc_corrected_profile(frag, tb, str(sb), output_file=str(tmp_path / "p.tsv.gz"), flank=flank, gc_bias=model,
                               quality_threshold=q)
    with gzip.open(tmp_path / "p.tsv.gz", "rt") as fh:
        assert fh.read() == CO.profile_text(p.count, p.corrected, flank)
    res = CliRunner().invoke(main_cli, ["gc-corrected-profile", frag, tb, str(sb), "--gc-bias", model_tsv, "-q", "20",
                                        "--flank", str(flank)])
    assert res.exit_code == 0, res.output
    lines = res.output.splitlines()
    assert lines[0] == "offset\tcount\tcorrected" and len(lines) == 2 * flank + 2
    cli = np.array([[float(v) for v in ln.split("\t")] for ln in lines[1:]])
    assert np.array_equal(cli[:, 0], np.arange(-flank, flank + 1)) and np.array_equal(cli[:, 1], count)
    assert np.allclose(cli[:, 2], corr, rtol=1e-12, atol=0)


def test_api_errors(tmp_path, manifest, golden):
    import finaletoolkit_b200 as F
    frag, tb, _, _ = G.motif_files(tmp_path, manifest, golden)
    ivl, sb = tmp_path / "i.bed", tmp_path / "s.bed"
    ivl.write_text(_IVL_BED); sb.write_text(_SITE_BED)
    model = F.gc_bias(frag, tb, min_length=100, max_length=220, quality_threshold=20)
    for fn, bed in ((F.gc_corrected_coverage, ivl), (F.gc_corrected_profile, sb)):
        with pytest.raises(ValueError):
            fn(frag, tb, str(bed), output_file="x.txt", gc_bias=model)
        with pytest.raises(TypeError):
            fn(frag, tb, str(bed), output_file=3, gc_bias=model)
        for kw in [{"min_length": 99}, {"max_length": 221}, {"gc_regions": str(ivl)}]:
            with pytest.raises(ValueError):
                fn(frag, tb, str(bed), gc_bias=model, **kw)
        with pytest.raises(TypeError):
            fn(frag, tb, str(bed), gc_bias=3)
        with pytest.raises(ValueError):
            fn(frag, tb, str(bed), min_length=0, max_length=10)          # fitting rejects the lengths
        bad = tmp_path / "bad.tsv"
        bad.write_text("length\tgc\tobserved\texpected\tratio\n5\t0\t1\t1\t1.0\n")
        with pytest.raises(ValueError):
            fn(frag, tb, str(bed), gc_bias=str(bad))
    for flank in (-1, 2 ** 20 + 1, 2.5):
        with pytest.raises(ValueError):
            F.gc_corrected_profile(frag, tb, str(sb), flank=flank, gc_bias=model)
    with pytest.raises(ValueError):
        F.gc_corrected_profile("-", tb, "-", gc_bias=model)
    for text in ("chrM1\t500\t400\n", "chrM1\t500\n"):
        (tmp_path / "b.bed").write_text(text)
        with pytest.raises(ValueError):
            F.gc_corrected_profile(frag, tb, str(tmp_path / "b.bed"), gc_bias=model)


def check_bam(bam):
    """BAM input: each interval's and each site's fragments are the rows an indexed fetch of it yields."""
    import finaletoolkit_b200 as F
    from finaletoolkit_b200.io.fragments import as_table
    from finaletoolkit_b200.io.reference import open_reference
    tab = as_table(bam["path"])
    ref = open_reference(bam["tb"])
    tiles = [ln.split("\t") for ln in bam["m"]["tiles"].splitlines()]
    rows = [(t[0], int(t[1]), int(t[2])) for t in tiles[::3]] + [("chrA", 0, 1), ("chrA", 480, 12345)]
    bed = bam["dir"] / "gcc_intervals.bed"; bed.write_text("".join(f"{c}\t{a}\t{b}\n" for c, a, b in rows))
    srows = [f"{t[0]}\t{t[1]}\t{t[2]}\t.\t0\t{'+-'[k % 2]}\n" for k, t in enumerate(tiles[:10])]
    srows += ["chrA\t0\t1\n", "chrA\t480\t12345\t.\t0\t-\n"]
    sbed = bam["dir"] / "gcc_sites.bed"; sbed.write_text("".join(srows))
    for lo, hi, q, flank in [(50, 600, 0, 300), (100, 220, 20, 1000)]:
        model = F.gc_bias(bam["path"], bam["tb"], min_length=lo, max_length=hi, quality_threshold=q)
        W = CO.weights(model.ratio)
        got = F.gc_corrected_coverage(bam["path"], bam["tb"], str(bed), gc_bias=model, quality_threshold=q)
        for r, (c, a, b) in zip(got, rows):
            codes, nm = ref.contig_arrays(c)
            st, sp, mq, _ = tab.fetched(c, a, b).host(c)
            k, w = CO.intervals(st, sp, mq, codes, nm, ref.chroms[c], [a], [b], W, lo, hi, q)
            assert r.count == k[0] and math.isclose(r.corrected, w[0], rel_tol=1e-12, abs_tol=0), (r, lo, hi, q)
        assert sum(r.count for r in got) > 0 and sum(r.corrected for r in got) > 0
        p = F.gc_corrected_profile(bam["path"], bam["tb"], str(sbed), flank=flank, gc_bias=model, quality_threshold=q)
        count, corr = np.zeros(2 * flank + 1, np.int64), np.zeros(2 * flank + 1)
        for c, x, flip in VO.read_sites(srows):
            codes, nm = ref.contig_arrays(c)
            st, sp, mq, _ = tab.fetched(c, max(x - flank, 0), x + flank + 1).host(c)
            k, w = CO.sites(st, sp, mq, codes, nm, ref.chroms[c], [x], [flip], flank, W, lo, hi, q)
            count += k; corr += w
        assert np.array_equal(p.count, count) and np.allclose(p.corrected, corr, rtol=1e-12, atol=0)
        assert count.sum() > 0 and corr.sum() > 0


@pytest.fixture(scope="module")
def bam(tmp_path_factory, golden):
    import bam_replay as R
    from finaletoolkit_b200.io import fragments
    fragments._CACHE.clear()
    yield R.make_fixture(tmp_path_factory.mktemp("gcc_bam"), golden)
    fragments._CACHE.clear()


def test_bam_fetch_semantics(bam):
    check_bam(bam)
