"""CUDA orientation-aware fragment end profiles (ocf, device.ocf_sites, ftk_ocf_u64) against the numpy definition
in tests/ocf_oracle.py, the V-plot kernel, the BAM fetch semantics, the int32 coordinate ceiling, a side stream and
a device that is not the current one."""
import gzip
import math

import numpy as np
import pytest

import ocf_oracle as OO
import vplot_oracle as VO
from test_gpu_api import fx, syn  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

# (min_length, max_length, q) per seed: bounded, unbounded, only a lower bound, one length
_FILTERS = [(0, 500, 30), (None, None, 0), (100, None, 60), (150, 150, 20)]
N_SETS = 4   # set 3 has no site on the contig


def _random_case(seed):
    """A synthetic contig and its sites: mixed '+' / '-' / '.', duplicates, overlapping windows, windows past both
    contig ends, negative centres, sites without a single candidate fragment, three sets and an empty fourth."""
    from finaletoolkit_b200.synth import synth_fragments
    rng = np.random.default_rng(190 + seed)
    clen = int(rng.integers(30_000, 90_000)); n = int(rng.integers(100, 40_000))
    st, sp, mq, _ = synth_fragments(clen, n, seed, seed_base=655)
    c = rng.integers(0, clen, 24).tolist()
    c += [c[0], c[0], c[1] + 3, c[1] - 20, 0, 2, clen - 1, clen + 400, -5, clen + 50_000, -50_000]
    flip = (rng.integers(0, 3, len(c)) == 2).tolist()     # a third '-'; '+' and '.' do not flip
    flip[1] = not flip[0]                                 # the duplicated site with both orientations
    sets = rng.integers(0, N_SETS - 1, len(c)).tolist()
    return clen, st, sp, mq, c, flip, sets


@pytest.mark.parametrize("flank", [0, 1, 37, 1000])
@pytest.mark.parametrize("seed", range(4))
def test_random_vs_numpy(seed, flank):
    import torch
    from finaletoolkit_b200.device import ContigFragments, ocf_sites
    clen, st, sp, mq, c, flip, sets = _random_case(seed)
    lo, hi, q = _FILTERS[seed]
    fr = ContigFragments(st, sp, mq, device="cuda:0")
    got = ocf_sites(fr, c, flip, sets, N_SETS, flank, lo, hi, q)
    assert got.dtype == torch.int64 and tuple(got.shape) == (N_SETS, 2, 2 * flank + 1)
    exp = OO.ends(st, sp, mq, c, flip, sets, N_SETS, flank, lo, hi, q)
    assert np.array_equal(got.cpu().numpy(), exp), (seed, flank)
    assert not exp[N_SETS - 1].any()
    if flank >= 37:
        assert exp[:, 0].sum() > 0 and exp[:, 1].sum() > 0


SPLITS = (1, 2, 3, 7, 1000)


@pytest.fixture(scope="module")
def slice_data():
    from finaletoolkit_b200 import device as D
    from finaletoolkit_b200.synth import synth_fragments
    clen, n = 400_000, 160_000
    st, sp, mq, _ = synth_fragments(clen, n, 3, seed_base=2025)
    fr = D.ContigFragments(st, sp, mq, device="cuda:0")
    rng = np.random.default_rng(18)
    c = rng.integers(0, clen, 64).tolist() + [0, clen - 1]
    flip = (rng.integers(0, 2, len(c)) == 1).tolist()
    sets = rng.integers(0, 3, len(c)).tolist()
    return clen, st, sp, mq, fr, c, flip, sets


@pytest.mark.parametrize("splits", SPLITS)
def test_slices(slice_data, splits, monkeypatch):
    """Candidate ranges start at every residue mod 4; 1000 splits make many slices shorter than a vector or empty."""
    from finaletoolkit_b200 import device as D
    clen, st, sp, mq, fr, c, flip, sets = slice_data
    monkeypatch.setattr(D, "_splits_for", lambda *a, **k: splits)
    for flank, lo, hi, q in [(1000, None, None, 30), (73, 120, 180, 0)]:
        reach = min(fr.max_len, hi or fr.max_len)
        assert set(np.searchsorted(st, np.asarray(c) - flank - reach) % 4) == {0, 1, 2, 3}
        got = D.ocf_sites(fr, c, flip, sets, 3, flank, lo, hi, q).cpu().numpy()
        assert np.array_equal(got, OO.ends(st, sp, mq, c, flip, sets, 3, flank, lo, hi, q)), (splits, flank)


@pytest.mark.parametrize("threshold", [1, 5, 1000, 30_000])
def test_flush_path(slice_data, threshold, monkeypatch):
    """A small flush threshold makes every CTA add its counters to the output many times (1 and 5: rounds larger
    than the threshold, run one warp at a time); the result is the same."""
    from finaletoolkit_b200 import device as D
    clen, st, sp, mq, fr, c, flip, sets = slice_data
    plain = D.ocf_sites(fr, c, flip, sets, 3, 500, None, None, 0).cpu().numpy()
    monkeypatch.setattr(D, "OCF_FLUSH_CANDIDATES", threshold)
    for splits in (1, 7):
        monkeypatch.setattr(D, "_splits_for", lambda *a, **k: splits)
        got = D.ocf_sites(fr, c, flip, sets, 3, 500, None, None, 0).cpu().numpy()
        assert np.array_equal(got, plain), (threshold, splits)
    assert np.array_equal(plain, OO.ends(st, sp, mq, c, flip, sets, 3, 500, None, None, 0))


def test_accumulate_empty_and_no_sites(monkeypatch):
    import torch
    from finaletoolkit_b200 import device as D
    clen, st, sp, mq, c, flip, sets = _random_case(0)
    fr = D.ContigFragments(st, sp, mq, device="cuda:0")
    a = D.ocf_sites(fr, c[:10], flip[:10], sets[:10], N_SETS, 100, 0, 400, 30)
    b = D.ocf_sites(fr, c[10:], flip[10:], sets[10:], N_SETS, 100, 0, 400, 30, out=a.clone())
    assert torch.equal(b, D.ocf_sites(fr, c, flip, sets, N_SETS, 100, 0, 400, 30))
    assert np.array_equal(b.cpu().numpy(), OO.ends(st, sp, mq, c, flip, sets, N_SETS, 100, 0, 400, 30))
    for empty in (D.ContigFragments(st, sp, np.zeros_like(mq), device="cuda:0"),       # every mapq below q
                  D.ContigFragments(st[:0], sp[:0], mq[:0], device="cuda:0")):        # no fragment at all
        z = D.ocf_sites(empty, c, flip, sets, N_SETS, 100, 0, 400, 30)
        assert tuple(z.shape) == (N_SETS, 2, 201) and int(z.abs().sum()) == 0

    def no_call():
        raise AssertionError("a launch without sites")
    monkeypatch.setattr(D, "lib", no_call)
    z = D.ocf_sites(fr, [], [], [], N_SETS, 100, 0, 400, 30, out=a)
    assert z is a
    for bad in ((N_SETS, 2, 200), (N_SETS, 401), (N_SETS - 1, 2, 201)):
        with pytest.raises(ValueError):
            D.ocf_sites(fr, c, flip, sets, N_SETS, 100, 0, 400, 30, out=torch.zeros(bad, dtype=torch.int64, device="cuda:0"))
    with pytest.raises(ValueError):
        D.ocf_sites(fr, c, flip, sets, N_SETS, 100, 0, 400, 30, out=torch.zeros((N_SETS, 2, 201), device="cuda:0"))
    for kw in ({"n_sets": 0}, {"flank": -1}, {"flank": 8193}, {"min_length": -1}, {"min_length": 300, "max_length": 200}):
        args = dict(n_sets=N_SETS, flank=100, min_length=0, max_length=400); args.update(kw)
        with pytest.raises(ValueError):
            D.ocf_sites(fr, c, flip, sets, **args)
    with pytest.raises(ValueError):
        D.ocf_sites(fr, c, flip, [N_SETS] * len(c), N_SETS, 100)       # a set out of range
    with pytest.raises(ValueError):
        D.ocf_sites(fr, c, flip[:-1], sets, N_SETS, 100)               # lengths differ


@pytest.mark.parametrize("seed", range(3))
def test_pins_to_vplot(seed):
    """For one fragment length L and an unflipped site, the U row is the V-plot row of L shifted by L // 2 and the D
    row the same row shifted by -(L - 1 - L // 2), read from a V-plot of flank G = F + L."""
    from finaletoolkit_b200.device import ContigFragments, ocf_sites, vplot_sites
    clen, st, sp, mq, c, _, _ = _random_case(seed)
    fr = ContigFragments(st, sp, mq, device="cuda:0")
    L_all = (sp.astype(np.int64) - st)
    lengths = [int(np.bincount(L_all).argmax()), 1, 2, 147] if L_all.max() >= 147 else [int(np.bincount(L_all).argmax())]
    for x, F in [(c[0], 1000), (c[3], 37), (5, 400), (clen - 3, 250)]:
        for L in lengths:
            got = ocf_sites(fr, [x], [False], [0], 1, F, L, L, 0).cpu().numpy()[0]
            G = F + L
            V = vplot_sites(fr, [x], [False], G, L, L, 0).cpu().numpy()[0]
            off = np.arange(-F, F + 1)
            assert np.array_equal(got[0], V[off + L // 2 + G]), (seed, x, F, L)
            assert np.array_equal(got[1], V[off - (L - 1 - L // 2) + G]), (seed, x, F, L)
    assert any(ocf_sites(fr, [c[0]], [False], [0], 1, 1000, lengths[0], lengths[0], 0).cpu().numpy().ravel())


def test_flip_invariance():
    from finaletoolkit_b200.device import ContigFragments, ocf_sites
    from finaletoolkit_b200.frag._ocf import ocf_values
    clen, st, sp, mq, c, flip, sets = _random_case(1)
    fr = ContigFragments(st, sp, mq, device="cuda:0")
    a = ocf_sites(fr, c, flip, sets, N_SETS, 300, None, None, 0).cpu().numpy()
    b = ocf_sites(fr, c, [not f for f in flip], sets, N_SETS, 300, None, None, 0).cpu().numpy()
    assert np.array_equal(b[:, 0], a[:, 1, ::-1]) and np.array_equal(b[:, 1], a[:, 0, ::-1])
    va, vb = ocf_values(a, 300, 60, 20), ocf_values(b, 300, 60, 20)
    assert np.array_equal(va[:3], vb[:3]) and math.isnan(va[3]) and math.isnan(vb[3])
    for k in range(3):
        assert va[k] == OO.ocf_value(a[k, 0], a[k, 1], 300)


def test_phased_nucleosomes_give_a_positive_ocf():
    """Fragments [c + a, c + a + 147) and [c - a - 147, c - a) (a nucleosome each side of an open site) put U at +a
    and D at -a - 1: a positive OCF for a near 60, of either sign of strand; background alone gives about 0."""
    from finaletoolkit_b200.device import ContigFragments, ocf_sites
    from finaletoolkit_b200.frag._ocf import ocf_values
    rng = np.random.default_rng(7)
    centres = np.arange(10_000, 200_000, 10_000)
    starts, stops = [], []
    for x in centres:
        a = rng.integers(52, 68, 40)
        starts += (x + a).tolist() + (x - a - 147).tolist()
        stops += (x + a + 147).tolist() + (x - a).tolist()
    bg = rng.integers(0, 210_000, 4000)
    starts += bg.tolist(); stops += (bg + rng.integers(100, 250, bg.size)).tolist()
    order = np.argsort(starts, kind="stable")
    st = np.asarray(starts, np.int32)[order]; sp = np.asarray(stops, np.int32)[order]
    mq = np.full(st.size, 60, np.uint8)
    fr = ContigFragments(st, sp, mq, device="cuda:0")
    flips = (np.arange(centres.size) % 2).astype(bool)
    got = ocf_sites(fr, centres, flips, [0] * centres.size, 1, 1000).cpu().numpy()
    assert np.array_equal(got, OO.ends(st, sp, mq, centres, flips, [0] * centres.size, 1, 1000))
    v = ocf_values(got, 1000, 60, 20)[0]
    assert v > 10 and v == OO.ocf_value(got[0, 0], got[0, 1], 1000)
    shifted = ocf_sites(fr, centres + 5000, flips, [0] * centres.size, 1, 1000).cpu().numpy()
    assert abs(ocf_values(shifted, 1000, 60, 20)[0]) < v / 4


# ------------------------------------------------------------------------------------------ public API
def _host(path, contig):
    from finaletoolkit_b200.io.fragments import as_table
    st, sp, mq, _ = as_table(path).host(contig)
    return st, sp, mq


def expected_texts(labels, n_sites, counts, flank, peak_offset=60, peak_width=20):
    """The summary and profile text, from the oracle's counts."""
    summary = "set\tsites\tends\tocf\n"
    prof = "set\tend\t" + "\t".join(str(x) for x in range(-flank, flank + 1)) + "\n"
    for k, label in enumerate(labels):
        v = OO.ocf_value(counts[k, 0], counts[k, 1], flank, peak_offset, peak_width)
        summary += f"{label}\t{n_sites[k]}\t{int(counts[k].sum())}\t{v!r}\n"
        for j, end in enumerate("UD"):
            prof += f"{label}\t{end}\t" + "\t".join(str(int(x)) for x in counts[k, j]) + "\n"
    return summary, prof


_FX_SITES = ("# promoter set\ntrack name=sites\nbrowser position 12:34443000-34447000\n\n"
             "12\t34443300\t34443301\t.\t0\t+\n12\t34444000\t34444100\tx\t0\t-\n12\t34445500\t34445502\n"
             "12\t34445500\t34445502\n7\t100\t200\t.\t0\t-\n12\t34446000\t34446000\tname\t0\t.\n")
_FX_SITES_B = "12\t34444300\t34444400\tp1\t0\t+\n12\t34445000\t34445001\tp2\t0\t-\nchrZ\t10\t20\tp3\n"


def _fx_expected(fx, beds, kw):
    from finaletoolkit_b200.io.fragments import as_table
    full = dict(flank=1000, min_length=None, max_length=None, quality_threshold=30, peak_offset=60, peak_width=20)
    full.update(kw)
    held = set(as_table(fx["frag"]).contigs)
    st, sp, mq = _host(fx["frag"], "12")
    counts = np.zeros((len(beds), 2, 2 * full["flank"] + 1), np.int64)
    n_sites = []
    for k, text in enumerate(beds):
        sites = VO.read_sites(text.splitlines())
        n_sites.append(sum(s[0] in held for s in sites))
        on12 = [s for s in sites if s[0] == "12"]
        counts[k] = OO.ends(st, sp, mq, [s[1] for s in on12], [s[2] for s in on12], [0] * len(on12), 1,
                            full["flank"], full["min_length"], full["max_length"], full["quality_threshold"])[0]
    return counts, n_sites, full


def test_ocf_api_fx(fx, tmp_path):
    import finaletoolkit_b200 as F
    from click.testing import CliRunner
    from finaletoolkit_b200.cli.main_cli import main_cli
    a = tmp_path / "promoters.bed"; a.write_text(_FX_SITES)
    b = tmp_path / "liver_ocr"; b.write_text(_FX_SITES_B)            # no .bed suffix: the label is the whole name
    for kw in [{}, {"quality_threshold": 0}, {"flank": 200, "min_length": 100, "max_length": 300, "quality_threshold": 0},
               {"flank": 100, "min_length": 120, "max_length": 200, "quality_threshold": 0, "peak_offset": 30,
                "peak_width": 7}]:
        got = F.ocf(fx["frag"], [str(a), str(b)], **kw)
        counts, n_sites, full = _fx_expected(fx, [_FX_SITES, _FX_SITES_B], kw)
        assert got.labels == ["promoters", "liver_ocr"]
        assert got.n_sites.dtype == np.int64 and got.n_sites.tolist() == n_sites
        assert got.upstream.dtype == np.int64 and np.array_equal(got.upstream, counts[:, 0]), kw
        assert np.array_equal(got.downstream, counts[:, 1]), kw
        assert (got.flank, got.peak_offset, got.peak_width) == (full["flank"], full["peak_offset"], full["peak_width"])
        assert got.ocf.dtype == np.float64
        for k in range(2):
            exp = OO.ocf_value(counts[k, 0], counts[k, 1], full["flank"], full["peak_offset"], full["peak_width"])
            assert got.ocf[k] == exp or (math.isnan(got.ocf[k]) and math.isnan(exp)), (kw, k)
        assert counts.sum() > 0
    one = F.ocf(fx["frag"], str(a), quality_threshold=0)                 # a single path
    assert one.labels == ["promoters"] and np.array_equal(one.upstream, F.ocf(fx["frag"], [a], quality_threshold=0).upstream)
    # exact text: .tsv, .tsv.gz and the CLI on stdout
    kw = dict(flank=200, min_length=100, max_length=300, quality_threshold=0)
    counts, n_sites, _ = _fx_expected(fx, [_FX_SITES, _FX_SITES_B], kw)
    summary, prof = expected_texts(["promoters", "liver_ocr"], n_sites, counts, 200)
    tsv, tgz = str(tmp_path / "o.tsv"), str(tmp_path / "p.tsv.gz")
    F.ocf(fx["frag"], [str(a), str(b)], output_file=tsv, profile_file=tgz, **kw)
    assert open(tsv).read() == summary
    with gzip.open(tgz, "rt") as fh:
        assert fh.read() == prof
    F.ocf(fx["frag"], [str(a), str(b)], output_file=tgz, profile_file=tsv, **kw)
    assert open(tsv).read() == prof
    with gzip.open(tgz, "rt") as fh:
        assert fh.read() == summary
    args = ["ocf", fx["frag"], str(a), str(b), "--flank", "200", "--min-length", "100", "--max-length", "300", "-q", "0"]
    r = CliRunner().invoke(main_cli, args)
    assert r.exit_code == 0, r.output
    assert r.output == summary
    r = CliRunner().invoke(main_cli, args + ["-o", tsv, "--profiles", "-"])
    assert r.exit_code == 0, r.output
    assert r.output == prof and open(tsv).read() == summary
    empty = tmp_path / "nothing_here.bed"; empty.write_text("chrZ\t10\t20\n")
    res = F.ocf(fx["frag"], [str(empty)], output_file=tsv)
    assert res.n_sites.tolist() == [0] and not res.upstream.any() and math.isnan(res.ocf[0])
    assert open(tsv).read() == "set\tsites\tends\tocf\nnothing_here\t0\t0\tnan\n"


def test_ocf_api_syn(syn, manifest, tmp_path):
    import finaletoolkit_b200 as F
    sizes = dict(manifest["synth_small"]["contigs"])
    rng = np.random.default_rng(6)
    texts = []
    for k in range(3):
        rows = []
        for c, n in sizes.items():
            for x in rng.integers(0, n, 5).tolist() + [0, n - 1]:
                rows.append(f"{c}\t{x}\t{x + int(rng.integers(0, 40))}\tpeak{k}\t0\t{'+-.'[int(rng.integers(0, 3))]}\n")
        rows.insert(2, "chrZ\t10\t20\n")   # a contig the input does not hold
        texts.append("".join(rows))
    beds = []
    for k, text in enumerate(texts):
        p = tmp_path / f"tissue{k}.bed"; p.write_text(text); beds.append(str(p))
    for kw in [{}, {"flank": 300, "min_length": 50, "max_length": 250, "quality_threshold": 0}]:
        full = dict(flank=1000, min_length=None, max_length=None, quality_threshold=30); full.update(kw)
        exp = np.zeros((3, 2, 2 * full["flank"] + 1), np.int64)
        for k, text in enumerate(texts):
            sites = VO.read_sites(text.splitlines())
            for c in sizes:
                sel = [s for s in sites if s[0] == c]
                exp[k] += OO.ends(*_host(syn["frag"], c), [s[1] for s in sel], [s[2] for s in sel], [0] * len(sel), 1,
                                  full["flank"], full["min_length"], full["max_length"], full["quality_threshold"])[0]
        got = F.ocf(syn["frag"], beds, **kw)
        assert got.labels == ["tissue0", "tissue1", "tissue2"] and got.n_sites.tolist() == [7 * len(sizes)] * 3
        assert np.array_equal(got.upstream, exp[:, 0]) and np.array_equal(got.downstream, exp[:, 1]), kw
        assert exp.sum() > 0


def test_ocf_errors(fx, tmp_path):
    import finaletoolkit_b200 as F
    bed = tmp_path / "e.bed"; bed.write_text(_FX_SITES)
    for kw in [{"flank": -1}, {"flank": 8193}, {"peak_width": 0}, {"peak_offset": 10, "peak_width": 20},
               {"peak_offset": 60, "peak_width": 20, "flank": 68}, {"peak_offset": 1.5}, {"min_length": -1},
               {"min_length": 300, "max_length": 200}]:
        with pytest.raises(ValueError):
            F.ocf(fx["frag"], str(bed), **kw)
    F.ocf(fx["frag"], str(bed), flank=69)                                   # P+ = [50, 69] just fits
    F.ocf(fx["frag"], str(bed), peak_offset=1, peak_width=1, flank=1)       # P+ = [1, 1]
    other = tmp_path / "sub"; other.mkdir(); (other / "e.bed").write_text(_FX_SITES)
    for beds in ([str(bed), str(other / "e.bed")], [str(bed), "-"], ["-", "-"], []):
        with pytest.raises(ValueError):
            F.ocf(fx["frag"], beds)
    with pytest.raises(ValueError):
        F.ocf("-", "-")
    for kw in ({"output_file": "x.txt"}, {"profile_file": "x.bed"}, {"output_file": "-", "profile_file": "-"}):
        with pytest.raises(ValueError):
            F.ocf(fx["frag"], str(bed), **kw)
    for kw in ({"output_file": 3}, {"profile_file": 3}):
        with pytest.raises(TypeError):
            F.ocf(fx["frag"], str(bed), **kw)
    bad = tmp_path / "bad.bed"
    for text in ("12\t34443300\t34443200\n", "12\t34443300\n"):
        bad.write_text(text)
        with pytest.raises(ValueError):
            F.ocf(fx["frag"], [str(bed), str(bad)])


def check_bam(bam):
    """BAM input: the oracle summed over the rows an indexed fetch of each site's window yields."""
    import finaletoolkit_b200 as F
    from finaletoolkit_b200.io.fragments import as_table
    tab = as_table(bam["path"])
    tiles = [ln.split("\t") for ln in bam["m"]["tiles"].splitlines()]
    texts = ["".join(f"{t[0]}\t{t[1]}\t{t[2]}\t.\t0\t{'+-'[k % 2]}\n" for k, t in enumerate(tiles[j:10:2]))
             for j in range(2)]
    texts[1] += "chrA\t0\t1\nchrA\t480\t12345\t.\t0\t-\n"
    beds = []
    for k, text in enumerate(texts):
        p = bam["dir"] / f"ocf_sites{k}.bed"; p.write_text(text); beds.append(str(p))
    for flank, lo, hi, q in [(300, None, None, 0), (1000, 100, 220, 20)]:
        got = F.ocf(bam["path"], beds, flank=flank, min_length=lo, max_length=hi, quality_threshold=q)
        exp = np.zeros((2, 2, 2 * flank + 1), np.int64)
        for k, text in enumerate(texts):
            for c, x, flip in VO.read_sites(text.splitlines()):
                st, sp, mq, _ = tab.fetched(c, max(x - flank, 0), x + flank + 1).host(c)
                exp[k] += OO.ends(st, sp, mq, [x], [flip], [0], 1, flank, lo, hi, q)[0]
        assert np.array_equal(got.upstream, exp[:, 0]) and np.array_equal(got.downstream, exp[:, 1]), (flank, lo, hi, q)
        assert exp.sum() > 0


@pytest.fixture(scope="module")
def bam(tmp_path_factory, golden):
    import bam_replay as R
    from finaletoolkit_b200.io import fragments
    fragments._CACHE.clear()
    yield R.make_fixture(tmp_path_factory.mktemp("ocf_bam"), golden)
    fragments._CACHE.clear()


def test_bam_fetch_semantics(bam):
    check_bam(bam)


# ------------------------------------------------------------------------------- int32 coordinate ceiling
@pytest.mark.parametrize("flank,lo,hi", [(1000, None, None), (37, 120, 180), (0, 1, 3000)])
def test_windows_reaching_the_ceiling(flank, lo, hi):
    """Fragments ending at 2^31 - 1 (and a 300-fold pile-up there) with sites whose windows reach or pass it."""
    from finaletoolkit_b200 import device as D
    from finaletoolkit_b200.synth import synth_fragments
    top = 2 ** 31 - 1
    rng = np.random.default_rng(2032)
    st, sp, mq, _ = (a.astype(np.int64) for a in synth_fragments(200_000, 30_000, 0, seed_base=7732))
    B = top - 200_400
    st += B; sp += B
    hand_st = np.array([top - 170, top, top - 1, top - 2500] + [top - 167] * 300, np.int64)
    hand_sp = np.full(hand_st.size, top, np.int64)
    st = np.concatenate([st, hand_st]); sp = np.minimum(np.concatenate([sp, hand_sp]), top)
    mq = np.concatenate([mq, np.full(hand_st.size, 60, np.uint8)])
    order = np.argsort(st, kind="stable")
    st, sp, mq = st[order], sp[order], mq[order]
    assert int(sp.max()) == top
    fr = D.ContigFragments(st.astype(np.int32), sp.astype(np.int32), mq, device="cuda:0")
    c = np.array([top, top - 3, top - flank, top - max(flank - 1, 0), top - 2 * flank - 1, B + 100_000, top - 500,
                  top - 100], np.int64)
    flip = (np.arange(c.size) % 2).astype(bool)
    sets = (np.arange(c.size) % 3).tolist()
    got = D.ocf_sites(fr, c, flip, sets, 3, flank, lo, hi, 30).cpu().numpy()
    exp = OO.ends(st, sp, mq, c, flip, sets, 3, flank, lo, hi, 30)
    assert np.array_equal(got, exp), (flank, lo, hi)
    assert exp.sum() > 0
    with pytest.raises(ValueError, match="int32"):
        D.ocf_sites(fr, np.array([top + 1]), [False], [0], 1, flank)


# ------------------------------------------------------------------ a side stream and a non-current device
# A compact copy of the decoy method of test_gpu_streams_devices.py: the mapq column holds zeros (the decoy) until
# the real values are copied in on the op's own stream; a launch that escapes that stream reads the decoy.
SLEEP_CYCLES = 1 << 26
HOLD_CYCLES = 1 << 29


def _stream_case(dev):
    import torch
    from finaletoolkit_b200 import device as D
    from finaletoolkit_b200.synth import synth_fragments
    st, sp, mq, _ = synth_fragments(200_000, 40_000, 0, seed_base=6161)
    mq_real = torch.from_numpy(mq).to(dev)
    mq_buf = torch.zeros_like(mq_real)
    fr = D.ContigFragments(torch.from_numpy(st).to(dev), torch.from_numpy(sp).to(dev), mq_buf, device=dev,
                           max_len=int((sp.astype(np.int64) - st).max()))
    assert fr.mapq is mq_buf
    c = np.array([5000, 31_337, 100_000, 100_001, 150_500, 199_990], np.int64)
    flip = (np.arange(c.size) % 2).astype(bool)
    sets = [0, 1, 0, 1, 1, 0]
    exp = OO.ends(st, sp, mq, c, flip, sets, 2, 500, 100, 220, 30)
    assert exp.sum() > 0
    return mq_buf, mq_real, lambda: D.ocf_sites(fr, c, flip, sets, 2, 500, 100, 220, 30), exp


def test_side_stream():
    import torch
    dev = torch.device("cuda", 0)
    buf, real, op, exp = _stream_case(dev)
    decoy = buf.clone()
    buf.copy_(real)
    assert np.array_equal(op().cpu().numpy(), exp)      # loads the kernel: a lazy module load waits for the device
    buf.copy_(decoy)
    torch.cuda.synchronize()
    torch.cuda._sleep(SLEEP_CYCLES + HOLD_CYCLES)        # the default stream: whatever lands there waits,
    buf.copy_(decoy)                                     # then finds the decoy back in the buffer
    side = torch.cuda.Stream(dev)
    with torch.cuda.stream(side):
        torch.cuda._sleep(SLEEP_CYCLES)
        buf.copy_(real)
        res = op()
    side.synchronize()
    assert np.array_equal(res.cpu().numpy(), exp)
    torch.cuda.synchronize()


@pytest.mark.skipif(not __import__("torch").cuda.is_available() or __import__("torch").cuda.device_count() < 2,
                    reason="needs two CUDA devices")
def test_non_current_device():
    import torch
    dev = torch.device("cuda", 1)
    with torch.cuda.device(0):
        buf, real, op, exp = _stream_case(dev)
        buf.copy_(real)
        res = op()
        assert torch.cuda.current_device() == 0
    torch.cuda.synchronize(dev)
    assert res.device == dev
    assert np.array_equal(res.cpu().numpy(), exp)
