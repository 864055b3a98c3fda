"""WPS periodograms (wps_spectrum, distributed.wps_spectrum_genome, device.spectrum_segments, ftk_spectrum_i32_f64 /
ftk_spectrum_f64_f64) against the numpy direct sum in tests/spectrum_oracle.py: series lengths and value limits,
constant and analytic series, period limits, determinism and batch independence, cross-pins to the WPS, adjust and
genome paths, the coordinate ceiling, the public API, the CLI and the BAM fetch semantics."""
import gzip
import io
import warnings
from contextlib import redirect_stderr

import numpy as np
import pytest

import spectrum_oracle as SO
from test_gpu_coord_ceiling import top  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu

I32 = 2 ** 31 - 1


def _D():
    from finaletoolkit_b200 import device as D
    return D


def _batch(series, dtype):
    """The series back to back as one CUDA tensor + host offsets."""
    import torch
    off = np.zeros(len(series) + 1, np.int64)
    np.cumsum([len(s) for s in series], out=off[1:])
    x = np.concatenate([np.asarray(s) for s in series]) if series else np.zeros(0)
    return torch.from_numpy(x.astype(dtype)).cuda(), off


def _series(P=193):
    rng = np.random.default_rng(9)
    lengths = [1, 2, P - 1, P, P + 1, 10_000, 100_003]
    small = [rng.integers(-400, 400, n) for n in lengths]
    huge = [rng.choice([-I32, I32], n) if k % 2 else rng.integers(-I32, I32, n, endpoint=True)
            for k, n in enumerate(lengths)]
    return small + huge + [np.zeros(0, np.int64), np.full(5000, I32), np.full(777, -I32), np.full(300, -7)]


@pytest.mark.parametrize("lo,hi", [(120, 280), (193, 193), (2, 40), (1000, 1024)])
def test_int32_vs_direct_sum(lo, hi):
    import torch
    D = _D()
    series = _series()
    x, off = _batch(series, np.int32)
    got = D.spectrum_segments(x, off, lo, hi).cpu().numpy()
    assert got.shape == (len(series), hi - lo + 1) and got.dtype == np.float64
    for k, s in enumerate(series):
        SO.check_row(got[k], s, lo, hi)
    for k in range(len(series) - 3, len(series)):
        assert (got[k] == 0).all()                                   # constant series: exactly 0
    again = D.spectrum_segments(x, off, lo, hi)
    assert torch.equal(again.view(torch.int64).cpu(), torch.from_numpy(got).view(torch.int64))   # bit-identical
    for k, s in enumerate(series):                                   # alone == inside the batch, bit for bit
        xa, oa = _batch([s], np.int32)
        alone = D.spectrum_segments(xa, oa, lo, hi).cpu().numpy()
        assert np.array_equal(alone[0].view(np.int64), got[k].view(np.int64)), k


def test_full_period_range():
    D = _D()
    rng = np.random.default_rng(4)
    series = [rng.integers(-300, 300, 5000), rng.normal(size=3001) * 50.0, rng.integers(-I32, I32, 1500)]
    for k, s in enumerate(series):
        x, off = _batch([s], np.float64 if k == 1 else np.int32)
        SO.check_row(D.spectrum_segments(x, off, 2, 1024).cpu().numpy()[0], s, 2, 1024)


def test_float64_vs_direct_sum():
    D = _D()
    rng = np.random.default_rng(11)
    series = [rng.normal(size=n) * 10.0 ** rng.integers(-3, 6) for n in (1, 2, 192, 193, 194, 10_000, 120_001)]
    series += [np.zeros(0), np.full(4000, 3.5), rng.normal(size=7) + 1e6]
    x, off = _batch(series, np.float64)
    for lo, hi in [(120, 280), (2, 2), (1024, 1024)]:
        got = D.spectrum_segments(x, off, lo, hi).cpu().numpy()
        for k, s in enumerate(series):
            SO.check_row(got[k], s, lo, hi)
        assert (got[len(series) - 2] == 0).all()
        for k, s in enumerate(series):
            xa, oa = _batch([s], np.float64)
            alone = D.spectrum_segments(xa, oa, lo, hi).cpu().numpy()[0]
            assert np.array_equal(alone.view(np.int64), got[k].view(np.int64))


def test_analytic_cosine():
    D = _D()
    for A, k in [(1000.0, 50), (3.0, 7), (25.0, 600)]:
        N = 193 * k
        x, off = _batch([A * np.cos(2 * np.pi * np.arange(N) / 193)], np.float64)
        got = D.spectrum_segments(x, off, 120, 280).cpu().numpy()[0]
        assert abs(got[193 - 120] - A * A * N / 4) <= 1e-9 * A * A * N / 4
        SO.check_row(got, x.cpu().numpy(), 120, 280)
        if k >= 50:   # over a few repeats the folds at 192 and 194 still add almost in phase: no clear peak yet
            assert int(np.argmax(got)) == 193 - 120


def test_spectrum_segments_errors(monkeypatch):
    import torch
    D = _D()
    x, off = _batch([np.arange(500)], np.int32)
    for lo, hi in [(1, 10), (10, 9), (2, 1025), (2.5, 10), (True, 10), (None, 10)]:
        with pytest.raises(ValueError):
            D.spectrum_segments(x, off, lo, hi)
    for bad in (x.cpu(), x.to(torch.float32), x.to(torch.int64)):
        with pytest.raises(ValueError):
            D.spectrum_segments(bad, off, 120, 280)
    for bad_off in ([0, 501], [-1, 500], [0, 300, 200], []):
        with pytest.raises(ValueError):
            D.spectrum_segments(x, bad_off, 120, 280)
    with pytest.raises(ValueError):
        D.spectrum_segments(x, off, 120, 280, out=torch.empty((1, 160), dtype=torch.float64, device="cuda"))
    out = torch.empty((1, 161), dtype=torch.float64, device="cuda")
    assert D.spectrum_segments(x, off, 120, 280, out=out) is out

    def no_call():
        raise AssertionError("a launch without segments")
    monkeypatch.setattr(D, "lib", no_call)
    assert tuple(D.spectrum_segments(x, [0], 120, 280).shape) == (0, 161)


def _wps_rows(D, frags, s, e, size, **kw):
    plan = D.WpsPlan(s, e, size, kw.get("max_length", 180), frags.device)
    return plan.run(frags, **kw), plan.offsets


_KW = dict(window_size=120, min_length=120, max_length=180, quality_threshold=30)


def test_wps_and_adjust_cross_pins(top):
    """Raw and adjusted WPS of windows reaching 2^31 - 1 on the translated contig: the oracle of the scores the
    untranslated WPS / adjust path produces."""
    from oracle import oracle as O
    D, B, T = top["D"], top["B"], top["T"]
    s = np.array([5000, 20_000, T - 10_000, T - 3000, T - 1015, 150_000], np.int64)
    e = np.array([15_000, 140_000, T, T - 1, T, 150_000], np.int64)
    exp, eoff = O.wps_intervals(top["ofr"], s, e, T, 120, 120, 180, 30)
    x, off = _wps_rows(D, top["frB"], s + B, e + B, B + T, **_KW)
    assert np.array_equal(off, eoff) and np.array_equal(x.cpu().numpy().astype(np.int64), exp)
    got = D.spectrum_segments(x, off, 120, 280).cpu().numpy()
    for k in range(len(s)):
        SO.check_row(got[k], exp[eoff[k]: eoff[k + 1]], 120, 280)
    aplan = D.AdjustPlan(np.diff(off), 1000, True, 21, 2, x.device, skip_short=True)
    adj, aoff = D.adjust_segments(x, None, plan=aplan)
    assert list(np.diff(aoff)) == [9000, 119_000, 9000, 1999, 0, 0]
    got = D.spectrum_segments(adj, aoff, 120, 280).cpu().numpy()
    host = adj.cpu().numpy()
    for k in range(len(s)):
        SO.check_row(got[k], host[aoff[k]: aoff[k + 1]], 120, 280)
    assert np.isnan(got[4]).all() and np.isnan(got[5]).all()


def test_genome_driver():
    import torch
    from finaletoolkit_b200 import device as D
    from finaletoolkit_b200.distributed import adjust_wps_genome, multi_wps_genome, wps_spectrum_genome
    from finaletoolkit_b200.io.fragments import FragmentTable
    from finaletoolkit_b200.synth import synth_fragments
    clen = 400_000
    st, sp, mq, sd = synth_fragments(clen, 80_000, 0, seed_base=4242)
    h = st.size // 3
    table = FragmentTable({"a": (st, sp, mq, sd), "b": (st[:h], sp[:h], mq[:h], sd[:h])})
    sites = {"a": (np.array([0, 10_000, 50_000, 300_000]), np.array([10_000, 30_000, 51_010, 399_000])),
             "b": (np.array([1000, 200_000]), np.array([9000, 205_000]))}
    chrom_sizes = [("a", clen), ("b", clen)]
    for adjust in (None, dict(median_window_size=1000)):
        res, _, _ = multi_wps_genome(table, chrom_sizes, sites, adjust=adjust, contigs=["a", "b"], reduce=False)
        spec = wps_spectrum_genome(res, 150, 260)
        for c, r in res.items():
            x, off = (r.wps, r.offsets) if adjust is None else (r.adjusted, r.adj_offsets)
            ref = D.spectrum_segments(x, off, 150, 260)
            assert torch.equal(spec[c].view(torch.int64), ref.view(torch.int64))
            host = x.cpu().numpy()
            for k in range(len(off) - 1):
                SO.check_row(spec[c][k].cpu().numpy(), host[off[k]: off[k + 1]], 150, 260)
        if adjust is not None:
            assert np.isnan(spec["a"][2].cpu().numpy()).all()      # 1010 positions: too short for the filters
    # adjust_wps_genome on raw results, then the spectra of its series
    res, _, _ = multi_wps_genome(table, chrom_sizes, sites, contigs=["a", "b"], reduce=False)
    adjust_wps_genome(res, median_window_size=1000)
    spec = wps_spectrum_genome(res)
    for c, r in res.items():
        assert torch.equal(spec[c].view(torch.int64), D.spectrum_segments(r.adjusted, r.adj_offsets).view(torch.int64))
    with pytest.raises(ValueError):
        wps_spectrum_genome(res, 1, 10)


# ------------------------------------------------------------------------------------------ public API
_BED = ("# windows\ntrack name=w\n\nchrM1\t100\t10100\tg1\nchrM1\t5000\t25000\tg2\nchrM2\t85000\t95000\tclip\n"
        "chrZ\t5\t5000\tmissing\nchrM1\t-500\t4000\tneg\nchrM1\t300000\t420001\tlong\nchrM1\t9000\t10010\tshort\n"
        "chrM1\t700\t700\tempty\nchrM2\t0\t1\tone\nchrM1\t2000\t12000\n")


def api_files(tmp_path, manifest, golden):
    import test_gpu_gc_bias as G
    frag, _, _, cols = G.motif_files(tmp_path, manifest, golden)
    sizes = dict(manifest["motif"]["contigs"])
    cs = tmp_path / "m.chrom.sizes"; cs.write_text("".join(f"{c}\t{n}\n" for c, n in sizes.items()))
    bed = tmp_path / "w.bed"; bed.write_text(_BED)
    return frag, str(cs), str(bed), sizes


def expected_rows(frag, sizes, adjust, lo=120, hi=280, wkw=None):
    """(n, series) per BED row: the scores of the `wps` API for the clipped window, adjusted on the GPU."""
    import finaletoolkit_b200 as F
    from finaletoolkit_b200 import device as D
    wkw = wkw or {}
    out = []
    for ln in _BED.splitlines():
        if not ln.strip() or ln.startswith(("#", "track")):
            continue
        p = ln.split("\t")
        c, a, b = p[0], max(int(p[1]), 0), min(int(p[2]), sizes.get(p[0], 0))
        if b <= a:
            out.append(np.zeros(0))
            continue
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            x = F.wps(frag, c, a, b, sizes[c], **wkw)["wps"]
        if adjust:
            import torch
            xd = torch.from_numpy(x.astype(np.int32)).to(D.require_cuda())
            aplan = D.AdjustPlan([x.size], 1000, True, 21, 2, xd.device, skip_short=True)
            x = D.adjust_segments(xd, [x.size], plan=aplan)[0].cpu().numpy() if aplan.n_total else np.zeros(0)
        out.append(x)
    return out


def test_api_text_and_cli(tmp_path, manifest, golden):
    import finaletoolkit_b200 as F
    from click.testing import CliRunner
    from finaletoolkit_b200.cli.main_cli import main_cli
    frag, cs, bed, sizes = api_files(tmp_path, manifest, golden)
    for adjust in (False, True):
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            res = F.wps_spectrum(frag, bed, cs, adjust=adjust)
        assert [str(x.message) for x in w if issubclass(x.category, UserWarning)] == [
            "wps_spectrum: rows on contigs missing from the chromosome sizes are NaN: chrZ"]
        assert isinstance(res, F.WpsSpectrum) and np.array_equal(res.periods, np.arange(120, 281))
        assert [iv[3] for iv in res.intervals] == ["g1", "g2", "clip", "missing", "neg", "long", "short", "empty",
                                                   "one", "."]
        exp = expected_rows(frag, sizes, adjust)
        assert list(res.n) == [len(x) for x in exp]
        assert res.intensity.shape == (10, 161) and res.intensity.dtype == np.float64
        for row, x in zip(res.intensity, exp):
            SO.check_row(row, x, 120, 280)
        assert np.nansum(res.intensity) > 0
    assert list(res.n) == [9000, 19000, 4000, 0, 3000, 119_001, 0, 0, 0, 9000]
    text = SO.text(res.intervals, res.n, res.periods, res.intensity)
    tsv, tgz = str(tmp_path / "s.tsv"), str(tmp_path / "s.tsv.gz")
    assert np.array_equal(F.wps_spectrum(frag, bed, cs, output_file=tsv).intensity, res.intensity, equal_nan=True)
    assert open(tsv).read() == text
    F.wps_spectrum(frag, bed, cs, output_file=tgz)
    with gzip.open(tgz, "rt") as fh:
        assert fh.read() == text
    out = CliRunner().invoke(main_cli, ["wps-spectrum", frag, bed, "--chrom-sizes", cs])
    assert out.exit_code == 0, out.output
    assert out.output == text
    # other periods, filters and WPS settings reach the kernels
    kw = dict(min_period=150, max_period=230, savgol=False, median_window_size=500, window_size=60, min_length=100,
              max_length=200, quality_threshold=20)
    res = F.wps_spectrum(frag, bed, cs, adjust=False, **kw)
    exp = expected_rows(frag, sizes, False, wkw=dict(window_size=60, min_length=100, max_length=200,
                                                      quality_threshold=20))
    for row, x in zip(res.intensity, exp):
        SO.check_row(row, x, 150, 230)
    out = CliRunner().invoke(main_cli, ["wps-spectrum", frag, bed, "--chrom-sizes", cs, "--no-adjust", "--min-period",
                                        "150", "--max-period", "230", "-W", "60", "--min-length", "100",
                                        "--max-length", "200", "-q", "20"])
    assert out.exit_code == 0 and out.output == SO.text(res.intervals, res.n, res.periods, res.intensity)
    res = F.wps_spectrum(frag, bed, cs, **kw)
    assert list(res.n) == [9500, 19500, 4500, 0, 3500, 119_501, 510, 0, 0, 9500]


def test_api_errors(tmp_path, manifest, golden):
    import finaletoolkit_b200 as F
    frag, cs, bed, _ = api_files(tmp_path, manifest, golden)
    for kw in [dict(min_period=1), dict(max_period=1025), dict(min_period=200, max_period=199), dict(min_period=2.5),
               dict(output_file="x.txt"), dict(median_window_size=999), dict(median_window_size=0),
               dict(savgol_window_size=20), dict(savgol_poly_deg=21), dict(min_length=100, fraction_low=100)]:
        with pytest.raises(ValueError):
            F.wps_spectrum(frag, bed, cs, **kw)
    with pytest.raises(TypeError):
        F.wps_spectrum(frag, bed, cs, output_file=3)
    with pytest.raises(ValueError):
        F.wps_spectrum(frag, bed)                      # a fragment file needs chromosome sizes
    with pytest.raises(ValueError):
        F.wps_spectrum("-", "-", cs)
    F.wps_spectrum(frag, bed, cs, median_window_size=999, adjust=False)   # the filters apply only with adjust


def check_bam(bam):
    """BAM input: each window's scores are those multi_wps computes for it (an indexed fetch of its padded window)."""
    import finaletoolkit_b200 as F
    tiles = [ln.split("\t") for ln in bam["m"]["tiles"].splitlines()]
    # the 1-kb tiles that do not overlap: multi_wps with interval_size=1000 keeps them as they are
    rows = sorted({(t[0], int(t[1]), int(t[2])) for t in tiles if int(t[2]) - int(t[1]) == 1000 and int(t[1]) % 1000 == 0})
    assert len(rows) > 40
    sites = bam["dir"] / "spec_sites.bed"
    sites.write_text("".join(f"{c}\t{a}\t{b}\n" for c, a, b in rows))
    out = str(bam["dir"] / "spec_mw.bed.gz")
    kw = dict(min_length=100, max_length=220)
    with redirect_stderr(io.StringIO()):
        F.multi_wps(bam["path"], str(sites), chrom_sizes=bam["cs"], output_file=out, interval_size=1000, **kw)
    with gzip.open(out, "rt") as fh:
        score = {(p[0], int(p[1])): int(p[3]) for p in (ln.split("\t") for ln in fh.read().splitlines())}
    res = F.wps_spectrum(bam["path"], str(sites), adjust=False, min_period=100, max_period=300, **kw)
    assert list(res.n) == [b - a for _, a, b in rows]
    for row, (c, a, b) in zip(res.intensity, rows):
        SO.check_row(row, [score[(c, p)] for p in range(a, b)], 100, 300)
    assert np.nansum(res.intensity) > 0
    # and the same fetch rule with the adjusted series of longer windows
    big = [(c, 0, n) for c, n in bam["sizes"].items()]
    (bam["dir"] / "spec_big.bed").write_text("".join(f"{c}\t{a}\t{b}\n" for c, a, b in big))
    res = F.wps_spectrum(bam["path"], str(bam["dir"] / "spec_big.bed"), chrom_sizes=bam["cs"], **kw)
    assert list(res.n) == [n - 1000 for _, _, n in big] and np.isfinite(res.intensity).all()


@pytest.fixture(scope="module")
def bam(tmp_path_factory, golden):
    import bam_replay as R
    from finaletoolkit_b200.io import fragments
    fragments._CACHE.clear()
    yield R.make_fixture(tmp_path_factory.mktemp("spec_bam"), golden)
    fragments._CACHE.clear()


def test_bam_fetch_semantics(bam):
    check_bam(bam)
