"""CUDA site-centred V-plots (vplot, device.vplot_sites, ftk_vplot_u64) against the numpy definition in
tests/vplot_oracle.py, the interval length-histogram kernel and the BAM fetch semantics."""
import gzip

import numpy as np
import pytest

import vplot_oracle as VO
from test_gpu_api import fx, syn  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

_FILTERS = [(0, 500, 30), (100, 200, 0), (0, 600, 60), (150, 150, 20)]   # (min_length, max_length, q) per seed


def _random_case(seed):
    """A synthetic contig and its sites: mixed '+' / '-' / '.', duplicates, overlapping windows, windows past
    both contig ends and sites without a single candidate fragment."""
    from finaletoolkit_b200.synth import synth_fragments
    rng = np.random.default_rng(90 + seed)
    clen = int(rng.integers(30_000, 90_000)); n = int(rng.integers(100, 40_000))
    st, sp, mq, _ = synth_fragments(clen, n, seed, seed_base=555)
    c = rng.integers(0, clen, 24).tolist()
    c += [c[0], c[0], c[1] + 3, c[1] - 20, 0, 2, clen - 1, clen + 400, -5, clen + 50_000, -50_000]
    flip = (rng.integers(0, 3, len(c)) == 2).tolist()     # a third '-'; '+' and '.' do not flip
    flip[1] = not flip[0]                                 # the duplicated site with both orientations
    return clen, st, sp, mq, c, flip


@pytest.mark.parametrize("flank", [0, 1, 37, 1000])
@pytest.mark.parametrize("seed", range(4))
def test_random_vs_numpy(seed, flank):
    import torch
    from finaletoolkit_b200.device import ContigFragments, vplot_sites
    clen, st, sp, mq, c, flip = _random_case(seed)
    lo, hi, q = _FILTERS[seed]
    fr = ContigFragments(st, sp, mq, device="cuda:0")
    got = vplot_sites(fr, c, flip, flank, lo, hi, q)
    assert got.dtype == torch.int64 and tuple(got.shape) == (hi - lo + 1, 2 * flank + 1)
    exp = VO.vplot(st, sp, mq, c, flip, flank, lo, hi, q)
    assert np.array_equal(got.cpu().numpy(), exp), (seed, flank)
    if flank >= 37:
        assert exp.sum() > 0


SPLITS = (1, 2, 3, 7, 1000)


@pytest.fixture(scope="module")
def slice_data():
    from finaletoolkit_b200 import device as D
    from finaletoolkit_b200.synth import synth_fragments
    clen, n = 400_000, 160_000
    st, sp, mq, _ = synth_fragments(clen, n, 3, seed_base=2024)
    fr = D.ContigFragments(st, sp, mq, device="cuda:0")
    rng = np.random.default_rng(17)
    c = rng.integers(0, clen, 64).tolist() + [0, clen - 1]
    flip = (rng.integers(0, 2, len(c)) == 1).tolist()
    return clen, st, sp, mq, fr, c, flip


@pytest.mark.parametrize("splits", SPLITS)
def test_slices(slice_data, splits, monkeypatch):
    """Candidate ranges start at every residue mod 4; 1000 splits make many slices shorter than a vector or empty."""
    from finaletoolkit_b200 import device as D
    clen, st, sp, mq, fr, c, flip = slice_data
    monkeypatch.setattr(D, "_splits_for", lambda *a, **k: splits)
    for flank, lo, hi, q in [(1000, 0, 600, 30), (73, 120, 180, 0)]:
        reach = min(fr.max_len, hi) >> 1
        assert set(np.searchsorted(st, np.asarray(c) - flank - reach) % 4) == {0, 1, 2, 3}
        got = D.vplot_sites(fr, c, flip, flank, lo, hi, q).cpu().numpy()
        assert np.array_equal(got, VO.vplot(st, sp, mq, c, flip, flank, lo, hi, q)), (splits, flank)


def test_accumulate_empty_and_no_sites(monkeypatch):
    import torch
    from finaletoolkit_b200 import device as D
    clen, st, sp, mq, c, flip = _random_case(0)
    fr = D.ContigFragments(st, sp, mq, device="cuda:0")
    a = D.vplot_sites(fr, c[:10], flip[:10], 100, 0, 400, 30)
    b = D.vplot_sites(fr, c[10:], flip[10:], 100, 0, 400, 30, out=a.clone())
    assert torch.equal(b, D.vplot_sites(fr, c, flip, 100, 0, 400, 30))
    assert np.array_equal(b.cpu().numpy(), VO.vplot(st, sp, mq, c, flip, 100, 0, 400, 30))
    for empty in (D.ContigFragments(st, sp, np.zeros_like(mq), device="cuda:0"),       # every mapq below q
                  D.ContigFragments(st[:0], sp[:0], mq[:0], device="cuda:0")):        # no fragment at all
        z = D.vplot_sites(empty, c, flip, 100, 0, 400, 30)
        assert tuple(z.shape) == (401, 201) and int(z.abs().sum()) == 0
    def no_call():
        raise AssertionError("a launch without sites")
    monkeypatch.setattr(D, "lib", no_call)
    z = D.vplot_sites(fr, [], [], 100, 0, 400, 30, out=a)
    assert z is a and torch.equal(z, D.vplot_sites(fr, np.zeros(0, np.int64), [], 100, 0, 400, 30, out=a.clone()))
    with pytest.raises(ValueError):
        D.vplot_sites(fr, c, flip, 100, 0, 400, 30, out=torch.zeros((401, 200), dtype=torch.int64, device="cuda:0"))


@pytest.mark.parametrize("seed", range(3))
def test_pins_to_interval_hist(seed):
    """A '-' site is the column-reversed '+' site; the row sums of one site are the midpoint length histogram of
    interval_hist (pinned to the reference goldens) over [c - flank, c + flank + 1)."""
    from finaletoolkit_b200.device import ContigFragments, interval_hist, vplot_sites
    clen, st, sp, mq, c, _ = _random_case(seed)
    lo, hi, q = _FILTERS[seed]
    lo = max(lo, 1)   # interval_hist's overlap test drops a zero-length fragment at the window's first base
    fr = ContigFragments(st, sp, mq, device="cuda:0")
    for x, flank in [(c[0], 1000), (c[3], 37), (5, 400), (clen - 3, 250)]:
        plus = vplot_sites(fr, [x], [False], flank, lo, hi, q).cpu().numpy()
        minus = vplot_sites(fr, [x], [True], flank, lo, hi, q).cpu().numpy()
        assert np.array_equal(minus, plus[:, ::-1])
        _, h, _ = interval_hist(fr, [x - flank], [x + flank + 1], "midpoint", lo, hi, q, n_bins=hi + 1)
        assert np.array_equal(plus.sum(axis=1), h[0].cpu().numpy()[lo:]), (seed, x, flank)


# ------------------------------------------------------------------------------------------ public API
def _host(path, contig):
    from finaletoolkit_b200.io.fragments import as_table
    st, sp, mq, _ = as_table(path).host(contig)
    return st, sp, mq


def expected_text(M, flank, min_length):
    out = "length\t" + "\t".join(str(d) for d in range(-flank, flank + 1)) + "\n"
    for j, row in enumerate(M):
        out += f"{min_length + j}\t" + "\t".join(str(int(v)) for v in row) + "\n"
    return out


_FX_SITES = ("# promoter set\ntrack name=sites\nbrowser position 12:34443000-34447000\n\n"
             "12\t34443300\t34443301\t.\t0\t+\n12\t34444000\t34444100\tx\t0\t-\n12\t34445500\t34445502\n"
             "12\t34445500\t34445502\n7\t100\t200\t.\t0\t-\n12\t34446000\t34446000\tname\t0\t.\n")


def test_vplot_api_fx(fx, tmp_path):
    import finaletoolkit_b200 as F
    from click.testing import CliRunner
    from finaletoolkit_b200.cli.main_cli import main_cli
    bed = tmp_path / "fx_sites.bed"; bed.write_text(_FX_SITES)
    sites = [s for s in VO.read_sites(_FX_SITES.splitlines()) if s[0] == "12"]
    assert len(sites) == 5
    st, sp, mq = _host(fx["frag"], "12")
    for kw in [{}, {"quality_threshold": 0}, {"flank": 200, "min_length": 100, "max_length": 300, "quality_threshold": 0},
               {"flank": 0, "min_length": 160, "max_length": 160, "quality_threshold": 0}]:
        full = dict(flank=1000, min_length=0, max_length=500, quality_threshold=30); full.update(kw)
        got = F.vplot(fx["frag"], str(bed), **kw)
        exp = VO.vplot(st, sp, mq, [s[1] for s in sites], [s[2] for s in sites], full["flank"], full["min_length"],
                       full["max_length"], full["quality_threshold"])
        assert got.dtype == np.int64 and np.array_equal(got, exp), kw
        assert exp.sum() > 0 or full["flank"] == 0
    # exact text: .tsv, .tsv.gz and the CLI on stdout
    kw = dict(flank=200, min_length=100, max_length=300, quality_threshold=0)
    M = F.vplot(fx["frag"], str(bed), **kw)
    text = expected_text(M, 200, 100)
    assert M.sum() > 0
    tsv, tgz = str(tmp_path / "v.tsv"), str(tmp_path / "v.tsv.gz")
    assert np.array_equal(F.vplot(fx["frag"], str(bed), output_file=tsv, **kw), M)
    assert open(tsv).read() == text
    F.vplot(fx["frag"], str(bed), output_file=tgz, **kw)
    with gzip.open(tgz, "rt") as fh:
        assert fh.read() == text
    r = CliRunner().invoke(main_cli, ["vplot", fx["frag"], str(bed), "--flank", "200", "--min-length", "100",
                                      "--max-length", "300", "-q", "0"])
    assert r.exit_code == 0, r.output
    assert r.output == text


def test_vplot_api_syn(syn, manifest, tmp_path):
    import finaletoolkit_b200 as F
    sizes = dict(manifest["synth_small"]["contigs"])
    rng = np.random.default_rng(5)
    rows = []
    for c, n in sizes.items():
        for x in rng.integers(0, n, 6).tolist() + [0, n - 1]:
            rows.append(f"{c}\t{x}\t{x + int(rng.integers(0, 40))}\t.\t0\t{'+-.'[int(rng.integers(0, 3))]}\n")
    rows.insert(3, "chrZ\t10\t20\n")   # a contig the input does not hold
    bed = tmp_path / "syn_sites.bed"; bed.write_text("".join(rows))
    sites = VO.read_sites(rows)
    for kw in [{}, {"flank": 300, "min_length": 50, "max_length": 250, "quality_threshold": 0}]:
        full = dict(flank=1000, min_length=0, max_length=500, quality_threshold=30); full.update(kw)
        exp = np.zeros((full["max_length"] - full["min_length"] + 1, 2 * full["flank"] + 1), np.int64)
        for c in sizes:
            sel = [s for s in sites if s[0] == c]
            exp += VO.vplot(*_host(syn["frag"], c), [s[1] for s in sel], [s[2] for s in sel], full["flank"],
                            full["min_length"], full["max_length"], full["quality_threshold"])
        assert np.array_equal(F.vplot(syn["frag"], str(bed), **kw), exp), kw
        assert exp.sum() > 0


def test_vplot_errors(fx, tmp_path):
    import finaletoolkit_b200 as F
    bed = tmp_path / "e.bed"; bed.write_text(_FX_SITES)
    for kw in [{"max_length": None}, {"min_length": None}, {"min_length": -1}, {"min_length": 300, "max_length": 200},
               {"flank": -1}, {"flank": 2 ** 20 + 1}, {"flank": 2 ** 20, "max_length": 600}]:
        with pytest.raises(ValueError):
            F.vplot(fx["frag"], str(bed), **kw)
    with pytest.raises(ValueError):
        F.vplot("-", "-")
    with pytest.raises(ValueError):
        F.vplot(fx["frag"], str(bed), output_file="x.txt")
    with pytest.raises(TypeError):
        F.vplot(fx["frag"], str(bed), output_file=3)
    bad = tmp_path / "bad.bed"
    for text in ("12\t34443300\t34443200\n", "12\t34443300\n"):
        bad.write_text(text)
        with pytest.raises(ValueError):
            F.vplot(fx["frag"], str(bad))


def check_bam(bam):
    """BAM input: the oracle summed over the rows an indexed fetch of each site's window yields."""
    import finaletoolkit_b200 as F
    from finaletoolkit_b200.io.fragments import as_table
    tab = as_table(bam["path"])
    tiles = [ln.split("\t") for ln in bam["m"]["tiles"].splitlines()]
    rows = [f"{t[0]}\t{t[1]}\t{t[2]}\t.\t0\t{'+-'[k % 2]}\n" for k, t in enumerate(tiles[:10])]
    rows += ["chrA\t0\t1\n", "chrA\t480\t12345\t.\t0\t-\n"]
    bed = bam["dir"] / "vplot_sites.bed"; bed.write_text("".join(rows))
    for flank, lo, hi, q in [(300, 0, 600, 0), (1000, 100, 220, 20)]:
        got = F.vplot(bam["path"], str(bed), flank=flank, min_length=lo, max_length=hi, quality_threshold=q)
        exp = np.zeros_like(got)
        for c, x, flip in VO.read_sites(rows):
            st, sp, mq, _ = tab.fetched(c, max(x - flank, 0), x + flank + 1).host(c)
            exp += VO.vplot(st, sp, mq, [x], [flip], flank, lo, hi, q)
        assert np.array_equal(got, exp), (flank, lo, hi, q)
        assert exp.sum() > 0


@pytest.fixture(scope="module")
def bam(tmp_path_factory, golden):
    import bam_replay as R
    from finaletoolkit_b200.io import fragments
    fragments._CACHE.clear()
    yield R.make_fixture(tmp_path_factory.mktemp("vplot_bam"), golden)
    fragments._CACHE.clear()


def test_bam_fetch_semantics(bam):
    check_bam(bam)
