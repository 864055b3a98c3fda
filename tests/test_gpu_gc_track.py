"""GC-corrected per-base depth tracks (gc_corrected_coverage_profile / multi_gc_corrected_coverage_profile,
device.gc_depth_intervals, ftk_gc_depth_tiles_f64) against the exact numpy definition in tests/gc_track_oracle.py,
cross-pinned to depth_intervals and gc_weighted_intervals, with determinism, batching, the overflow flag, the
coordinate ceiling, a side stream, a second device, the public API, the CLI and the BAM fetch semantics."""
import warnings

import numpy as np
import pytest

import gc_correct_oracle as CO
import gc_track_oracle as TO
import test_gpu_gc_bias as G
from test_gpu_coord_ceiling import big_ref, top  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu


def _intervals(seed, clen):
    """1-bp ones, both contig ends, ones shorter than a tile, ones spanning many tiles, random ones."""
    rng = np.random.default_rng(2100 + seed)
    ivs = [(0, clen), (0, 1), (clen - 1, clen), (100, 5219), (100, 5220), (7, 20_500), (5119, 5121),
           (clen - 700, clen)]
    ivs += [(int(s), int(min(s + rng.integers(1, 12_000), clen))) for s in rng.integers(0, clen - 1, 8)]
    return [a for a, _ in ivs], [b for _, b in ivs]


def _weights(seed, shape):
    """Real weights around 1 with zeros, a few large ones and a few below 2^-32 (quantised to 0 or 1)."""
    rng = np.random.default_rng(2200 + seed)
    w = rng.random(shape) * 3.0
    w[rng.random(shape) < 0.1] = 0.0
    w[rng.random(shape) < 0.01] = 1e3
    w[rng.random(shape) < 0.01] = 2.0 ** -33 * 3
    return w


def _dev(codes, nm, st, sp, mq):
    from finaletoolkit_b200 import device as D
    return D, D.PackedContig.from_codes(codes, nm, device="cuda:0"), D.ContigFragments(st, sp, mq, device="cuda:0")


@pytest.mark.parametrize("midpoint", [False, True])
@pytest.mark.parametrize("seed", range(4))
def test_random_vs_numpy(seed, midpoint):
    import torch
    clen, codes, nm, (st, sp, mq), _ = G._case(seed)
    lo, hi, q = G._FILTERS[seed]
    D, ref, fr = _dev(codes, nm, st, sp, mq)
    s, e = _intervals(seed, clen)
    W = _weights(seed, (hi - lo + 1, hi + 1))
    out, off = D.gc_depth_intervals(fr, ref, s, e, clen, W, lo, hi, q, midpoint)
    assert out.dtype == torch.float64
    exp, eoff = TO.track_intervals(st, sp, mq, codes, nm, clen, s, e, W, lo, hi, q, midpoint)
    assert np.array_equal(off, eoff)
    got = out.cpu().numpy()
    assert np.array_equal(got.view(np.int64), exp.view(np.int64)), (seed, midpoint)   # bit for bit
    assert (exp != 0).sum() > 100 and (exp == 0).sum() > 0


def test_cross_pins():
    """All-ones weights == depth_intervals on fragments with a defined placement (both modes); dyadic weights: the
    midpoint track summed over an interval == gc_weighted_intervals' corrected sum."""
    clen, codes, nm, (st, sp, mq), _ = G._case(0)
    lo, hi, q = 50, 500, 30
    shape = (hi - lo + 1, hi + 1)
    _, _, _, defined = CO.fragment_weights(st, sp, mq, codes, nm, clen, np.ones((1200, 1201)), 0, 1199, 0)
    D, ref, fr = _dev(codes, nm, st[defined], sp[defined], mq[defined])
    s, e = _intervals(0, clen)
    for midpoint in (False, True):
        got, off = D.gc_depth_intervals(fr, ref, s, e, clen, np.ones(shape), lo, hi, q, midpoint)
        dep, off2 = D.depth_intervals(fr, s, e, clen, lo, hi, q, midpoint)
        assert np.array_equal(off, off2) and int(dep.sum()) > 0
        assert np.array_equal(got.cpu().numpy(), dep.cpu().numpy().astype(np.float64)), midpoint
    rng = np.random.default_rng(5)
    Wd = rng.integers(0, 4096, shape) * 2.0 ** -10
    D, ref, fr = _dev(codes, nm, st, sp, mq)
    track, off = D.gc_depth_intervals(fr, ref, s, e, clen, Wd, lo, hi, q, True)
    track = track.cpu().numpy()
    _, corr = D.gc_weighted_intervals(fr, ref, s, e, Wd, lo, hi, q)
    sums = [float(track[off[k]: off[k + 1]].sum()) for k in range(len(s))]
    assert sums == corr.cpu().numpy().tolist() and sum(sums) > 0


def test_determinism_and_batching():
    """Two runs are bitwise equal; one launch over all intervals == one launch per interval."""
    import torch
    clen, codes, nm, (st, sp, mq), _ = G._case(1)
    lo, hi, q = 1, 64, 0
    D, ref, fr = _dev(codes, nm, st, sp, mq)
    s, e = _intervals(1, clen)
    W = _weights(1, (hi - lo + 1, hi + 1))
    for midpoint in (False, True):
        a, off = D.gc_depth_intervals(fr, ref, s, e, clen, W, lo, hi, q, midpoint)
        b, _ = D.gc_depth_intervals(fr, ref, s, e, clen, W, lo, hi, q, midpoint)
        assert torch.equal(a.view(torch.int64), b.view(torch.int64))
        for k in range(len(s)):
            one, _ = D.gc_depth_intervals(fr, ref, [s[k]], [e[k]], clen, W, lo, hi, q, midpoint)
            assert torch.equal(one.view(torch.int64), a[off[k]: off[k + 1]].view(torch.int64)), (midpoint, k)


def test_overflow_flag_and_limits(monkeypatch):
    """A deep pile-up of a huge weight raises OverflowError; a shallow one sums exactly near 2^63; weights of 2^30
    and more, bad tables and bad lengths are refused; no intervals means no launch."""
    clen = 20_000
    codes = np.full(clen, 1, np.uint8); nm = np.zeros(clen, bool)    # all C: g = L
    lo, hi = 100, 200
    W = np.zeros((hi - lo + 1, hi + 1)); W[150 - lo, 150] = 2.0 ** 29 + 0.5   # Q = 2^61 + 2^31
    for n_pile, ok in ((3, True), (5000, False)):
        st = np.full(n_pile, 9000, np.int32); sp = st + 150
        D, ref, fr = _dev(codes, nm, st, sp, np.full(n_pile, 60, np.uint8))
        for midpoint in (False, True):
            if ok:
                got, _ = D.gc_depth_intervals(fr, ref, [8000], [12_000], clen, W, lo, hi, 30, midpoint)
                got = got.cpu().numpy()
                at = 9075 - 8000 if midpoint else slice(1000, 1150)
                assert np.all(got[at] == 3 * (2.0 ** 29 + 0.5)) and got.sum() == 3 * (2.0 ** 29 + 0.5) * (
                    1 if midpoint else 150)
            else:
                with pytest.raises(OverflowError, match="contig"):
                    D.gc_depth_intervals(fr, ref, [8000, 0], [12_000, 10], clen, W, lo, hi, 30, midpoint)
    shape = (hi - lo + 1, hi + 1)
    for bad in (np.full(shape, 2.0 ** 30), np.zeros((3, 3)), np.full(shape, np.nan), np.full(shape, -1.0),
                np.full(shape, np.inf)):
        with pytest.raises(ValueError):
            D.gc_depth_intervals(fr, ref, [0], [10], clen, bad, lo, hi, 30)
    for bad in [(0, 10), (10, 9), (1, 1025), (None, 10)]:
        with pytest.raises(ValueError):
            D.gc_depth_intervals(fr, ref, [0], [10], clen, np.zeros((2, 2)), *bad)

    def no_launch(*a):
        raise AssertionError("a launch without tiles")
    monkeypatch.setattr(D, "_launch", no_launch)
    out, off = D.gc_depth_intervals(fr, ref, [], [], clen, np.ones(shape), lo, hi, 30)
    assert out.numel() == 0 and off.tolist() == [0]
    out, off = D.gc_depth_intervals(fr, ref, [5], [5], clen, np.ones(shape), lo, hi, 30)
    assert out.numel() == 0 and off.tolist() == [0, 0]


def test_coordinate_ceiling(top, big_ref):
    """Intervals reaching 2^31 - 1 on the translated reference (a 300-fold pile-up at the top): the oracle of the
    untranslated contig."""
    from test_gpu_coord_ceiling import _ivs
    D, B, T = top["D"], top["B"], top["T"]
    ivs = _ivs(T, T)
    for lo, hi, q in [(50, 500, 30), (1, 1024, 0)]:
        W = _weights(7, (hi - lo + 1, hi + 1))
        for midpoint in (False, True):
            got, off = D.gc_depth_intervals(top["frB"], big_ref, [a + B for a, _ in ivs], [b + B for _, b in ivs],
                                            B + T, W, lo, hi, q, midpoint)
            exp, eoff = TO.track_intervals(top["st"], top["sp"], top["mq"], top["codes"], top["nm"], T,
                                           [a for a, _ in ivs], [b for _, b in ivs], W, lo, hi, q, midpoint)
            assert np.array_equal(off, eoff) and np.array_equal(got.cpu().numpy(), exp), (lo, hi, midpoint)
            assert exp.sum() > 0


# ------------------------------------------------------------------------------------------ streams and devices
def _stream_case(dev):
    """Fragments whose mapq column holds a decoy (zeros: nothing passes); returns (mapq buffer, real mapq, op,
    expected results of both modes)."""
    import torch
    from finaletoolkit_b200 import device as D
    clen, codes, nm, (st, sp, mq), _ = G._case(2)
    lo, hi, q = 50, 500, 30
    s, e = _intervals(2, clen)
    W = _weights(2, (hi - lo + 1, hi + 1))
    real = torch.from_numpy(mq).to(dev)
    buf = torch.zeros_like(real)
    fr = D.ContigFragments(torch.from_numpy(st).to(dev), torch.from_numpy(sp).to(dev), buf, device=dev)
    ref = D.PackedContig.from_codes(codes, nm, device=dev)
    exp = [TO.track_intervals(st, sp, mq, codes, nm, clen, s, e, W, lo, hi, q, m)[0] for m in (False, True)]

    def op():
        return [D.gc_depth_intervals(fr, ref, s, e, clen, W, lo, hi, q, m)[0] for m in (False, True)]
    return buf, real, op, exp


def test_side_stream():
    """As tests/test_gpu_streams_devices.py: a launch that escapes the current stream reads the decoy."""
    import torch
    from test_gpu_streams_devices import HOLD_CYCLES, SLEEP_CYCLES
    dev = torch.device("cuda", 0)
    buf, real, op, exp = _stream_case(dev)
    decoy = buf.clone()
    buf.copy_(real)
    assert all(np.array_equal(g.cpu().numpy(), x) for g, x in zip(op(), exp))   # loads the kernels first
    torch.cuda.synchronize()
    torch.cuda._sleep(SLEEP_CYCLES + HOLD_CYCLES)
    buf.copy_(decoy)
    side = torch.cuda.Stream(dev)
    with torch.cuda.stream(side):
        torch.cuda._sleep(SLEEP_CYCLES)
        buf.copy_(real)
        res = op()
    side.synchronize()
    for got, x in zip(res, exp):
        assert np.array_equal(got.cpu().numpy(), x) and x.sum() > 0
    torch.cuda.synchronize()


def _two_gpus():
    import torch
    return torch.cuda.is_available() and torch.cuda.device_count() >= 2


@pytest.mark.skipif(not _two_gpus(), reason="needs two CUDA devices")
def test_non_current_device():
    import torch
    dev = torch.device("cuda", 1)
    with torch.cuda.device(0):
        buf, real, op, exp = _stream_case(dev)
        buf.copy_(real)
        res = op()
        assert torch.cuda.current_device() == 0
    torch.cuda.synchronize(dev)
    for got, x in zip(res, exp):
        assert got.device == dev and np.array_equal(got.cpu().numpy(), x)


# ------------------------------------------------------------------------------------------ public API
_BED = ("chrM1\t100\t5000\nchrM1\t4000\t9000\nchrM1\t9000\t9001\nchrM1\t20000\t31000\nchrZ\t5\t10\n"
        "chrM2\t0\t1\nchrM2\t89000\t95000\nchrQ\t1\t2\n")   # in the order of the sizes, as a bigWig needs
_SIZES = "chrM1\t1200345\nchrM2\t90000\nchrQ\t1000\n"   # chrQ: in the sizes, not in the input or the reference


def _merged(lines, left, right, sizes):
    """(contig, start, stop) of _read_intervals: expanded, clamped, neighbours merged."""
    from oracle import oracle as O
    return O.cleavage_intervals(lines, left, right, sizes)


def _exp_tracks(cols, seqs, model, q, midpoint, ivls, scale=1.0):
    W = CO.weights(model.ratio)
    out = []
    for c, a, b in ivls:
        if c in seqs:
            codes, nm = seqs[c]
            v = TO.track(*cols[c][:3], codes, nm, len(codes), a, b, W, model.min_length, model.max_length, q, midpoint)
        else:
            v = np.zeros(b - a)
        out.append((c, a, v * scale))
    return out


def _bedgraph(tracks):
    return "".join(f"{c}\t{p}\t{p + 1}\t{v}\n" for c, a, vals in tracks for p, v in zip(range(a, a + len(vals)),
                                                                                      vals.tolist()))


def test_api_models_text_and_cli(tmp_path, manifest, golden):
    import finaletoolkit_b200 as F
    from click.testing import CliRunner
    from finaletoolkit_b200.cli.main_cli import main_cli
    from finaletoolkit_b200.io import bigwig
    from helpers import read_gz
    frag, tb, seqs, cols = G.motif_files(tmp_path, manifest, golden)
    bed, cs = tmp_path / "i.bed", tmp_path / "sizes.txt"
    bed.write_text(_BED); cs.write_text(_SIZES)
    sizes = {c: int(n) for c, n in (ln.split("\t") for ln in _SIZES.splitlines())}
    lo, hi, q = 100, 220, 20
    model = F.gc_bias(frag, tb, min_length=lo, max_length=hi, quality_threshold=q)
    model_tsv = str(tmp_path / "model.tsv")
    F.gc_bias(frag, tb, output_file=model_tsv, min_length=lo, max_length=hi, quality_threshold=q)
    # the single-region function: three ways to give the model, padding clamped to the contig
    for gcb, extra in ((model, {}), (model_tsv, {}), (None, dict(min_length=lo, max_length=hi))):
        for midpoint in (False, True):
            r = F.gc_corrected_coverage_profile(frag, tb, sizes["chrM2"], "chrM2", 300, 89_990, left=500, right=50,
                                                gc_bias=gcb, quality_threshold=q, midpoint=midpoint, **extra)
            assert r.dtype.names == ("contig", "pos", "depth") and r["depth"].dtype == np.float64
            assert np.all(r["contig"] == "chrM2") and np.array_equal(r["pos"], np.arange(0, 90_000))
            exp = _exp_tracks(cols, seqs, model, q, midpoint, [("chrM2", 0, 90_000)])[0][2]
            assert np.array_equal(r["depth"], exp) and exp.sum() > 0
    assert F.gc_corrected_coverage_profile(frag, tb, 90_000, "chrM2", 5, 5, gc_bias=model).shape == (0,)
    with pytest.warns(UserWarning, match="chrQ"):
        r = F.gc_corrected_coverage_profile(frag, tb, 1000, "chrQ", 10, 20, gc_bias=model)
    assert np.array_equal(r["depth"], np.zeros(10))
    # the multi-interval function: text, bigWig, scaling, normalisation
    lines = _BED.splitlines()
    for j, kw in enumerate([{}, {"midpoint": True, "left": 100, "right": 50, "quality_threshold": 0},
                            {"scale_factor": 2.5}, {"normalize": True, "scale_factor": 1e6}]):
        qq, m = kw.get("quality_threshold", 30), model
        ivls = _merged(lines, kw.get("left", 0), kw.get("right", 0), sizes)
        s = kw.get("scale_factor", 1.0)
        if kw.get("normalize"):
            total = F.single_coverage(frag, min_length=lo, max_length=hi, quality_threshold=qq).coverage
            s = s / total
        exp = _exp_tracks(cols, seqs, m, qq, kw.get("midpoint", False), ivls, s)
        assert sum(float(v.sum()) for _, _, v in exp) > 0
        for suffix in ("bed.gz", "bedgraph.gz", "bw"):
            out = str(tmp_path / f"m{j}.{suffix}")
            with warnings.catch_warnings(record=True) as w:
                warnings.simplefilter("always")
                assert F.multi_gc_corrected_coverage_profile(frag, tb, str(bed), str(cs), output_file=out, gc_bias=m,
                                                             **kw) == out
            msgs = [str(x.message) for x in w if issubclass(x.category, UserWarning)]
            assert any("chrZ" in x for x in msgs) and msgs[-1] == (
                "multi_gc_corrected_coverage_profile: intervals on contigs that the input or the reference lacks "
                "count 0: chrQ")
            if suffix == "bw":
                r = bigwig.open(out)
                for c, a, vals in exp:
                    assert np.array_equal(r.values(c, a, a + len(vals)), vals.astype(np.float32)), (kw, c, a)
            else:
                assert read_gz(out) == _bedgraph(exp), (kw, suffix)
    # the CLI == the API
    args = [["--gc-bias", model_tsv, "-q", "20", "--midpoint", "--pad-left", "40", "--pad-right", "7"],
            ["--min-length", str(lo), "--max-length", str(hi), "-q", "20", "--scale-factor", "3", "-n", "-t", "2"]]
    kwargs = [dict(gc_bias=model_tsv, quality_threshold=20, midpoint=True, left=40, right=7),
              dict(min_length=lo, max_length=hi, quality_threshold=20, scale_factor=3.0, normalize=True, workers=2)]
    for j, (a, kw) in enumerate(zip(args, kwargs)):
        cli_out, api_out = str(tmp_path / f"cli{j}.bed.gz"), str(tmp_path / f"api{j}.bed.gz")
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            res = CliRunner().invoke(main_cli, ["gc-corrected-coverage-profile", frag, tb, str(bed), str(cs),
                                                "-o", cli_out] + a)
            assert res.exit_code == 0, res.output
            F.multi_gc_corrected_coverage_profile(frag, tb, str(bed), str(cs), output_file=api_out, **kw)
        assert read_gz(cli_out) == read_gz(api_out) and len(read_gz(cli_out)) > 0, a


def test_api_errors(tmp_path, manifest, golden):
    import finaletoolkit_b200 as F
    frag, tb, _, _ = G.motif_files(tmp_path, manifest, golden)
    bed, cs = tmp_path / "i.bed", tmp_path / "sizes.txt"
    bed.write_text(_BED); cs.write_text(_SIZES)
    model = F.gc_bias(frag, tb, min_length=100, max_length=220, quality_threshold=20)
    multi = lambda **kw: F.multi_gc_corrected_coverage_profile(frag, tb, str(bed), str(cs), **kw)   # noqa: E731
    single = lambda **kw: F.gc_corrected_coverage_profile(frag, tb, 90_000, "chrM2", 0, 100, **kw)   # noqa: E731
    with pytest.raises(ValueError):
        multi(output_file="x.txt", gc_bias=model)
    with pytest.raises(TypeError):
        multi(output_file=3, gc_bias=model)
    with pytest.raises(ValueError):
        F.multi_gc_corrected_coverage_profile("-", tb, "-", str(cs), gc_bias=model)
    with pytest.raises(ValueError):
        F.multi_gc_corrected_coverage_profile(frag, tb, str(bed), None, gc_bias=model)
    for fn in (multi, single):
        for kw in [{"min_length": 99}, {"max_length": 221}, {"gc_regions": str(bed)}]:
            with pytest.raises(ValueError):
                fn(gc_bias=model, **kw)
        with pytest.raises(TypeError):
            fn(gc_bias=3)
        with pytest.raises(ValueError):
            fn(min_length=0, max_length=10)          # fitting rejects the lengths
        bad = tmp_path / "bad.tsv"
        bad.write_text("length\tgc\tobserved\texpected\tratio\n5\t0\t1\t1\t1.0\n")
        with pytest.raises(ValueError):
            fn(gc_bias=str(bad))


def check_bam(bam):
    """BAM input: each region's fragments are the rows an indexed fetch of it yields."""
    import finaletoolkit_b200 as F
    from finaletoolkit_b200.io.fragments import as_table
    from finaletoolkit_b200.io.reference import open_reference
    from helpers import read_gz
    tab = as_table(bam["path"])
    ref = open_reference(bam["tb"])
    tiles = [ln.split("\t") for ln in bam["m"]["tiles"].splitlines()]
    regions = [(t[0], int(t[1]), int(t[2])) for t in tiles[:6]] + [("chrA", 0, 1), ("chrA", 480, 12_345)]
    lo, hi, q = 50, 600, 0
    model = F.gc_bias(bam["path"], bam["tb"], min_length=lo, max_length=hi, quality_threshold=q)
    W = CO.weights(model.ratio)
    total = 0.0
    for midpoint in (False, True):
        for c, a, b in regions:
            r = F.gc_corrected_coverage_profile(bam["path"], bam["tb"], bam["sizes"][c], c, a, b, gc_bias=model,
                                                quality_threshold=q, midpoint=midpoint)
            codes, nm = ref.contig_arrays(c)
            st, sp, mq, _ = tab.fetched(c, a, b).host(c)
            exp = TO.track(st, sp, mq, codes, nm, ref.chroms[c], a, b, W, lo, hi, q, midpoint)
            assert np.array_equal(r["depth"], exp), (c, a, b, midpoint)
            total += float(exp.sum())
    assert total > 0
    out = str(bam["dir"] / "gc_depth.bed.gz")
    F.multi_gc_corrected_coverage_profile(bam["path"], bam["tb"], bam["tiles"], bam["cs"], output_file=out,
                                          gc_bias=model, quality_threshold=q)
    exp = []
    for c, a, b in _merged(bam["m"]["tiles"].splitlines(), 0, 0, bam["sizes"]):
        codes, nm = ref.contig_arrays(c)
        st, sp, mq, _ = tab.fetched(c, a, b).host(c)
        exp.append((c, a, TO.track(st, sp, mq, codes, nm, ref.chroms[c], a, b, W, lo, hi, q)))
    assert read_gz(out) == _bedgraph(exp)


@pytest.fixture(scope="module")
def bam(tmp_path_factory, golden):
    import bam_replay as R
    from finaletoolkit_b200.io import fragments
    fragments._CACHE.clear()
    yield R.make_fixture(tmp_path_factory.mktemp("gc_track_bam"), golden)
    fragments._CACHE.clear()


def test_bam_fetch_semantics(bam):
    check_bam(bam)
