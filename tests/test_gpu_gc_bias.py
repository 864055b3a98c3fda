"""CUDA fragment GC bias (gc_bias, device.gc_observed / gc_expected, ftk_gc_observed_u64 / ftk_gc_expected_u64)
against the numpy definition in tests/gc_oracle.py, the observed == expected cross-check, the coordinate ceiling,
the public API, the CLI and the BAM fetch semantics."""
import gzip
import warnings

import numpy as np
import pytest

import gc_oracle as GO
from helpers import golden_codes, write_2bit, write_frag_gz
from test_gpu_coord_ceiling import big_ref, top  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

_FILTERS = [(50, 500, 30), (1, 64, 0), (160, 160, 20), (1, 1024, 0), (200, 1024, 60)]   # (min, max, q) per seed


def _contig(seed, clen):
    """Random ACGT with many short N blocks, several starting or ending at offsets 0, 15, 16, 31 (mod 32)."""
    rng = np.random.default_rng(700 + seed)
    codes = rng.integers(0, 4, clen, dtype=np.uint8)
    nm = np.zeros(clen, bool)
    for _ in range(int(rng.integers(20, 60))):
        a = int(rng.integers(0, clen)); nm[a: a + int(rng.integers(1, 300))] = True
    for r in (0, 15, 16, 31):
        a = 32 * int(rng.integers(1, clen // 32 - 2)) + r; nm[a: a + int(rng.integers(1, 40))] = True   # starts at r
        b = 32 * int(rng.integers(1, clen // 32 - 2)) + r; nm[max(b - int(rng.integers(1, 40)), 0): b + 1] = True   # ends at r
    return codes, nm


def _frags(seed, clen):
    """synth_fragments plus uniform lengths up to 1100, rows past the contig end and rows before 0."""
    from finaletoolkit_b200.synth import synth_fragments
    rng = np.random.default_rng(800 + seed)
    st, sp, mq, _ = synth_fragments(clen, int(rng.integers(2_000, 40_000)), seed, seed_base=909)
    st, sp = st.astype(np.int64), sp.astype(np.int64)
    u = rng.integers(0, clen, 3000); ul = rng.integers(1, 1100, 3000)
    st = np.concatenate([st, u, clen - rng.integers(0, 300, 50), [0, 0, clen - 1]])
    sp = np.concatenate([sp, u + ul, st[-53:-3] + rng.integers(1, 600, 50), [1, 1024, clen]])
    mq = np.concatenate([mq, rng.integers(0, 61, 3053).astype(np.uint8)])
    order = np.argsort(st, kind="stable")
    return st[order].astype(np.int32), sp[order].astype(np.int32), mq[order]


def _regions(seed, clen):
    """Overlapping, touching, 1-bp regions, one at 0, one at the contig end and one past it; merged as gc_bias does."""
    rng = np.random.default_rng(900 + seed)
    rows = []
    for _ in range(12):
        a = int(rng.integers(0, clen)); rows.append(("c", a, a + int(rng.integers(1, 6000))))
    rows += [("c", rows[0][2], rows[0][2] + 500), ("c", rows[1][1] + 3, rows[1][1] + 4), ("c", 0, 300), ("c", 0, 1),
             ("c", clen - 700, clen), ("c", clen + 10, clen + 900), ("c", clen - 5, clen + 50)]
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        return GO.merge_regions(rows, {"c": clen})["c"]


def _case(seed):
    clen = int(np.random.default_rng(seed).integers(30_000, 90_000)) | 1   # odd: not a multiple of 16
    codes, nm = _contig(seed, clen)
    return clen, codes, nm, _frags(seed, clen), _regions(seed, clen)


@pytest.mark.parametrize("seed", range(5))
def test_random_vs_numpy(seed):
    import torch
    from finaletoolkit_b200 import device as D
    clen, codes, nm, (st, sp, mq), (rs, re) = _case(seed)
    lo, hi, q = _FILTERS[seed]
    ref = D.PackedContig.from_codes(codes, nm, device="cuda:0")
    fr = D.ContigFragments(st, sp, mq, device="cuda:0")
    O = D.gc_observed(fr, ref, rs, re, lo, hi, q)
    E = D.gc_expected(ref, rs, re, lo, hi)
    assert O.dtype == torch.int64 and tuple(O.shape) == tuple(E.shape) == (hi - lo + 1, hi + 1)
    eo = GO.observed(st, sp, mq, codes, nm, clen, rs, re, lo, hi, q)
    ee = GO.expected(codes, nm, clen, rs, re, lo, hi)
    assert np.array_equal(O.cpu().numpy(), eo), seed
    assert np.array_equal(E.cpu().numpy(), ee), seed
    assert eo.sum() > 0 and ee.sum() > 0


def test_observed_equals_expected():
    """A fragment table holding every placement (p, L) whose midpoint lies in the regions, once, at mapq 60."""
    from finaletoolkit_b200 import device as D
    clen = 4099
    codes, nm = _contig(11, clen)
    rs, re = np.array([0, 700, 2001, 4000]), np.array([500, 2000, 2002, 4099])
    st, sp = [], []
    for L in range(1, 65):
        p = np.arange(0, clen - L + 1)
        p = p[GO.in_regions(p + L // 2, rs, re)]
        st.append(p); sp.append(p + L)
    st, sp = np.concatenate(st), np.concatenate(sp)
    ref = D.PackedContig.from_codes(codes, nm, device="cuda:0")
    fr = D.ContigFragments(st, sp, np.full(st.size, 60, np.uint8), device="cuda:0")
    for lo, hi in [(1, 64), (7, 40), (64, 64)]:
        O = D.gc_observed(fr, ref, rs, re, lo, hi, 30).cpu().numpy()
        E = D.gc_expected(ref, rs, re, lo, hi).cpu().numpy()
        assert np.array_equal(O, E) and E.sum() > 0, (lo, hi)


@pytest.mark.parametrize("splits,tile", [(1, 1), (2, 7), (3, 100), (7, 2048), (1000, 16384)])
def test_slices_tiles_and_accumulation(splits, tile, monkeypatch):
    import torch
    from finaletoolkit_b200 import device as D
    clen, codes, nm, (st, sp, mq), (rs, re) = _case(1)
    monkeypatch.setattr(D, "_splits_for", lambda *a, **k: splits)
    monkeypatch.setattr(D, "_gc_tile_for", lambda *a, **k: tile)
    ref = D.PackedContig.from_codes(codes, nm, device="cuda:0")
    fr = D.ContigFragments(st, sp, mq, device="cuda:0")
    lo, hi = (20, 300) if tile > 1 else (100, 131)
    eo = GO.observed(st, sp, mq, codes, nm, clen, rs, re, lo, hi, 30)
    ee = GO.expected(codes, nm, clen, rs, re, lo, hi)
    assert np.array_equal(D.gc_observed(fr, ref, rs, re, lo, hi, 30).cpu().numpy(), eo)
    assert np.array_equal(D.gc_expected(ref, rs, re, lo, hi).cpu().numpy(), ee)
    k = len(rs) // 2   # accumulation: the two halves of the region list into one matrix
    a = D.gc_observed(fr, ref, rs[:k], re[:k], lo, hi, 30)
    assert np.array_equal(D.gc_observed(fr, ref, rs[k:], re[k:], lo, hi, 30, out=a).cpu().numpy(), eo)
    b = D.gc_expected(ref, rs[:k], re[:k], lo, hi)
    assert np.array_equal(D.gc_expected(ref, rs[k:], re[k:], lo, hi, out=b).cpu().numpy(), ee)
    if splits == 1:
        for empty in (D.ContigFragments(st, sp, np.zeros_like(mq), device="cuda:0"),     # every mapq below q
                      D.ContigFragments(st[:0], sp[:0], mq[:0], device="cuda:0")):      # no fragment at all
            assert int(D.gc_observed(empty, ref, rs, re, lo, hi, 30).abs().sum()) == 0

        def no_call():
            raise AssertionError("a launch without regions")
        monkeypatch.setattr(D, "lib", no_call)
        z = torch.zeros((hi - lo + 1, hi + 1), dtype=torch.int64, device="cuda:0")
        assert D.gc_observed(fr, ref, [], [], lo, hi, 30, out=z) is z and D.gc_expected(ref, [], [], lo, hi, out=z) is z
        assert int(z.abs().sum()) == 0
        with pytest.raises(ValueError):
            D.gc_expected(ref, rs, re, lo, hi, out=torch.zeros((3, 3), dtype=torch.int64, device="cuda:0"))
        for bad in [(0, 10), (10, 9), (1, 1025), (1.5, 10)]:
            with pytest.raises(ValueError):
                D.gc_check(*bad)


def test_coordinate_ceiling(top, big_ref):
    """Regions and fragments reaching 2^31 - 1 on the translated reference: the oracle of the untranslated contig."""
    D, B, T = top["D"], top["B"], top["T"]
    rs = np.array([5000, 100_000, T - 5000, T - 2], np.int64); re = np.array([60_000, 150_000, T - 10, T], np.int64)
    for lo, hi, q in [(50, 500, 30), (1, 1024, 0)]:
        got = D.gc_observed(top["frB"], big_ref, rs + B, re + B, lo, hi, q).cpu().numpy()
        exp = GO.observed(top["st"], top["sp"], top["mq"], top["codes"], top["nm"], T, rs, re, lo, hi, q)
        assert np.array_equal(got, exp) and exp.sum() > 0, (lo, hi, q)
    sel = (rs[2:], re[2:])   # the expected counts near the top (the whole contig would take the oracle minutes)
    got = D.gc_expected(big_ref, sel[0] + B, sel[1] + B, 1, 1024).cpu().numpy()
    exp = GO.expected(top["codes"], top["nm"], T, sel[0], sel[1], 1, 1024)
    assert np.array_equal(got, exp) and exp.sum() > 0


# ------------------------------------------------------------------------------------------ public API
def motif_files(tmp_path, manifest, golden):
    """The motif golden's two contigs as a fragment file and a .2bit; returns (frag, 2bit, {contig: (codes, nm)}, cols)."""
    g = golden("motif"); m = manifest["motif"]
    sizes = dict(m["contigs"])
    cols = {c: tuple(g[f"{c}_{k}"] for k in ("start", "stop", "mapq", "strand")) for c in sizes}
    seqs = {c: golden_codes(g, c, n) for c, n in sizes.items()}
    frag = write_frag_gz(tmp_path / "gc.frag.gz", cols)
    tb = write_2bit(tmp_path / "gc.2bit", [(c, *seqs[c]) for c in sizes])
    return frag, tb, seqs, cols


def expected_result(cols, seqs, regions, lo, hi, q):
    O = np.zeros((hi - lo + 1, hi + 1), np.int64); E = O.copy()
    for c, (rs, re) in regions.items():
        codes, nm = seqs[c]
        E += GO.expected(codes, nm, len(codes), rs, re, lo, hi)
        st, sp, mq = cols[c][:3]
        O += GO.observed(st, sp, mq, codes, nm, len(codes), rs, re, lo, hi, q)
    return O, E


_BED = ("# regions\ntrack name=r\nbrowser position chrM1:1-100\n\nchrM1\t100\t5000\nchrM1\t4000\t9000\nchrM1\t9000\t9001\n"
        "chrM2\t0\t1\nchrM2\t30\t20000000\nchrZ\t5\t10\nchrM1\t-50\t40\nchrQ\t1\t2\n")


def test_gc_bias_api(tmp_path, manifest, golden):
    import finaletoolkit_b200 as F
    from click.testing import CliRunner
    from finaletoolkit_b200.cli.main_cli import main_cli
    frag, tb, seqs, cols = motif_files(tmp_path, manifest, golden)
    sizes = {c: len(s[0]) for c, s in seqs.items()}
    whole = {c: (np.array([0]), np.array([n])) for c, n in sizes.items()}
    bed = tmp_path / "r.bed"; bed.write_text(_BED)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        merged = GO.merge_regions([ln.split()[:3] for ln in _BED.splitlines()
                                   if ln.strip() and not ln.startswith(("#", "track", "browser"))], sizes)
    # (the oracle's expected counts over the 1.2-Mb contig take seconds per hundred lengths: one setting there)
    for regions, interval_file, settings in ((whole, None, [(100, 220, 30)]),
                                             (merged, str(bed), [(50, 500, 30), (1, 1024, 0), (167, 167, 0)])):
        for lo, hi, q in settings:
            with warnings.catch_warnings(record=True) as w:
                warnings.simplefilter("always")
                r = F.gc_bias(frag, tb, interval_file, min_length=lo, max_length=hi, quality_threshold=q)
            assert [str(x.message) for x in w if issubclass(x.category, UserWarning)] == \
                ([] if interval_file is None else ["gc_bias: regions on contigs that the input or the reference lacks "
                                                   "were skipped: chrZ, chrQ"])
            O, E = expected_result(cols, seqs, regions, lo, hi, q)
            assert isinstance(r, F.GCBias) and (r.min_length, r.max_length) == (lo, hi)
            assert r.observed.dtype == r.expected.dtype == np.int64 and r.ratio.dtype == np.float64
            assert np.array_equal(r.observed, O) and np.array_equal(r.expected, E), (interval_file, lo, hi, q)
            assert np.array_equal(r.ratio, GO.ratio(O, E), equal_nan=True)
            assert O.sum() > 0
    # text: .tsv, .tsv.gz and the CLI on stdout
    r = F.gc_bias(frag, tb, str(bed), min_length=100, max_length=220, quality_threshold=0)
    text = GO.text(r.observed, r.expected, r.ratio, 100)
    tsv, tgz = str(tmp_path / "g.tsv"), str(tmp_path / "g.tsv.gz")
    F.gc_bias(frag, tb, str(bed), output_file=tsv, min_length=100, max_length=220, quality_threshold=0)
    assert open(tsv).read() == text
    F.gc_bias(frag, tb, str(bed), output_file=tgz, min_length=100, max_length=220, quality_threshold=0)
    with gzip.open(tgz, "rt") as fh:
        assert fh.read() == text
    res = CliRunner().invoke(main_cli, ["gc-bias", frag, tb, "--regions", str(bed), "--min-length", "100",
                                        "--max-length", "220", "-q", "0"])
    assert res.exit_code == 0, res.output
    assert res.output == text


def test_gc_bias_fasta_iupac(tmp_path):
    """FASTA input: every character other than ACGTacgt is N (IUPAC codes included)."""
    import finaletoolkit_b200 as F
    rng = np.random.default_rng(4)
    alphabet = np.frombuffer(b"ACGTacgtNnRYKMSWBDHV", np.uint8)
    seq = rng.choice(alphabet[:8], 20_011)
    seq[rng.integers(0, seq.size, 120)] = rng.choice(alphabet[8:], 120)
    fa = tmp_path / "r.fa"
    fa.write_text(">chrF desc\n" + "\n".join(seq[i:i + 60].tobytes().decode() for i in range(0, seq.size, 60)) + "\n")
    lut = {ord(ch): v for ch, v in zip("ACGTacgt", (0, 1, 2, 3, 0, 1, 2, 3))}
    codes = np.array([lut.get(int(x), 0) for x in seq], np.uint8)
    nm = np.array([int(x) not in lut for x in seq])
    st = np.sort(rng.integers(0, 20_000, 5000)); sp = st + rng.integers(30, 400, 5000)
    mq = rng.integers(0, 61, 5000).astype(np.uint8)
    frag = write_frag_gz(tmp_path / "f.frag.gz", {"chrF": (st, sp, mq, np.ones(5000, np.uint8))})
    r = F.gc_bias(frag, str(fa), min_length=30, max_length=400, quality_threshold=20)
    full = (np.array([0]), np.array([seq.size]))
    assert np.array_equal(r.observed, GO.observed(st, sp, mq, codes, nm, seq.size, *full, 30, 400, 20))
    assert np.array_equal(r.expected, GO.expected(codes, nm, seq.size, *full, 30, 400))
    assert r.observed.sum() > 0


def test_gc_bias_errors(tmp_path, manifest, golden):
    import finaletoolkit_b200 as F
    frag, tb, _, _ = motif_files(tmp_path, manifest, golden)
    for kw in [{"min_length": 0}, {"min_length": 300, "max_length": 200}, {"max_length": 1025}, {"min_length": None},
               {"max_length": 12.5}]:
        with pytest.raises(ValueError):
            F.gc_bias(frag, tb, **kw)
    with pytest.raises(ValueError):
        F.gc_bias(frag, tb, output_file="x.txt")
    with pytest.raises(TypeError):
        F.gc_bias(frag, tb, output_file=3)
    bad = tmp_path / "bad.bed"
    for text in ("chrM1\t500\t400\n", "chrM1\t500\n"):
        bad.write_text(text)
        with pytest.raises(ValueError):
            F.gc_bias(frag, tb, str(bad))


def check_bam(bam):
    """BAM input: each merged region's fragments are the rows an indexed fetch of the region yields."""
    import finaletoolkit_b200 as F
    from finaletoolkit_b200.io.fragments import as_table
    from finaletoolkit_b200.io.reference import open_reference
    tab = as_table(bam["path"])
    ref = open_reference(bam["tb"])
    tiles = [ln.split("\t") for ln in bam["m"]["tiles"].splitlines()]
    rows = [(t[0], int(t[1]), int(t[2])) for t in tiles[::3]] + [("chrA", 0, 1), ("chrA", 480, 12345)]
    bed = bam["dir"] / "gc_regions.bed"; bed.write_text("".join(f"{c}\t{a}\t{b}\n" for c, a, b in rows))
    sizes = {c: ref.chroms[c] for c in tab.contigs if c in ref.chroms}
    regions = GO.merge_regions(rows, sizes)
    for lo, hi, q in [(50, 600, 0), (100, 220, 20)]:
        r = F.gc_bias(bam["path"], bam["tb"], str(bed), min_length=lo, max_length=hi, quality_threshold=q)
        O = np.zeros_like(r.observed); E = np.zeros_like(r.expected)
        for c, (rs, re) in regions.items():
            codes, nm = ref.contig_arrays(c)
            E += GO.expected(codes, nm, sizes[c], rs, re, lo, hi)
            for a, b in zip(rs.tolist(), re.tolist()):
                st, sp, mq, _ = tab.fetched(c, a, b).host(c)
                O += GO.observed(st, sp, mq, codes, nm, sizes[c], [a], [b], lo, hi, q)
        assert np.array_equal(r.observed, O) and np.array_equal(r.expected, E), (lo, hi, q)
        assert O.sum() > 0


@pytest.fixture(scope="module")
def bam(tmp_path_factory, golden):
    import bam_replay as R
    from finaletoolkit_b200.io import fragments
    fragments._CACHE.clear()
    yield R.make_fixture(tmp_path_factory.mktemp("gc_bam"), golden)
    fragments._CACHE.clear()


def test_bam_fetch_semantics(bam):
    check_bam(bam)
