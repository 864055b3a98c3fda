"""CUDA per-base fragment depth (coverage_profile / multi_coverage_profile, ftk_depth_tiles_i32) against the
numpy definition in tests/depth_oracle.py, the cleavage kernel and the BAM fetch semantics."""
import numpy as np
import pytest

import depth_oracle as DO
from oracle import oracle as O
from test_gpu_api import fx, syn  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

_FILTERS = [(None, None, 30), (100, 200, 0), (0, 600, 60), (150, None, 20)]   # (min_length, max_length, q) per seed


def _random_case(seed):
    """A synthetic contig with a few fragments longer than one 5120-position tile, and its intervals:
    1-bp ones, both contig ends, ones longer than a tile, random ones."""
    from finaletoolkit_b200.synth import synth_fragments
    rng = np.random.default_rng(70 + seed)
    clen = int(rng.integers(30_000, 90_000)); n = int(rng.integers(100, 40_000))
    st, sp, mq, sd = synth_fragments(clen, n, seed, seed_base=321)
    ls = rng.integers(5200, 15_000, 6); ss = rng.integers(0, clen - 1, 6)
    st = np.concatenate([st, ss.astype(np.int32)]); sp = np.concatenate([sp, np.minimum(ss + ls, clen).astype(np.int32)])
    mq = np.concatenate([mq, np.full(6, 60, np.uint8)]); sd = np.concatenate([sd, np.ones(6, np.uint8)])
    order = np.argsort(st, kind="stable")
    ivs = [(0, clen), (0, 1), (clen - 1, clen), (100, 5219), (100, 5220), (7, 20_500), (5119, 5121)]
    ivs += [(int(s), int(min(s + rng.integers(1, 12_000), clen))) for s in rng.integers(0, clen - 1, 8)]
    return clen, st[order], sp[order], mq[order], sd[order], ivs


@pytest.mark.parametrize("midpoint", [False, True])
@pytest.mark.parametrize("seed", range(4))
def test_random_vs_numpy(seed, midpoint):
    import torch
    from finaletoolkit_b200.device import ContigFragments, depth_intervals
    clen, st, sp, mq, sd, ivs = _random_case(seed)
    lo, hi, q = _FILTERS[seed]
    fr = ContigFragments(st, sp, mq, sd, device="cuda:0")
    out, off = depth_intervals(fr, [a for a, _ in ivs], [b for _, b in ivs], clen, lo, hi, q, midpoint)
    assert out.dtype == torch.int32
    exp, exp_off = DO.depth_intervals(st, sp, mq, [a for a, _ in ivs], [b for _, b in ivs], lo, hi, q, midpoint)
    assert np.array_equal(off, exp_off)
    got = out.cpu().numpy()
    for k, (a, b) in enumerate(ivs):
        assert np.array_equal(got[off[k]:off[k + 1]], exp[off[k]:off[k + 1]]), (seed, midpoint, a, b)


@pytest.mark.parametrize("midpoint", [False, True])
def test_contig_without_passing_fragments(midpoint):
    from finaletoolkit_b200.device import ContigFragments, depth_intervals
    clen, st, sp, mq, sd, ivs = _random_case(0)
    for fr in (ContigFragments(st, sp, np.zeros_like(mq), sd, device="cuda:0"),          # every mapq below q
               ContigFragments(st[:0], sp[:0], mq[:0], sd[:0], device="cuda:0")):     # no fragment at all
        out, off = depth_intervals(fr, [a for a, _ in ivs], [b for _, b in ivs], clen, None, None, 30, midpoint)
        assert out.numel() == off[-1] == sum(b - a for a, b in ivs) and int(out.abs().sum()) == 0
    out, off = depth_intervals(fr, [], [], clen, None, None, 30, midpoint)
    assert out.numel() == 0 and off.tolist() == [0]


@pytest.mark.parametrize("seed", range(3))
def test_span_depth_pins_the_cleavage_kernel(seed):
    """cleavage_intervals (pinned to the reference goldens) == numpy ends / new depth * 100 where depth != 0."""
    from finaletoolkit_b200.device import ContigFragments, cleavage_intervals, depth_intervals
    clen, st, sp, mq, sd, ivs = _random_case(seed)
    lo, hi, q = _FILTERS[seed]
    fr = ContigFragments(st, sp, mq, sd, device="cuda:0")
    starts, stops = [a for a, _ in ivs], [b for _, b in ivs]
    clv, off = cleavage_intervals(fr, starts, stops, clen, lo, hi, q)
    dep, off2 = depth_intervals(fr, starts, stops, clen, lo, hi, q)
    assert np.array_equal(off, off2)
    clv, dep = clv.cpu().numpy(), dep.cpu().numpy()
    ok = DO.passing(st, sp, mq, lo, hi, q)
    for k, (a, b) in enumerate(ivs):
        sel = ok & (sp > a) & (st < b)                     # frag_array(..., "any") of the interval
        endpos = np.where(sd[sel] == 1, st[sel], sp[sel]).astype(np.int64) - a
        ends = np.bincount(endpos[(endpos >= 0) & (endpos < b - a)], minlength=b - a)
        d = dep[off[k]:off[k + 1]].astype(np.int64)
        exp = np.zeros(b - a); nz = d != 0
        exp[nz] = ends[nz] / d[nz] * 100
        assert np.array_equal(clv[off[k]:off[k + 1]], exp), (seed, a, b)


def test_chromosome_scale_tiling():
    """30 Mb, 9 M fragments: the whole contig in one interval == a 5-kb tiling (depth is local), and a
    200-kb window against numpy."""
    import torch
    from finaletoolkit_b200.device import ContigFragments, depth_intervals
    from finaletoolkit_b200.synth import synth_fragments
    clen, n = 30_000_000, 9_000_000
    st, sp, mq, sd = synth_fragments(clen, n, 9)
    fr = ContigFragments(st, sp, mq, sd, device="cuda:0")
    edges = np.arange(0, clen + 5000, 5000).clip(max=clen)
    lo, hi = 12_000_000, 12_200_000
    for midpoint in (False, True):
        a, _ = depth_intervals(fr, [0], [clen], clen, None, None, 30, midpoint)
        b, _ = depth_intervals(fr, edges[:-1], edges[1:], clen, None, None, 30, midpoint)
        assert torch.equal(a, b)
        assert np.array_equal(a[lo:hi].cpu().numpy(), DO.depth(st, sp, mq, lo, hi, q=30, midpoint=midpoint))
        if midpoint:   # every passing fragment has its midpoint inside the contig
            assert int(a.sum()) == int(DO.passing(st, sp, mq, q=30).sum())


# ------------------------------------------------------------------------------------------ public API
def _host(path, contig):
    from finaletoolkit_b200.io.fragments import as_table
    st, sp, mq, _ = as_table(path).host(contig)
    return st, sp, mq


def _bedgraph(contigs_starts_values):
    return "".join(f"{c}\t{p}\t{p + 1}\t{v}\n" for c, s, vals in contigs_starts_values
                   for p, v in zip(range(s, s + len(vals)), vals.tolist()))


def test_coverage_profile_api(fx, syn, manifest):
    import finaletoolkit_b200 as F
    m = manifest["fixture17"]
    st, sp, mq = _host(fx["frag"], "12")
    cases = [(34443118, 34443538, {}), (34444968, 34446115, {"quality_threshold": 0}),
             (34443000, 34447000, {"quality_threshold": 0, "midpoint": True}),
             (34443000, 34447000, {"min_length": 150, "max_length": 200, "quality_threshold": 0, "left": 30, "right": 70})]
    for a, b, kw in cases:
        r = F.coverage_profile(fx["frag"], m["chrom_size"], "12", a, b, **kw)
        a2, b2 = a - kw.get("left", 0), b + kw.get("right", 0)
        assert r.dtype.names == ("contig", "pos", "depth") and r["depth"].dtype == np.int64
        assert np.all(r["contig"] == "12") and np.array_equal(r["pos"], np.arange(a2, b2))
        exp = DO.depth(st, sp, mq, a2, b2, kw.get("min_length"), kw.get("max_length"), kw.get("quality_threshold", 30),
                       kw.get("midpoint", False))
        assert np.array_equal(r["depth"], exp), kw
        assert exp.any()
    # padding clamped to the contig; an empty region
    sizes = dict(manifest["synth_small"]["contigs"])
    st, sp, mq = _host(syn["frag"], "chrC")
    r = F.coverage_profile(syn["frag"], sizes["chrC"], "chrC", 10, sizes["chrC"] - 10, left=50, right=50)
    assert np.array_equal(r["pos"], np.arange(sizes["chrC"]))
    assert np.array_equal(r["depth"], DO.depth(st, sp, mq, 0, sizes["chrC"]))
    assert F.coverage_profile(syn["frag"], sizes["chrC"], "chrC", 5, 5).shape == (0,)


def test_multi_coverage_profile_api(syn, manifest, tmp_path):
    """bedGraph text exactly, bigWig values, normalisation, errors and the unknown-contig warning."""
    import finaletoolkit_b200 as F
    from finaletoolkit_b200.io import bigwig
    from helpers import read_gz
    sizes = dict(manifest["synth_small"]["contigs"])
    bed = tmp_path / "ivl.bed"; bed.write_text(manifest["cleavage"]["bed"])   # merges, an unknown contig, out of order
    cols = {c: _host(syn["frag"], c) for c in sizes}
    for j, kw in enumerate([{}, {"midpoint": True, "left": 100, "right": 50, "quality_threshold": 0},
                            {"min_length": 100, "max_length": 200, "scale_factor": 2.5},
                            {"normalize": True, "scale_factor": 1e6, "min_length": 120}]):
        ivls = O.cleavage_intervals(bed.read_text().splitlines(), kw.get("left", 0), kw.get("right", 0), sizes)
        flt = (kw.get("min_length"), kw.get("max_length"), kw.get("quality_threshold", 30))
        s = kw.get("scale_factor", 1.0)
        if kw.get("normalize"):
            total = sum(int(DO.passing(*cols[c], *flt).sum()) for c in sizes)
            assert total == F.single_coverage(syn["frag"], min_length=flt[0], max_length=flt[1],
                                              quality_threshold=flt[2]).coverage
            s = s / total
        exp = [(c, a, DO.depth(*cols[c], a, b, *flt, kw.get("midpoint", False)).astype(np.float64) * s)
               for c, a, b in ivls]
        for suffix in ("bed.gz", "bedgraph.gz"):
            out = str(tmp_path / f"m{j}.{suffix}")
            with pytest.warns(UserWarning):
                assert F.multi_coverage_profile(syn["frag"], str(bed), syn["cs"], output_file=out, **kw) == out
            assert read_gz(out) == _bedgraph(exp), (kw, suffix)
        out = str(tmp_path / f"m{j}.bw")
        with pytest.warns(UserWarning):
            F.multi_coverage_profile(syn["frag"], str(bed), syn["cs"], output_file=out, **kw)
        r = bigwig.open(out)
        last = {}
        for c, a, vals in exp:
            if a < last.get(c, 0):   # an interval out of order is skipped by the writer, as for cleavage profiles
                continue
            last[c] = a + len(vals)
            assert np.array_equal(r.values(c, a, a + len(vals)), vals.astype(np.float32)), (kw, c, a)
    with pytest.raises(ValueError):
        F.multi_coverage_profile(syn["frag"], str(bed), syn["cs"], output_file="x.txt")
    with pytest.raises(TypeError):
        F.multi_coverage_profile(syn["frag"], str(bed), syn["cs"], output_file=3)
    with pytest.raises(ValueError):
        F.multi_coverage_profile("-", "-", syn["cs"])
    with pytest.raises(ValueError):
        F.multi_coverage_profile(syn["frag"], str(bed), None)


def check_bam(bam):
    """BAM input: the oracle over the rows an indexed fetch of each region yields (FragmentTable.fetched)."""
    import finaletoolkit_b200 as F
    from finaletoolkit_b200.io.fragments import as_table
    from helpers import read_gz
    tab = as_table(bam["path"])
    tiles = [ln.split("\t") for ln in bam["m"]["tiles"].splitlines()]
    regions = [(t[0], int(t[1]), int(t[2])) for t in tiles[:6]] + [("chrA", 0, 1), ("chrA", 480, 12_345)]
    for midpoint in (False, True):
        for c, a, b in regions:
            r = F.coverage_profile(bam["path"], bam["sizes"][c], c, a, b, quality_threshold=0, midpoint=midpoint)
            st, sp, mq, _ = tab.fetched(c, a, b).host(c)
            assert np.array_equal(r["depth"], DO.depth(st, sp, mq, a, b, q=0, midpoint=midpoint)), (c, a, b, midpoint)
    out = str(bam["dir"] / "depth.bed.gz")
    F.multi_coverage_profile(bam["path"], bam["tiles"], bam["cs"], output_file=out, min_length=100)
    ivls = O.cleavage_intervals(bam["m"]["tiles"].splitlines(), 0, 0, bam["sizes"])
    exp = []
    for c, a, b in ivls:
        st, sp, mq, _ = tab.fetched(c, a, b).host(c)
        exp.append((c, a, DO.depth(st, sp, mq, a, b, 100).astype(np.float64)))
    assert read_gz(out) == _bedgraph(exp)


@pytest.fixture(scope="module")
def bam(tmp_path_factory, golden):
    import bam_replay as R
    from finaletoolkit_b200.io import fragments
    fragments._CACHE.clear()
    yield R.make_fixture(tmp_path_factory.mktemp("depth_bam"), golden)
    fragments._CACHE.clear()


def test_bam_fetch_semantics(bam):
    check_bam(bam)
