"""Interval kernels give the same result whatever the number of slices each interval's candidate range is split into.

Each (interval, split) unit streams a slice that starts at an arbitrary fragment index, widened left to a 16-byte
boundary; the lanes left of the slice must not be counted.  The intervals below have candidate ranges starting at
every residue mod 4, and 1000 splits make many slices shorter than one vector or empty.
"""
import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu

SPLITS = (1, 2, 3, 7, 1000)


@pytest.fixture(scope="module")
def data():
    from finaletoolkit_b200 import device as D
    from finaletoolkit_b200.synth import synth_fragments, synth_twobit
    dev = D.require_cuda("cuda:0")
    clen, n = 400_000, 160_000
    st, sp, mq, sd = synth_fragments(clen, n, 3, seed_base=2024)
    keep = sp <= clen   # end motifs: the reference raises on a fragment ending past the contig
    st, sp, mq, sd = st[keep], sp[keep], mq[keep], sd[keep]
    codes, nm = synth_twobit(clen, 3, seed_base=2025, telomere=600, block_len=2500)
    seq = np.frombuffer(b"ACGT", np.uint8)[codes].copy(); seq[nm] = ord("N")
    fr = D.ContigFragments(st, sp, mq, sd, device=dev)
    rng = np.random.default_rng(7)
    starts = rng.integers(0, clen - 30_000, 48)
    ivs = [(int(s), int(s + rng.integers(1, 30_000))) for s in starts] + [(0, clen), (5, 6), (clen - 1000, clen)]
    # the candidate ranges (lower bound of start - max_frag_len) start at every residue mod 4
    assert set(np.searchsorted(st, [a - fr.max_len for a, _ in ivs]) % 4) == {0, 1, 2, 3}
    return dict(D=D, clen=clen, fr=fr, ofr=O.Frags(st, sp, mq, sd), seq=seq.tobytes(),
                ref=D.PackedContig.from_codes(codes, nm, device=dev), ivs=ivs)


@pytest.fixture(params=SPLITS)
def splits(request, monkeypatch):
    from finaletoolkit_b200 import device as D
    monkeypatch.setattr(D, "_splits_for", lambda *a, **k: request.param)
    return request.param


def _np(x):
    return None if x is None else x.cpu().numpy()


def test_interval_hist_slices(data, splits):
    D, fr, ofr = data["D"], data["fr"], data["ofr"]
    ivs = data["ivs"] + [(None, 50_000), (120_000, None), (None, None)]
    s, e = [a for a, _ in ivs], [b for _, b in ivs]
    nb = fr.max_len + 1
    for pol, lo, hi, q in [("midpoint", None, None, 30), ("any", 100, 220, 0)]:
        cnt = _np(D.interval_hist(fr, s, e, pol, lo, hi, q)[0])
        assert cnt.tolist() == [O.single_coverage(ofr, a, b, lo, hi, pol, q) for a, b in ivs], (pol, splits)
        c1, h1, f1 = map(_np, D.interval_hist(fr, s, e, pol, lo, hi, q, n_bins=nb, first_seen=True))
        assert np.array_equal(c1, cnt)
        for j, (a, b) in enumerate(ivs):
            exp = O.length_dist(ofr, a, b, lo, hi, pol, q)
            nz = np.flatnonzero(h1[j])
            got = {int(nz[i]): int(h1[j][nz[i]]) for i in np.argsort(f1[j][nz], kind="stable")}
            assert got == exp and list(got) == list(exp), (pol, a, b, splits)
        c2, h2, f2 = map(_np, D.interval_hist(fr, s, e, pol, lo, hi, q, n_bins=nb, pooled="hist", first_seen=True))
        assert np.array_equal(c2, cnt) and np.array_equal(h2[0], h1.sum(0)) and np.array_equal(f2[0], f1.min(0))


def test_delfi_windows_slices(data, splits):
    D, fr, ofr, clen = data["D"], data["fr"], data["ofr"], data["clen"]
    ivs = data["ivs"]
    rng = np.random.default_rng(11)
    r0 = np.sort(rng.integers(0, clen, 80)); r1 = r0 + rng.integers(1, 20_000, 80)
    order = np.lexsort((r1, r0)); blk = (r0[order], r1[order])
    gaps = ((clen // 2, clen // 2 + 3000), [(0, 700), (clen - 700, clen)])
    got = _np(D.delfi_windows(fr, data["ref"], [a for a, _ in ivs], [b for _, b in ivs], blacklist=blk, gaps=gaps,
                              quality_threshold=30))
    for j, (a, b) in enumerate(ivs):
        assert np.array_equal(got[j], O.delfi_counts(ofr, data["seq"], a, b, blk, gaps, 30)), (a, b, splits)


@pytest.mark.parametrize("breakpoint", [False, True])
def test_end_motif_hist_slices(data, splits, breakpoint):
    D, fr, ofr = data["D"], data["fr"], data["ofr"]
    ivs = data["ivs"]
    k = 6 if breakpoint else 4
    got = _np(D.end_motif_hist(fr, data["ref"], [a for a, _ in ivs], [b for _, b in ivs], k=k, strand_mode=0,
                               quality_threshold=30, breakpoint=breakpoint))
    ref_fn = O.region_breakpoint_motifs if breakpoint else O.region_end_motifs
    for j, (a, b) in enumerate(ivs):
        assert np.array_equal(got[j], ref_fn(ofr, data["seq"], a, b, k, True, False, 30)), (a, b, splits)
