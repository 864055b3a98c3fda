"""Fused pass (WPS + per-interval coverage + pooled length histogram in one sweep over the fragments,
``ftk_wps_cov_tiles``) vs the CPU oracle and vs the separate kernels; the fused (six-group) and the plain
(two-group) shape of the WPS kernel must give identical scores."""
import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    from finaletoolkit_b200.device import require_cuda
    return require_cuda("cuda:0")


def _oracle_hist(ofr, ivs, lo, hi, q, n_bins):
    h = np.zeros(n_bins, np.int64)
    for s, e in ivs:
        for L, c in O.length_dist(ofr, s, e, lo, hi, "midpoint", q).items():
            if L < n_bins:
                h[L] += c
    return h


@pytest.mark.parametrize("seed", range(8))
def test_fused_random_vs_oracle(seed, dev):
    import torch
    from finaletoolkit_b200.device import ContigFragments, WpsPlan
    from finaletoolkit_b200.synth import synth_fragments
    rng = np.random.default_rng(100 + seed)
    clen = int(rng.integers(30_000, 150_000))
    n = int(rng.integers(1, 60_000)) if seed else 0
    st, sp, mq, sd = synth_fragments(clen, n, seed, seed_base=777)
    if n:
        # long outliers (> 1024: global-atomic bins), zero-length rows, a pile-up, rows past the contig end
        k = max(1, n // 200)
        idx = rng.choice(n, k, replace=False)
        sp[idx] = st[idx] + rng.integers(600, 3000, k).astype(np.int32)
        z = rng.choice(n, max(1, n // 500), replace=False)
        sp[z] = st[z]
        st[: n // 20] = st[0]
        sp[: n // 20] = st[0] + rng.integers(100, 200, n // 20).astype(np.int32)
        order = np.argsort(st, kind="stable"); st, sp, mq, sd = st[order], sp[order], mq[order], sd[order]
    ofr = O.Frags(st, sp, mq, sd)
    dfr = ContigFragments(st, sp, mq, sd, device=dev)
    W = int(rng.choice([2, 59, 120, 121, 200]))
    lo = int(rng.choice([0, 30, 120])); hi = int(lo + rng.choice([0, 60, 450]))
    q = int(rng.choice([0, 30, 60]))
    c_lo = [None, 0, 100, 150][int(rng.integers(0, 4))]
    c_hi = [None, 220, 167, 5000][int(rng.integers(0, 4))]
    cq = int(rng.choice([0, 20, 30, 61]))
    ivs = [(0, 5000), (5000, 10_000), (10_000, 10_000), (10_000, 22_345), (clen - 4000, clen), (clen - 10, clen + 50)]
    for _ in range(8):
        s = int(rng.integers(0, clen)); ivs.append((s, min(s + int(rng.integers(1, 13_000)), clen + 100)))
    n_bins = int(rng.choice([0, 601, 1024, 2500]))
    plan = WpsPlan([s for s, _ in ivs], [e for _, e in ivs], clen, hi, dev)
    for dt in (torch.int32, torch.int16):
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        out = torch.empty(max(plan.n_positions, 1), dtype=dt, device=dev)
        wps, cnt, hist = plan.run_fused(dfr, W, lo, hi, q, c_lo, c_hi, cq, n_bins=n_bins, out=out, overflow=flag)
        torch.cuda.synchronize()
        host = wps.cpu().numpy().astype(np.int64)
        if dt == torch.int16 and int(flag.item()):
            continue   # a > 32767-deep pile-up: the caller reruns in int32 (covered above)
        for i, (s, e) in enumerate(ivs):
            exp = O.wps_interval(ofr, s, e, clen, W, lo, hi, q)
            assert np.array_equal(host[plan.offsets[i]:plan.offsets[i + 1]], exp), (seed, W, lo, hi, q, s, e)
        live = [(s, e) for s, e in ivs if e > s]
        exp_cov = O.interval_coverage(ofr, [s for s, _ in ivs], [e for _, e in ivs], c_lo, c_hi, "midpoint", cq)
        exp_cov[[i for i, (s, e) in enumerate(ivs) if e <= s]] = 0   # a degenerate interval owns no tile
        assert np.array_equal(cnt.cpu().numpy(), exp_cov), (seed, c_lo, c_hi, cq)
        if n_bins:
            assert np.array_equal(hist.cpu().numpy(), _oracle_hist(ofr, live, c_lo, c_hi, cq, n_bins)), (seed, n_bins)


def test_fused_equals_plain_and_separate_kernels(dev):
    """3 M fragments: fused pass (six groups) == WpsPlan.run (plain, two groups) + interval_hist(pooled='hist')."""
    import torch
    from finaletoolkit_b200 import device as D
    from finaletoolkit_b200.synth import synth_fragments
    clen, n = 10_000_000, 3_200_000
    st, sp, mq, sd = synth_fragments(clen, n, 7)
    fr = D.ContigFragments(st, sp, mq, sd, device=dev)
    edges = np.arange(0, clen + 5000, 5000).clip(max=clen)
    plan = D.WpsPlan(edges[:-1], edges[1:], clen, 180, dev)
    n_bins = fr.max_len + 1
    wps, cnt, hist = plan.run_fused(fr, 120, 120, 180, 30, None, None, 30, n_bins=n_bins)
    ivl = D.IntervalSet(edges[:-1].tolist(), edges[1:].tolist(), dev)
    c2 = torch.zeros(ivl.n, dtype=torch.int64, device=dev); h2 = torch.zeros((1, n_bins), dtype=torch.int64, device=dev)
    D.interval_hist(fr, intersect_policy="midpoint", quality_threshold=30, n_bins=n_bins, pooled="hist", ivl_set=ivl,
                    out=(c2, h2, None))
    plain = plan.run(fr, 120, 120, 180, 30)
    torch.cuda.synchronize()
    assert torch.equal(wps, plain)
    assert torch.equal(cnt, c2) and torch.equal(hist, h2[0])
    # odd window + int8 output through the fused entry
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    o8 = torch.empty(plan.n_positions, dtype=torch.int8, device=dev)
    w8, cnt8, _ = plan.run_fused(fr, 121, 120, 180, 30, 100, 220, 0, n_bins=0, out=o8, overflow=flag)
    ref = plan.run(fr, 121, 120, 180, 30)
    c3, _, _ = D.interval_hist(fr, edges[:-1].tolist(), edges[1:].tolist(), "midpoint", 100, 220, 0)
    assert int(flag.item()) == 0 and torch.equal(w8.to(torch.int32), ref) and torch.equal(cnt8, c3)


def test_fused_few_tiles_and_accumulation(dev):
    """Fewer tiles than consumer groups; counts / hist accumulate across calls (two contigs, one buffer)."""
    import torch
    from finaletoolkit_b200.device import ContigFragments, WpsPlan
    from finaletoolkit_b200.synth import synth_fragments
    clen = 20_000
    st, sp, mq, sd = synth_fragments(clen, 5000, 1, seed_base=9)
    fr = ContigFragments(st, sp, mq, sd, device=dev); ofr = O.Frags(st, sp, mq, sd)
    for ivs in ([(100, 4000)], [(0, 5000), (5000, 9000), (9000, 9001)]):
        plan = WpsPlan([s for s, _ in ivs], [e for _, e in ivs], clen, 180, dev)
        cnt = torch.zeros(len(ivs), dtype=torch.int64, device=dev); hist = torch.zeros(700, dtype=torch.int64, device=dev)
        for _ in range(2):
            wps, _, _ = plan.run_fused(fr, n_bins=700, counts=cnt, hist=hist)
        exp = O.interval_coverage(ofr, [s for s, _ in ivs], [e for _, e in ivs], None, None, "midpoint", 30)
        assert np.array_equal(cnt.cpu().numpy(), 2 * exp)
        assert np.array_equal(hist.cpu().numpy(), 2 * _oracle_hist(ofr, ivs, None, None, 30, 700))
        host = wps.cpu().numpy()
        for i, (s, e) in enumerate(ivs):
            assert np.array_equal(host[plan.offsets[i]:plan.offsets[i + 1]], O.wps_interval(ofr, s, e, clen))


def test_fused_zero_length_rows_on_tile_and_interval_starts(dev):
    """tabix overlap (stop > S): a zero-length row ON an interval's start is outside its stream, the same
    row on an interior tile boundary of a longer interval is inside."""
    import torch
    from finaletoolkit_b200.device import ContigFragments, WpsPlan
    clen = 30_000
    st = np.array([0, 0, 4000, 4000, 4000, 8000, 11_999, 12_000, 12_000], np.int32)
    sp = st + np.array([0, 150, 0, 0, 160, 0, 0, 0, 1], np.int32)
    mq = np.full(st.size, 60, np.uint8)
    fr = ContigFragments(st, sp, mq, None, device=dev); ofr = O.Frags(st, sp, mq, np.ones(st.size, np.uint8))
    ivs = [(0, 12_000), (4000, 8000), (12_000, 12_500)]
    plan = WpsPlan([s for s, _ in ivs], [e for _, e in ivs], clen, 180, dev)
    assert plan.n_tiles == 3 + 1 + 1
    _, cnt, hist = plan.run_fused(fr, cov_quality_threshold=0, n_bins=200)
    exp = O.interval_coverage(ofr, [s for s, _ in ivs], [e for _, e in ivs], None, None, "midpoint", 0)
    assert cnt.cpu().tolist() == exp.tolist() == [6, 1, 1]
    assert int(hist[0]) == 4 + 0 + 0 and int(hist.sum()) == 8
