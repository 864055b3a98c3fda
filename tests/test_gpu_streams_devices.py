"""Every device entry point on a side stream, and on a device that is not the current one.

Each wrapper in ``device.py`` (and the pipeline and genome driver built on them) promises two things that the other
GPU tests, all on the default stream of the current device, cannot see:

* the work runs on torch's current stream of the tensors' device, so a caller can order it with its own streams
  (``pipeline.StreamedContig`` issues and graph-captures its launches on a stream of its own);
* the work runs on the device that holds the tensors, whichever device is current.

Side stream: every case puts a *decoy* in its input buffers - data of the same shape that differs only in values no
index is computed from (mapq zeroed, strand flipped, samples negated or zeroed, weights zeroed, an all-N mask), so
reading it gives wrong numbers, never a wrong address.  Then, on a fresh stream made current, the GPU sleeps, the
real input is copied into the buffers and the op runs.  A launch that escapes to an idle stream runs during that
sleep and reads the decoy.  Meanwhile the default stream sleeps longer and then writes the decoy back: a launch that
lands on the default stream runs after that, even when the op's own host work (a pageable upload synchronises its
stream) waited out the first sleep.  Either way the escaped kernel reads the decoy and fails the comparison with
the oracle, which reads the results on the default stream.

Second device (skipped with fewer than two GPUs): the kernels' shared-memory opt-in is set on each device a thread
launches on, and every case runs with all its inputs on ``cuda:1`` while ``cuda:0`` is current."""
import threading

import numpy as np
import pytest

import depth_oracle as DO
import gc_correct_oracle as GCO
import gc_oracle as GO
import spectrum_oracle as SO
import vplot_oracle as VO
from oracle import oracle as O

pytestmark = pytest.mark.gpu

CLEN = 200_000            # contig of the fragments
REF_LEN = CLEN + 5000     # the reference runs past the last fragment: no k-mer window leaves it
N_FRAG = 40_000
SLEEP_CYCLES = 1 << 26    # ~35 ms of torch.cuda._sleep on a B200: far longer than any op's launch
HOLD_CYCLES = 1 << 29     # ~0.27 s more on the default stream: longer than any op's host work after the first sleep
RTOL, ATOL = 1e-5, 1e-8   # adjust_wps, as in test_gpu_adjust.py


@pytest.fixture(scope="module")
def H():
    """Host inputs and the oracle's expectations (computed once, shared by every device and stream)."""
    from finaletoolkit_b200 import device as D
    from finaletoolkit_b200.synth import pack_twobit, synth_fragments, synth_twobit
    st, sp, mq, sd = synth_fragments(CLEN, N_FRAG, 0, seed_base=6161)
    codes, nm = synth_twobit(REF_LEN, 0, seed_base=6262, telomere=2000, n_blocks=3, block_len=3000)
    seq = np.frombuffer(b"ACGT", np.uint8)[codes].copy()
    seq[nm] = ord("N")
    edges = np.arange(5000, CLEN - 4000, 5000, dtype=np.int64)
    s, e = edges[:-1], edges[1:]
    s = np.append(s, [12_345, 150_000]); e = np.append(e, [12_346, 150_777])     # 1-bp and odd-length intervals
    order = np.argsort(s, kind="stable")
    return dict(D=D, st=st, sp=sp, mq=mq, sd=sd, codes=codes, nm=nm, seq=seq.tobytes(), ofr=O.Frags(st, sp, mq, sd),
                words=pack_twobit(codes, nm), s=s[order], e=e[order], max_len=int((sp.astype(np.int64) - st).max()),
                memo={})


def _memo(H, key, fn):
    if key not in H["memo"]:
        H["memo"][key] = fn()
    return H["memo"][key]


def _np(x):
    return x.cpu().numpy()


def _t(a, dev):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _frags(H, dev, flip_strand=False):
    """Fragments whose mapq (and, with ``flip_strand``, strand) columns hold the decoy; returns the fragments and
    the (buffer, real) pairs that restore them."""
    import torch
    mq_real, sd_real = _t(H["mq"], dev), _t(H["sd"], dev)
    mq_buf = torch.zeros_like(mq_real)
    sd_buf = (1 - sd_real) if flip_strand else sd_real.clone()
    fr = H["D"].ContigFragments(_t(H["st"], dev), _t(H["sp"], dev), mq_buf, sd_buf, device=dev, max_len=H["max_len"])
    assert fr.mapq is mq_buf and fr.strand is sd_buf
    return fr, [(mq_buf, mq_real)] + ([(sd_buf, sd_real)] if flip_strand else [])


def _ref(H, dev):
    return H["D"].PackedContig(*H["words"], REF_LEN, dev)


def _wps_exp(H):
    return _memo(H, "wps", lambda: O.wps_intervals(H["ofr"], H["s"], H["e"], CLEN, 120, 120, 180, 30, threads=4))


def _cov_hist_exp(H, n_bins):
    def f():
        cov = O.interval_coverage(H["ofr"], H["s"], H["e"], None, None, "midpoint", 30)
        hist = np.zeros(n_bins, np.int64)
        for a, b in zip(H["s"], H["e"]):
            for L, c in O.length_dist(H["ofr"], int(a), int(b), None, None, "midpoint", 30).items():
                hist[L] += c
        return cov, hist
    return _memo(H, ("cov_hist", n_bins), f)


# ---------------------------------------------------------------------------------------------------------------
# The cases: each returns (swaps, op, check).  ``swaps`` = [(buffer holding the decoy, real data)] on ``dev``;
# ``op()`` runs the entry point on the buffers; ``check(result)`` compares with the oracle.
# ---------------------------------------------------------------------------------------------------------------
def case_wps_run(H, dev):
    fr, swaps = _frags(H, dev)
    plan = H["D"].WpsPlan(H["s"], H["e"], CLEN, 180, dev)

    def check(out):
        exp, off = _wps_exp(H)
        assert np.array_equal(off, plan.offsets) and np.array_equal(_np(out).astype(np.int64), exp)
    return swaps, lambda: plan.run(fr, 120, 120, 180, 30), check


def _case_fused(H, dev, narrow):
    import torch
    fr, swaps = _frags(H, dev)
    plan = H["D"].WpsPlan(H["s"], H["e"], CLEN, 180, dev)
    n_bins = fr.max_len + 1
    out = torch.empty(plan.n_positions, dtype=torch.int16 if narrow else torch.int32, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    counts = torch.full((plan.n_intervals,), 7, dtype=torch.int64, device=dev)   # cleared by the range prepass

    def op():
        return plan.run_fused(fr, 120, 120, 180, 30, None, None, 30, n_bins=n_bins, out=out, counts=counts,
                              overflow=flag if narrow else None, zero_counts=True) + (flag,)

    def check(res):
        w, cov, hist, fl = res
        exp, _ = _wps_exp(H)
        assert int(np.abs(exp).max()) <= 32767      # the int16 output must hold this input
        exp_cov, exp_hist = _cov_hist_exp(H, n_bins)
        assert np.array_equal(_np(w).astype(np.int64), exp) and int(fl.item()) == 0
        assert np.array_equal(_np(cov), exp_cov) and np.array_equal(_np(hist), exp_hist)
    return swaps, op, check


def case_run_fused_i32(H, dev):
    return _case_fused(H, dev, False)


def case_run_fused_i16(H, dev):
    return _case_fused(H, dev, True)


def case_interval_hist(H, dev):
    D = H["D"]
    fr, swaps = _frags(H, dev)
    s, e = H["s"].tolist() + [None, 100_000], H["e"].tolist() + [30_000, None]
    nb = fr.max_len + 1

    def op():
        return [D.interval_hist(fr, s, e, "any", None, None, 30)]\
            + [D.interval_hist(fr, s, e, "midpoint", 100, 220, 30, n_bins=nb, pooled=p, first_seen=True)
               for p in (False, True, "hist")]

    def check(res):
        ofr = H["ofr"]
        assert _np(res[0][0]).tolist() == [O.single_coverage(ofr, a, b, None, None, "any", 30) for a, b in zip(s, e)]
        c1, h1, f1 = map(_np, res[1])
        for j, (a, b) in enumerate(zip(s, e)):
            exp = O.length_dist(ofr, a, b, 100, 220, "midpoint", 30)
            nz = np.flatnonzero(h1[j])
            got = {int(nz[i]): int(h1[j][nz[i]]) for i in np.argsort(f1[j][nz], kind="stable")}
            assert got == exp and list(got) == list(exp) and int(c1[j]) == sum(exp.values()), (a, b)
        c3, h3, f3 = map(_np, res[2])
        assert int(c3[0]) == int(c1.sum()) and np.array_equal(h3[0], h1.sum(0)) and np.array_equal(f3[0], f1.min(0))
        c2, h2, f2 = map(_np, res[3])
        assert np.array_equal(c2, c1) and np.array_equal(h2[0], h1.sum(0)) and np.array_equal(f2[0], f1.min(0))
    return swaps, op, check


def case_frag_lengths(H, dev):
    fr, swaps = _frags(H, dev)

    def check(got):
        assert np.array_equal(_np(got), O.frag_lengths(H["ofr"], 5000, 60_000, "midpoint", 30))
    return swaps, lambda: H["D"].frag_lengths(fr, 5000, 60_000, "midpoint", quality_threshold=30), check


def _case_motifs(H, dev, breakpoint):
    fr, swaps = _frags(H, dev, flip_strand=True)
    ref = _ref(H, dev)
    s, e = H["s"][::3], H["e"][::3]
    k = 6 if breakpoint else 4
    fn = O.region_breakpoint_motifs if breakpoint else O.region_end_motifs

    def check(got):
        got = _np(got)
        for j, (a, b) in enumerate(zip(s, e)):     # strand_mode 1: the '+' strand only, so the strand column matters
            assert np.array_equal(got[j], fn(H["ofr"], H["seq"], int(a), int(b), k, False, False, 30)), (a, b)
    return swaps, lambda: H["D"].end_motif_hist(fr, ref, s, e, k=k, strand_mode=1, quality_threshold=30,
                                                breakpoint=breakpoint), check


def case_end_motif_hist(H, dev):
    return _case_motifs(H, dev, False)


def case_breakpoint_motif_hist(H, dev):
    return _case_motifs(H, dev, True)


def case_delfi_windows(H, dev):
    fr, swaps = _frags(H, dev)
    ref = _ref(H, dev)
    ws = np.arange(0, CLEN, 40_000, dtype=np.int64)
    we = np.minimum(ws + 40_000, CLEN)
    rng = np.random.default_rng(5)
    r0 = np.sort(rng.integers(0, CLEN, 40)); r1 = np.minimum(r0 + rng.integers(1, 6000, 40), CLEN)
    order = np.lexsort((r1, r0)); blk = (r0[order], r1[order])
    gaps = ((80_000, 90_000), [(0, 3000), (CLEN - 3000, CLEN)])

    def check(got):
        got = _np(got)
        for j, (a, b) in enumerate(zip(ws, we)):
            assert np.array_equal(got[j], O.delfi_counts(H["ofr"], H["seq"], int(a), int(b), blk, gaps, 30)), (a, b)
    return swaps, lambda: H["D"].delfi_windows(fr, ref, ws, we, blacklist=blk, gaps=gaps, quality_threshold=30), check


def case_agg_signal(H, dev):
    rng = np.random.default_rng(11)
    n_seg, row_len, mws = 37, 501, 120
    rows = rng.normal(0, 50, (n_seg, row_len)).astype(np.float32)
    strands = rng.choice(["+", "-", "."], n_seg).tolist()
    real = _t(rows, dev)
    buf = -real
    code = [1 if c == "+" else -1 if c == "-" else 0 for c in strands]

    def check(got):
        assert np.array_equal(_np(got), O.agg_bw_core(list(rows), strands, mws).astype(np.float64))
    return [(buf, real)], lambda: H["D"].agg_signal(buf, code, mws // 2, row_len - mws), check


def case_adjust_segments(H, dev):
    """The rank kernel, the sliding-histogram path (``impl="hist"``), the mean and edge-subtraction variants."""
    rng = np.random.default_rng(12)
    lens = [3000, 4521, 2200]
    x = np.cumsum(rng.integers(-3, 4, sum(lens))).astype(np.int32)
    real = _t(x, dev)
    buf = -real
    runs = [dict(), dict(impl="hist"), dict(use_mean=True), dict(subtract_edges=True, edge_size=77),
            dict(use_mean=True, subtract_edges=True, edge_size=77)]

    def op():
        return [H["D"].adjust_segments(buf, lens, median_window_size=1000, **kw) for kw in runs]

    def check(res):
        off0 = np.concatenate([[0], np.cumsum(lens)])
        for kw, (got, off) in zip(runs, res):
            got = _np(got)
            for i in range(len(lens)):
                v = x[off0[i]: off0[i + 1]].astype(np.float64)
                if kw.get("subtract_edges"):
                    v = v - np.mean([np.mean(v[:77]), np.mean(v[-77:])])
                exp = O.adjust_core(v, 1000, kw.get("use_mean", False), True, 21, 2)
                np.testing.assert_allclose(got[off[i]: off[i + 1]], exp, rtol=RTOL, atol=ATOL, err_msg=f"{kw} seg {i}")
    return [(buf, real)], op, check


def case_cleavage_intervals(H, dev):
    fr, swaps = _frags(H, dev)
    s, e = H["s"], H["e"]

    def check(res):
        out, off = res
        out = _np(out)
        for k, (a, b) in enumerate(zip(s, e)):
            _, exp = O.cleavage_profile(H["ofr"], CLEN, int(a), int(b), 0, 0, None, None, 30)
            assert np.array_equal(out[off[k]: off[k + 1]], exp), (a, b)
    return swaps, lambda: H["D"].cleavage_intervals(fr, s, e, CLEN, None, None, 30), check


def case_depth_intervals(H, dev):
    fr, swaps = _frags(H, dev)
    s, e = H["s"], H["e"]

    def check(res):
        for midpoint, (got, off) in zip((False, True), res):
            exp, eoff = DO.depth_intervals(H["st"], H["sp"], H["mq"], s, e, 100, 220, 30, midpoint)
            assert np.array_equal(off, eoff) and np.array_equal(_np(got).astype(np.int64), exp), midpoint
    return swaps, lambda: [H["D"].depth_intervals(fr, s, e, CLEN, 100, 220, 30, m) for m in (False, True)], check


def _sites():
    c = np.array([5000, 31_337, 100_000, 100_001, 150_500, CLEN - 10], np.int64)
    return c, (np.arange(c.size) % 2).astype(bool)


def case_vplot_sites(H, dev):
    fr, swaps = _frags(H, dev)
    c, flip = _sites()

    def check(got):
        exp = VO.vplot(H["st"], H["sp"], H["mq"], c, flip, 500, 100, 220, 30)
        assert exp.sum() > 0 and np.array_equal(_np(got), exp)
    return swaps, lambda: H["D"].vplot_sites(fr, c, flip, 500, 100, 220, 30), check


_GC_LO, _GC_HI = 100, 220
_REGS = (np.array([0, 20_000, 90_000, 160_000], np.int64), np.array([12_000, 60_000, 91_000, REF_LEN], np.int64))


def case_gc_observed(H, dev):
    fr, swaps = _frags(H, dev)
    ref = _ref(H, dev)

    def check(got):
        exp = GO.observed(H["st"], H["sp"], H["mq"], H["codes"], H["nm"], REF_LEN, *_REGS, _GC_LO, _GC_HI, 30)
        assert exp.sum() > 0 and np.array_equal(_np(got), exp)
    return swaps, lambda: H["D"].gc_observed(fr, ref, *_REGS, _GC_LO, _GC_HI, 30), check


def case_gc_expected(H, dev):
    """Decoy: an N mask that covers every base (no placement counts)."""
    real = _ref(H, dev)
    decoy = H["D"].PackedContig(H["words"][0], np.full_like(H["words"][1], 0xFFFFFFFF), REF_LEN, dev)

    def check(got):
        exp = _memo(H, "gc_expected", lambda: GO.expected(H["codes"], H["nm"], REF_LEN, *_REGS, _GC_LO, _GC_HI))
        assert exp.sum() > 0 and np.array_equal(_np(got), exp)
    return [(decoy.nmask, real.nmask)], lambda: H["D"].gc_expected(decoy, *_REGS, _GC_LO, _GC_HI), check


def _weights(dev):
    import torch
    rng = np.random.default_rng(13)
    W = rng.uniform(0.25, 4.0, (_GC_HI - _GC_LO + 1, _GC_HI + 1))
    real = _t(W, dev)
    return W, torch.zeros_like(real), real


def case_gc_weighted_intervals(H, dev):
    fr, _ = _frags(H, dev)
    fr.mapq.copy_(_t(H["mq"], dev))
    ref = _ref(H, dev)
    W, buf, real = _weights(dev)
    s, e = H["s"], H["e"]

    def check(res):
        count, corr = map(_np, res)
        ec, er = GCO.intervals(H["st"], H["sp"], H["mq"], H["codes"], H["nm"], REF_LEN, s, e, W, _GC_LO, _GC_HI, 30)
        assert np.array_equal(count, ec) and er.sum() > 0
        np.testing.assert_allclose(corr, er, rtol=1e-12, atol=0)
    return [(buf, real)], lambda: H["D"].gc_weighted_intervals(fr, ref, s, e, buf, _GC_LO, _GC_HI, 30), check


def case_gc_weighted_sites(H, dev):
    fr, _ = _frags(H, dev)
    fr.mapq.copy_(_t(H["mq"], dev))
    ref = _ref(H, dev)
    W, buf, real = _weights(dev)
    c, flip = _sites()

    def check(res):
        count, corr = map(_np, res)
        ec, er = GCO.sites(H["st"], H["sp"], H["mq"], H["codes"], H["nm"], REF_LEN, c, flip, 500, W, _GC_LO, _GC_HI, 30)
        assert np.array_equal(count, ec) and er.sum() > 0
        np.testing.assert_allclose(corr, er, rtol=1e-12, atol=0)
    return [(buf, real)], lambda: H["D"].gc_weighted_sites(fr, ref, c, flip, 500, buf, _GC_LO, _GC_HI, 30), check


def _case_spectrum(H, dev, dtype):
    """Decoy: zeros (a periodogram cannot tell a series from its negation)."""
    import torch
    rng = np.random.default_rng(14)
    lens = [0, 1, 150, 1999, 10_000]
    x = (rng.integers(-1000, 1000, sum(lens)) if dtype == "i32" else rng.normal(0, 30, sum(lens)))
    x = x.astype(np.int32 if dtype == "i32" else np.float64)
    off = np.concatenate([[0], np.cumsum(lens)])
    real = _t(x, dev)
    buf = torch.zeros_like(real)

    def check(got):
        got = _np(got)
        for i in range(len(lens)):
            SO.check_row(got[i], x[off[i]: off[i + 1]], 120, 280)
    return [(buf, real)], lambda: H["D"].spectrum_segments(buf, off, 120, 280), check


def case_spectrum_i32(H, dev):
    return _case_spectrum(H, dev, "i32")


def case_spectrum_f64(H, dev):
    return _case_spectrum(H, dev, "f64")


def case_packed_unpack(H, dev):
    """``PackedFragments.to_device`` (H2D of the packed words + the unpack kernel), and the unpack kernel alone on
    device words that hold the packing of the same fragments with mapq zeroed and strand flipped."""
    import torch
    from finaletoolkit_b200.packed import PACK_BLOCK, PackedFragments
    pk = PackedFragments(H["st"], H["sp"], H["mq"], H["sd"])
    bad = PackedFragments(H["st"], H["sp"], np.zeros_like(H["mq"]), 1 - H["sd"])
    assert (bad.record_bytes, bad.n_raw) == (pk.record_bytes, pk.n_raw) and not torch.equal(bad.words, pk.words)
    real_w, real_a = pk.words.to(dev), pk.anchors.to(dev)
    buf_w, buf_a = bad.words.to(dev), bad.anchors.to(dev)
    raw = pk.raw_to_device(dev)
    n = pk.n
    npad = max(pk.n_blocks * PACK_BLOCK, 2)
    cols = [torch.empty(npad, dtype=dt, device=dev) for dt in (torch.int32, torch.int32, torch.uint8, torch.uint8)]

    def op():
        fr = pk.to_device(dev)
        pk.unpack_into(buf_w, buf_a, raw, n, *cols, dev)
        return fr.start, fr.stop, fr.mapq, fr.strand, *(c[:n] for c in cols)

    def check(res):
        exp = (H["st"], H["sp"], H["mq"], H["sd"])
        for got, want in zip(res, exp + exp):
            assert np.array_equal(_np(got), want)
    return [(buf_w, real_w), (buf_a, real_a)], op, check


def case_streamed_contig(H, dev):
    """Eager pass, graph capture + replay, and a second replay; the decoy sits in the pinned host outputs, so a
    result read before the pass drained into them fails."""
    from finaletoolkit_b200.packed import PackedFragments
    from finaletoolkit_b200.pipeline import StreamedContig
    pipe = StreamedContig(None, None, None, H["s"], H["e"], CLEN, 120, 120, 180, 30, n_chunks=3, device=dev,
                          packed=PackedFragments(H["st"], H["sp"], H["mq"], H["sd"]))

    def op():
        out = []
        for _ in range(3):
            pipe.h_wps.fill_(-9999); pipe.h_cov.fill_(-1); pipe.h_hist.fill_(-1)
            w, c, h, tot = pipe.run()
            out.append((w.numpy().copy(), c.numpy().copy(), h.numpy().copy(), int(tot[0])))
        assert pipe._graph is not None
        return out

    def check(res):
        exp, _ = _wps_exp(H)
        exp_cov, exp_hist = _cov_hist_exp(H, pipe.n_bins)
        for w, c, h, tot in res:
            assert np.array_equal(w[: pipe.n_positions].astype(np.int64), exp)
            assert np.array_equal(c[: pipe.n_ivl], exp_cov) and np.array_equal(h[0], exp_hist)
            assert tot == int(exp_cov.sum())
    return [], op, check


def case_multi_wps_genome(H, dev):
    """The genome driver over one contig, with adjustment; the decoy goes into the fragment columns of the shard it
    built on a first call."""
    from finaletoolkit_b200.distributed import multi_wps_genome
    from finaletoolkit_b200.io.fragments import FragmentTable
    import torch
    table = FragmentTable({"a": (H["st"], H["sp"], H["mq"], H["sd"])})
    sites = {"a": (H["s"], H["e"])}
    adjust = dict(median_window_size=1000)
    plans = {}

    def run():
        return multi_wps_genome(table, [("a", CLEN)], sites, 5000, 120, 120, 180, 30, coverage=True, length_hist=True,
                                adjust=adjust, device=dev, contigs=["a"], reduce=False, plans=plans)
    with torch.cuda.device(dev):
        run()
        torch.cuda.synchronize()
    (g,) = next(iter(plans.values())).groups
    real = g.frags.mapq.clone()
    g.frags.mapq.zero_()

    def check(res):
        r, hist, total = res
        r = r["a"]
        exp, off = _wps_exp(H)
        exp_cov, exp_hist = _cov_hist_exp(H, hist.numel())
        assert np.array_equal(_np(r.wps).astype(np.int64), exp) and np.array_equal(_np(r.cov), exp_cov)
        assert np.array_equal(_np(hist), exp_hist) and total == int(exp_cov.sum())
        adj = _np(r.adjusted)
        n_adj = 0
        for i in range(len(H["s"])):
            a0, a1 = r.adj_offsets[i], r.adj_offsets[i + 1]
            if a1 > a0:
                ref = O.adjust_core(exp[off[i]: off[i + 1]].astype(np.float64), 1000, False, True, 21, 2)
                np.testing.assert_allclose(adj[a0:a1], ref, rtol=RTOL, atol=ATOL, err_msg=str(i))
                n_adj += 1
        assert n_adj >= 30
    return [(g.frags.mapq, real)], run, check


CASES = {name[5:]: fn for name, fn in globals().items() if name.startswith("case_")}


def _cuda_tensors(res):
    import torch
    if torch.is_tensor(res):
        return [res] if res.is_cuda else []
    if isinstance(res, (list, tuple)):
        return [x for r in res for x in _cuda_tensors(r)]
    if isinstance(res, dict):
        return [x for r in res.values() for x in _cuda_tensors(r)]
    if hasattr(res, "__slots__"):       # distributed.ContigWps
        return [x for k in res.__slots__ for x in _cuda_tensors(getattr(res, k, None))]
    return []


# ---------------------------------------------------------------------------------------------------------------
# A. A side stream of one GPU
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(CASES))
def test_side_stream(H, name):
    import torch
    dev = H["D"].require_cuda("cuda:0")
    swaps, op, check = CASES[name](H, dev)
    decoys = [buf.clone() for buf, _ in swaps]
    if swaps:       # a first call on the real input loads the kernels: a lazy module load waits for the whole device
        for buf, real in swaps:
            buf.copy_(real)
        check(op())
        for (buf, _), decoy in zip(swaps, decoys):
            buf.copy_(decoy)
    torch.cuda.synchronize()
    torch.cuda._sleep(SLEEP_CYCLES + HOLD_CYCLES)       # the default stream: whatever lands there waits,
    for (buf, _), decoy in zip(swaps, decoys):          # then finds the decoy back in the buffers
        buf.copy_(decoy)
    side = torch.cuda.Stream(dev)
    with torch.cuda.stream(side):
        torch.cuda._sleep(SLEEP_CYCLES)
        for buf, real in swaps:
            buf.copy_(real)
        res = op()
    side.synchronize()
    check(res)                                          # reads on the default stream
    torch.cuda.synchronize()


def test_big_upload_on_a_side_stream(H):
    """Columns of 8 MB and more go through the reusable pinned staging buffers, with the copy on the current stream;
    three such uploads make the first buffer wait for its copy before it is reused."""
    import torch
    D = H["D"]
    dev = D.require_cuda("cuda:0")
    rng = np.random.default_rng(15)
    n = 3 << 20                                      # 12 MB int32 columns
    st = np.sort(rng.integers(0, 1 << 30, n)).astype(np.int32)
    sp = st + rng.integers(0, 600, n).astype(np.int32)
    third = rng.integers(-5, 5, n).astype(np.int32)
    torch.cuda.synchronize()
    side = torch.cuda.Stream(dev)
    with torch.cuda.stream(side):
        torch.cuda._sleep(SLEEP_CYCLES)
        fr = D.ContigFragments(st, sp, device=dev)
        x = D._to_device(third, dev, np.int32)
        got = [t.cpu() for t in (fr.start, fr.stop, x)]     # D2H on the side stream, after the uploads
    side.synchronize()
    assert "cuda:0" in D._STAGING
    for g, want in zip(got, (st, sp, third)):
        assert np.array_equal(g.numpy(), want)


# ---------------------------------------------------------------------------------------------------------------
# B. A second GPU
# ---------------------------------------------------------------------------------------------------------------
def _two_gpus():
    import torch
    return torch.cuda.is_available() and torch.cuda.device_count() >= 2


needs_two = pytest.mark.skipif(not _two_gpus(), reason="needs two CUDA devices")


@needs_two
def test_shared_memory_opt_in_on_each_device(H):
    """One host thread runs the kernels that need more than 48 KB of dynamic shared memory (the persistent WPS
    kernel, plain and fused, and the sliding-histogram adjust kernel) on device 0, then moves to device 1 and runs
    them again there: the opt-in must be made on each device.  A fresh thread, so that no earlier test has made it."""
    import torch
    D = H["D"]
    x = np.cumsum(np.random.default_rng(16).integers(-3, 4, 6000)).astype(np.int32)
    errors, results = [], {}

    def body():
        try:
            for d in (0, 1):
                torch.cuda.set_device(d)
                dev = torch.device("cuda", d)
                fr = D.ContigFragments(H["st"], H["sp"], H["mq"], H["sd"], device=dev)
                plan = D.WpsPlan(H["s"], H["e"], CLEN, 180, dev)
                w1 = plan.run(fr, 120, 120, 180, 30)
                w2, cov, hist = plan.run_fused(fr, 120, 120, 180, 30, None, None, 30, n_bins=fr.max_len + 1)
                adj, off = D.adjust_segments(_t(x, dev), [6000], median_window_size=1000, impl="hist")
                torch.cuda.synchronize(dev)
                results[d] = [_np(v) for v in (w1, w2, cov, hist, adj)] + [off]
        except BaseException as exc:     # re-raised on the test's thread
            errors.append(exc)

    th = threading.Thread(target=body)
    th.start()
    th.join()
    if errors:
        raise errors[0]
    exp, _ = _wps_exp(H)
    exp_cov, exp_hist = _cov_hist_exp(H, int(H["max_len"]) + 1)
    exp_adj = O.adjust_core(x.astype(np.float64), 1000, False, True, 21, 2)
    for d in (0, 1):
        w1, w2, cov, hist, adj, off = results[d]
        assert np.array_equal(w1.astype(np.int64), exp) and np.array_equal(w2.astype(np.int64), exp), d
        assert np.array_equal(cov, exp_cov) and np.array_equal(hist, exp_hist), d
        np.testing.assert_allclose(adj[off[0]: off[1]], exp_adj, rtol=RTOL, atol=ATOL, err_msg=str(d))


@needs_two
@pytest.mark.parametrize("name", sorted(CASES))
def test_non_current_device(H, name):
    """Every input on cuda:1 while cuda:0 is current: the work runs on cuda:1, results stay there and cuda:0 stays
    current."""
    import torch
    dev = torch.device("cuda", 1)
    with torch.cuda.device(0):
        swaps, op, check = CASES[name](H, dev)
        for buf, real in swaps:
            buf.copy_(real)
        res = op()
        assert torch.cuda.current_device() == 0
    torch.cuda.synchronize(dev)
    assert all(x.device == dev for x in _cuda_tensors(res)), name
    check(res)


@needs_two
def test_adjust_plan_on_another_device_is_refused():
    import torch
    from finaletoolkit_b200.device import AdjustPlan, adjust_segments
    x = torch.arange(3000, dtype=torch.int32, device="cuda:0")
    plan = AdjustPlan([3000], 1000, device="cuda:1")
    with pytest.raises(ValueError, match="one device"):
        adjust_segments(x, None, plan=plan)
