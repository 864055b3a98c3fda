"""adjust_segments, every kernel instantiation, against exact arithmetic.

What each check expects (u = 2^-53, the unit roundoff of fp64):

- Median windows before smoothing, on any path: bit for bit the reference's operations, ``xs = x - shift`` and then
  ``xs[w//2 : n - w//2] - np.median(sliding_window_view(xs, w)[:n - w], axis=1)``, with the shift the GPU computed.
  The kernels do the same fp64 operations in the same order (median of an even window = (lo + hi) / 2).
- The shift ``mean(mean(x[:e]), mean(x[-e:]))`` with Python's slice semantics for every ``e``: bit for bit for
  integer-valued samples, otherwise within ``shift_bound`` of the exact rational value.
- Mean windows: within ``mean_bound`` of the exact ``c - sum(x_i) / w`` (a shift cancels mathematically).
- Smoothing: ``savgol_oracle.check_smoothed``, the exact hat matrix applied to the same call's unsmoothed series.
- NaN samples (generic kernel): exactly the windows, and the smoothed outputs, that touch one are NaN.

A recorder around ``device._launch`` asserts which entry point and mode each case ran, and the last test that every
kernel instantiation was reached by the cases of this file."""
import warnings
from fractions import Fraction

import numpy as np
import pytest
from numpy.lib.stride_tricks import sliding_window_view

from savgol_oracle import check_smoothed

pytestmark = pytest.mark.gpu

U = np.finfo(np.float64).eps / 2

REACHED = set()                    # kernel instantiations the cases of this module launched


def _mom(sg_w, a, b, den):
    """The exact sliding-moment smoothing condition of ``ftk_adjust_rank_f64``."""
    if sg_w <= 0 or den == 0:
        return False
    h = sg_w >> 1
    s2 = h * (h + 1) * (2 * h + 1) // 3
    aa, bb = abs(a), abs(b)
    return ((s2 + 2 * h * (h + 1) + sg_w + 2 * (h + 1) ** 2) * (1 << 17) < (1 << 31) and aa < (1 << 31)
            and bb < (1 << 31) and aa * sg_w + bb * s2 < (1 << 36))


def _instantiation(name, args):
    """The kernel template instance a C-ABI call launches, from its arguments."""
    if name == "ftk_adjust_rank_f64":
        in_t = "int" if args[1] else "float"
        shift, sg_w = bool(args[4]), int(args[11])
        sgw = -1 if sg_w == 0 else 21 if sg_w == 21 else 0
        mom = (not shift) and _mom(sg_w, *args[15:18])
        return ("rank", in_t, shift, sgw, mom)
    if name == "ftk_adjust_wps_f64":
        return ("hist", bool(args[8]), bool(args[4]))              # <MEAN, SHIFT>
    if name == "ftk_adjust_wps_generic_f64":
        return ("generic", bool(args[9]), bool(args[4]))           # (mean, shift)
    if name == "ftk_savgol_f64":
        return ("savgol", 21 if int(args[4]) == 21 else 0)
    if name == "ftk_adjust_edge_shift_f64":
        return ("edge_shift",)
    return (name,)


ALL = ({("rank", t, True, s, False) for t in ("float", "int") for s in (21, 0, -1)}
       | {("rank", t, False, s, True) for t in ("float", "int") for s in (21, 0)}
       | {("rank", t, False, s, False) for t in ("float", "int") for s in (21, 0, -1)}
       | {("hist", m, s) for m in (False, True) for s in (False, True)}
       | {("generic", m, s) for m in (False, True) for s in (False, True)}
       | {("savgol", 21), ("savgol", 0), ("edge_shift",)})


@pytest.fixture
def rec(monkeypatch):
    """Calls to ``device._launch`` since the last ``rec.clear()``: ``(instantiation, name, args)``."""
    from finaletoolkit_b200 import device
    real = device._launch
    calls = []

    def launch(dev, name, *args):
        calls.append((_instantiation(name, args), name, args))
        REACHED.add(_instantiation(name, args))
        return real(dev, name, *args)

    monkeypatch.setattr(device, "_launch", launch)
    return calls


def kinds(calls):
    return [k for k, _, _ in calls]


def generic_runs(calls):
    """(flagged runs handed to the generic kernel, runs of the histogram kernel) of the last call."""
    n_list = sum(int(a[7]) for _, n, a in calls if n == "ftk_adjust_wps_generic_f64")
    n_runs = sum(int(a[6]) for _, n, a in calls if n == "ftk_adjust_wps_f64")
    return n_list, n_runs


@pytest.fixture(scope="module")
def dev():
    from finaletoolkit_b200.device import require_cuda
    return require_cuda("cuda:0")


def run(rec, x, lens, dev, **kw):
    """adjust_segments on float32 numpy input, or an int32 CUDA tensor when ``x`` is an integer array;
    returns (host output, out_off, launches of this call)."""
    import torch
    from finaletoolkit_b200.device import adjust_segments
    rec.clear()
    xin = torch.from_numpy(np.asarray(x, np.int32)).to(dev) if np.asarray(x).dtype.kind == "i" else np.asarray(x, np.float32)
    out, off = adjust_segments(xin, lens, **kw)
    return out.cpu().numpy(), off, list(rec)


def gpu_shift(x, lens, edge, dev):
    """The per-segment shift ``ftk_adjust_edge_shift_f64`` computes (what ``subtract_edges`` subtracts)."""
    import torch
    from finaletoolkit_b200 import device
    xf = torch.from_numpy(np.asarray(x, np.float32)).to(dev)
    seg = torch.from_numpy(np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)).to(dev)
    sh = torch.empty(len(lens), dtype=torch.float64, device=dev)
    device._launch(dev, "ftk_adjust_edge_shift_f64", xf.data_ptr(), seg.data_ptr(), len(lens), int(edge), sh.data_ptr())
    return sh.cpu().numpy()


def np_shift(x, e):
    """The reference's expression, on the float64 samples."""
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)        # mean of an empty slice
        return np.mean([np.mean(x[:e]), np.mean(x[-e:])])


def median_ref(x, w, shift):
    """The reference's median adjustment of one segment (float64 samples), in chunks of windows."""
    xs = np.asarray(x, np.float64) - shift
    n, h = xs.size, w // 2
    med = np.empty(max(n - w, 0))
    step = max(1, (1 << 23) // w)
    view = sliding_window_view(xs, w)[: n - w]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)        # inf - inf inside np.median
        for a in range(0, n - w, step):
            med[a: a + step] = np.median(view[a: a + step], axis=1)
        return xs[h: n - h] - med


def mean_bound(x, w, shift, hist_bins=256):
    """``|out - (c - sum x_i / w)|`` for every output, in both mean kernels.

    Generic kernel: ``t_i = fl(x_i - s)``, a left-to-right sum, ``/ w``, ``fl(c - s) - stat``: the terms are off
    by ``u |x_i - s|``, the sum by ``gamma_{w-1} sum |t_i|``, the quotient, the centre and the difference by one
    ``u`` each, so ``<= (w + 2) u (|c - s| + sum |x_i - s| / w)`` to first order.  Histogram kernel: an exact
    integer bin sum ``isum``, then ``fl(isum / w)`` (``isum / w < hist_bins``), ``+ base``, ``- s``, ``fl(c - s)``
    and the difference: five roundings, each of one of ``hist_bins``, ``sum |x_i| / w``, ``|mean - s|``, ``|c - s|``
    or the result.  ``(w + 4) u M`` with ``M`` the sum of all those magnitudes covers both, widened by 1e-6 for the
    second-order terms and the bound's own evaluation."""
    x = np.asarray(x, np.float64)
    n, h = x.size, w // 2
    c = x[h: n - h]
    ax, axs = np.abs(x), np.abs(x - shift)
    ma = (np.cumsum(np.concatenate([[0.0], ax]))[w:] - np.cumsum(np.concatenate([[0.0], ax]))[:-w])[: n - w] / w
    ms = (np.cumsum(np.concatenate([[0.0], axs]))[w:] - np.cumsum(np.concatenate([[0.0], axs]))[:-w])[: n - w] / w
    M = np.abs(c - shift) + ms + np.abs(c) + ma + hist_bins
    return (w + 4) * U * M * (1 + 1e-6)


def check_mean(got, x, w, bound, tag):
    """``got`` within ``bound`` of the exact ``c - sum(x[j:j+w]) / w``, decided in integers."""
    x = np.asarray(x, np.float64)
    n, h = x.size, w // 2
    ratios = [v.as_integer_ratio() for v in x.tolist()]
    K = max(q for _, q in ratios)
    P = [p * (K // q) for p, q in ratios]
    S = [0]
    for p in P:
        S.append(S[-1] + p)
    for j in range(n - w):
        exact = Fraction(P[j + h] * w - (S[j + w] - S[j]), w * K)
        assert abs(Fraction(float(got[j])) - exact) <= Fraction(float(bound[j])), (tag, j, float(got[j]), float(exact))


# ------------------------------------------------------------------------------------------------- inputs
def series(rng, n, kind):
    """One segment: integer-valued (numpy int64, run as float32 or int32) or float32 samples."""
    walk = np.cumsum(rng.integers(-1, 2, n))
    if kind == "int":
        return walk
    if kind == "frac":                 # non-integer float32
        return (walk + rng.normal(0, 0.7, n)).astype(np.float32)
    if kind == "one_frac":             # one non-integer sample in an integer segment
        v = walk.astype(np.float32)
        v[n // 2] += 0.5
        return v
    if kind == "edge32000":            # the int16 staging edge: +-32000 fits, +-32001 does not
        v = np.clip(walk * 200, -32001, 32001)
        k = min(n, 6)
        v[rng.choice(n, k, replace=False)] = [-32001, -32000, 32000, 32001, 32001, -32001][:k]
        return v
    if kind == "big":                  # |x| around 1e9, integer-valued and exact in float32
        return (10 ** 9 // 64 + walk) * 64
    raise ValueError(kind)


# ------------------------------------------------------------------------------ median, before smoothing
@pytest.mark.parametrize("kind", ["int", "int32", "frac", "one_frac", "edge32000", "big"])
def test_median_before_smoothing_is_bit_exact(rec, dev, kind):
    rng = np.random.default_rng(sum(map(ord, kind)))
    for w in (2, 4, 1000):
        lens = [w + 4096, w + 4097, w + 8193, w + 1, w + 37]   # rank tiles split; the last one is short
        xs = [series(rng, n, "int" if kind == "int32" else kind) for n in lens]
        x = np.concatenate(xs).astype(np.int32 if kind == "int32" else np.float32)
        for sub in (False, True):
            shifts = gpu_shift(x, lens, 77, dev) if sub else np.zeros(len(lens))
            for impl in (None, "hist"):
                got, off, calls = run(rec, x, lens, dev, median_window_size=w, savgol=False, subtract_edges=sub,
                                      edge_size=77, impl=impl)
                k = kinds(calls)
                integer_small = kind in ("int", "int32")
                rank = ("rank", "int" if kind == "int32" else "float", sub, -1, False)
                if impl is None and integer_small:             # the rank kernel alone
                    assert k[-1] == rank and not any(c[0] == "hist" for c in k), k
                else:                                          # the histogram kernel, after a flagged rank launch
                    assert ("hist", False, sub) in k and (rank in k) == (impl is None), k
                    n_list, n_runs = generic_runs(calls)
                    if kind == "frac":
                        assert n_list == n_runs, (n_list, n_runs)       # every run is non-integer
                    elif kind == "one_frac":
                        assert 0 < n_list < n_runs, (n_list, n_runs)    # only the runs around the one sample
                    elif integer_small:
                        assert n_list == 0
                for i, xi in enumerate(xs):
                    exp = median_ref(xi, w, shifts[i])
                    assert np.array_equal(got[off[i]: off[i + 1]], exp), (kind, w, sub, impl, i)


# ------------------------------------------------------------------------------------------- the shift
def shift_bound(x, e):
    """``|gpu - exact|`` of the shift: two left-to-right sums of ``k_a`` / ``k_b`` doubles (error ``gamma_{k-1}
    sum |x|``), two quotients, one sum and an exact halving: ``<= (k + 2) u (mean_a |x| + mean_b |x|) / 2`` with
    ``k = max(k_a, k_b)`` to first order.  Twice that is returned, which covers the second-order terms."""
    a, b = np.abs(x[:e]), np.abs(x[-e:])
    return (max(a.size, b.size) + 2) * U * (a.mean() + b.mean())


def test_edge_shift_follows_python_slices(rec, dev):
    rng = np.random.default_rng(7)
    lens = [1000, 1999, 4]
    for kind in ("int", "frac", "big"):
        xs = [series(rng, n, kind) for n in lens]
        x = np.concatenate(xs).astype(np.float32)
        for e in (0, 1, -1, -3, 3, 4, 5, 77, 999, 1000, 1001, 5000, -999, -1000, -5000):
            got = gpu_shift(x, lens, e, dev)
            assert kinds(rec)[-1] == ("edge_shift",)
            for i, xi in enumerate(xs):
                x64 = np.asarray(xi, np.float32).astype(np.float64)
                exp = np_shift(x64, e)
                tag = (kind, e, i)
                if np.isnan(exp):
                    assert np.isnan(got[i]), tag
                elif kind != "frac":
                    assert got[i] == exp, tag
                else:
                    ex = (Fraction(sum(Fraction(v) for v in x64[:e].tolist()), x64[:e].size)
                          + Fraction(sum(Fraction(v) for v in x64[-e:].tolist()), x64[-e:].size)) / 2
                    assert abs(Fraction(float(got[i])) - ex) <= Fraction(float(shift_bound(x64, e) * (1 + 1e-6))), tag
    # edge_size 0 shifts by NaN: every output of adjust_segments is NaN, as in the reference
    x = series(rng, 3000, "int").astype(np.float32)
    for kw in (dict(), dict(impl="hist"), dict(use_mean=True)):
        got, _, calls = run(rec, x, [3000], dev, median_window_size=100, subtract_edges=True, edge_size=0, **kw)
        assert np.isnan(got).all() and got.size == 2900, kw
    # a negative edge on the whole path
    got, off, _ = run(rec, x, [3000], dev, median_window_size=100, savgol=False, subtract_edges=True, edge_size=-40)
    assert np.array_equal(got, median_ref(x, 100, np_shift(x.astype(np.float64), -40)))


# ------------------------------------------------------------------------------------------ mean windows
@pytest.mark.parametrize("kind", ["int", "frac", "one_frac", "edge32000", "big"])
def test_mean_windows_within_bound(rec, dev, kind):
    rng = np.random.default_rng(11 + len(kind))
    for w, run_len in ((2, 7), (4, 1), (1000, 1024), (1000, None)):
        lens = [w + 3001, w + 57, w + 1]
        xs = [series(rng, n, kind) for n in lens]
        x = np.concatenate(xs).astype(np.float32)
        shifts = gpu_shift(x, lens, 33, dev)
        outs = {}
        for sub in (False, True):
            got, off, calls = run(rec, x, lens, dev, median_window_size=w, use_mean=True, savgol=False,
                                  subtract_edges=sub, edge_size=33, run_len=run_len)
            k = kinds(calls)
            assert ("hist", True, sub) in k, k
            if kind == "frac":
                assert ("generic", True, sub) in k
            outs[sub] = got
            for i, xi in enumerate(xs):
                s = shifts[i] if sub else 0.0
                xi64 = np.asarray(xi, np.float32).astype(np.float64)
                check_mean(got[off[i]: off[i + 1]], xi64, w, mean_bound(xi64, w, s), (kind, w, run_len, sub, i))
        # the shift cancels: with and without it the outputs differ by rounding only
        for i, xi in enumerate(xs):
            xi64 = np.asarray(xi, np.float32).astype(np.float64)
            lim = mean_bound(xi64, w, shifts[i]) + mean_bound(xi64, w, 0.0)
            assert (np.abs(outs[True][off[i]: off[i + 1]] - outs[False][off[i]: off[i + 1]]) <= lim).all(), (kind, w)


# --------------------------------------------------------------------------------------------- smoothing
SMOOTH = [(3, 0), (3, 1), (3, 2), (5, 0), (5, 3), (5, 4), (21, 0), (21, 1), (21, 2), (21, 3), (21, 4), (21, 5),
          (21, 7), (21, 12), (51, 2), (51, 4), (51, 5), (51, 7), (101, 2), (101, 3), (101, 8), (101, 10),
          (127, 2), (127, 5), (127, 7), (127, 12)]


@pytest.mark.parametrize("sg", SMOOTH, ids=[f"{m}-{d}" for m, d in SMOOTH])
def test_smoothing_against_exact_hat_matrix(rec, dev, sg):
    from finaletoolkit_b200.device import savgol_tables
    m, d = sg
    rng = np.random.default_rng(m * 31 + d)
    w = 100
    lens = [w + m, w + m + 1, w + 2 * m - 1, w + 1500 + m]     # every / nearly every output an edge fit, and a long one
    xs = [series(rng, n, "int") for n in lens]
    x = np.concatenate(xs).astype(np.float32)
    tables = savgol_tables(m, d)
    kw = dict(median_window_size=w, savgol_window_size=m, savgol_poly_deg=d, edge_size=50)
    for sub in (False, True):
        for impl in (None, "hist"):
            pre, off, _ = run(rec, x, lens, dev, savgol=False, subtract_edges=sub, impl=impl, **kw)
            got, off2, calls = run(rec, x, lens, dev, savgol=True, subtract_edges=sub, impl=impl, **kw)
            assert np.array_equal(off, off2)
            k = kinds(calls)
            if impl is None:
                assert k[-1][0] == "rank" and k[-1][2] == sub and k[-1][3] == (21 if m == 21 else 0), k
                # the int32 tensor runs the other instantiation of the same kernel, to the same bits
                got_i, _, calls_i = run(rec, x.astype(np.int32), lens, dev, savgol=True, subtract_edges=sub, **kw)
                assert kinds(calls_i)[-1][1] == "int" and np.array_equal(got_i, got)
            else:
                assert ("savgol", 21 if m == 21 else 0) in k, k
            for i in range(len(lens)):
                check_smoothed(got[off[i]: off[i + 1]], pre[off[i]: off[i + 1]], m, d, tables, (sg, sub, impl, i))


def test_smoothing_paths_reach_every_stencil(rec, dev):
    """Which rank instantiation a (window, degree) takes: the exact sliding moments for degree <= 3 on small
    windows, the fp64 stencil for degree >= 4 (window 21 unrolled, other windows at run time) and for windows
    whose moments could overflow int32 (127)."""
    x = series(np.random.default_rng(3), 3000, "int").astype(np.float32)
    for (m, d), want in (((21, 2), (21, True)), ((51, 3), (0, True)), ((21, 4), (21, False)),
                         ((51, 4), (0, False)), ((127, 2), (0, False))):
        for xin, t in ((x, "float"), (x.astype(np.int32), "int")):
            _, _, calls = run(rec, xin, [3000], dev, median_window_size=100, savgol_window_size=m, savgol_poly_deg=d)
            assert kinds(calls)[-1] == ("rank", t, False, want[0], want[1]), (m, d, t)


# ---------------------------------------------------------------------------------------- non-finite input
def test_non_finite_samples_on_the_generic_path(rec, dev):
    rng = np.random.default_rng(5)
    w = 100
    lens = [2000, 2000, 1300]
    xs = [(np.cumsum(rng.integers(-3, 4, n)) + 0.25).astype(np.float32) for n in lens]
    xs[0][[60, 700, 701, 1500]] = np.nan                   # isolated and adjacent NaNs, one inside the first window
    xs[1][[300, 1200]] = [np.inf, -np.inf]
    xs[2][[1000]] = np.nan
    xs[2][[200]] = np.inf
    x = np.concatenate(xs)
    for sub, e in ((False, 50), (True, 50)):
        shifts = gpu_shift(x, lens, e, dev) if sub else np.zeros(len(lens))
        for impl in (None, "hist"):
            pre, off, calls = run(rec, x, lens, dev, median_window_size=w, savgol=False, subtract_edges=sub,
                                  edge_size=e, impl=impl, run_len=None if impl is None else 257)
            assert ("generic", False, sub) in kinds(calls)
            for i, xi in enumerate(xs):
                exp = median_ref(xi, w, shifts[i])
                g = pre[off[i]: off[i + 1]]
                if i == 0:   # NaN exactly in the windows that hold one
                    nan = np.isnan(xi.astype(np.float64))
                    touch = sliding_window_view(nan, w)[: xi.size - w].any(axis=1)
                    assert np.array_equal(np.isnan(g), touch), (sub, impl)
                assert np.array_equal(g, exp, equal_nan=True), (sub, impl, i)
            # after smoothing: NaN reaches exactly the outputs whose stencil or edge fit touches one
            from finaletoolkit_b200.device import savgol_tables
            got, _, calls = run(rec, x, lens, dev, median_window_size=w, savgol_window_size=21, savgol_poly_deg=2,
                                subtract_edges=sub, edge_size=e, impl=impl)
            for i in (0,):
                check_smoothed(got[off[i]: off[i + 1]], pre[off[i]: off[i + 1]], 21, 2, savgol_tables(21, 2), (sub, impl))
    # mean windows: a NaN makes exactly its windows NaN
    got, off, calls = run(rec, x, lens, dev, median_window_size=w, use_mean=True, savgol=False)
    nan = np.isnan(xs[0].astype(np.float64))
    assert np.array_equal(np.isnan(got[off[0]: off[1]]), sliding_window_view(nan, w)[: lens[0] - w].any(axis=1))


# ------------------------------------------------------------------------------------------------ layouts
def test_many_tiny_segments(rec, dev):
    """> 3000 segments of 21..24 outputs back to back: the smoothing CTAs (1024 outputs, 4 per thread) straddle
    segment boundaries at every residue mod 4; every output but the middle one of a 21-output segment is an edge fit."""
    from finaletoolkit_b200.device import savgol_tables
    rng = np.random.default_rng(9)
    w, m, d = 4, 21, 3
    lens = [w + m + (i % 4) for i in range(3100)]
    xs = [series(rng, n, "int") for n in lens]
    x = np.concatenate(xs)
    tables = savgol_tables(m, d)
    for sub in (False, True):
        for impl in (None, "hist"):
            pre, off, _ = run(rec, x, lens, dev, median_window_size=w, savgol=False, subtract_edges=sub, edge_size=3,
                              impl=impl)
            got, _, _ = run(rec, x, lens, dev, median_window_size=w, savgol_window_size=m, savgol_poly_deg=d,
                            subtract_edges=sub, edge_size=3, impl=impl)
            shifts = gpu_shift(x, lens, 3, dev) if sub else np.zeros(len(lens))
            for i in range(0, len(lens), 7):
                assert np.array_equal(pre[off[i]: off[i + 1]], median_ref(xs[i], w, shifts[i])), (sub, impl, i)
                check_smoothed(got[off[i]: off[i + 1]], pre[off[i]: off[i + 1]], m, d, tables, (sub, impl, i))


def test_segments_of_exactly_the_window(rec, dev):
    """n == w: no output for that segment, with ``savgol=False`` and through a ``skip_short`` plan."""
    import torch
    from finaletoolkit_b200.device import AdjustPlan, adjust_segments, savgol_tables
    rng = np.random.default_rng(2)
    w = 200
    lens = [w, w + 500, w, w + 21, w + 20, w + 3000]
    xs = [series(rng, n, "int") for n in lens]
    x = np.concatenate(xs)
    got, off, _ = run(rec, x, lens, dev, median_window_size=w, savgol=False)
    assert list(np.diff(off)) == [n - w for n in lens]
    for i, xi in enumerate(xs):
        assert np.array_equal(got[off[i]: off[i + 1]], median_ref(xi, w, 0.0))
    plan = AdjustPlan(lens, w, True, 21, 2, dev, skip_short=True)
    assert list(plan.n_out) == [0, 500, 0, 21, 0, 3000]
    xd = torch.from_numpy(x.astype(np.int32)).to(dev)
    sm, _ = adjust_segments(xd, None, plan=plan, median_window_size=w)
    pre, _ = adjust_segments(xd, None, plan=AdjustPlan(lens, w, False, 21, 2, dev, skip_short=True),
                             median_window_size=w, savgol=False)
    sm, pre = sm.cpu().numpy(), pre.cpu().numpy()
    o = plan.out_off
    pre_off = np.concatenate([[0], np.cumsum(np.array(lens) - w)])
    for i in np.flatnonzero(plan.n_out):
        p = pre[pre_off[i]: pre_off[i + 1]]
        assert np.array_equal(p, median_ref(xs[i], w, 0.0))
        check_smoothed(sm[o[i]: o[i + 1]], p, 21, 2, savgol_tables(21, 2), i)


@pytest.mark.parametrize("kind", ["int", "frac"])
def test_widest_median_window(rec, dev, kind):
    """w = 32766: no rank plan fits, the sliding-histogram kernel runs (and the generic one for non-integer input)."""
    rng = np.random.default_rng(4)
    w = 32766
    lens = [w + 300, w + 41]
    if kind == "int":       # i.i.d. 0..99: every run stays inside the histogram kernel's 256-bin value window
        xs = [rng.integers(0, 100, n) for n in lens]
    else:   # nearly sorted: the generic kernel's insertion sort of a 32766-sample window stays short
        xs = [(0.25 * np.arange(n) + rng.normal(0, 0.1, n)).astype(np.float32) for n in lens]
    x = np.concatenate(xs)
    for sub in (False, True):
        shifts = gpu_shift(x, lens, 500, dev) if sub else np.zeros(2)
        got, off, calls = run(rec, x, lens, dev, median_window_size=w, savgol=False, subtract_edges=sub, edge_size=500)
        k = kinds(calls)
        assert not any(c[0] == "rank" for c in k) and ("hist", False, sub) in k
        assert (("generic", False, sub) in k) == (kind == "frac")
        for i, xi in enumerate(xs):
            assert np.array_equal(got[off[i]: off[i + 1]], median_ref(xi, w, shifts[i])), (kind, sub, i)


# ----------------------------------------------------------------------------------------- genome driver
@pytest.mark.parametrize("adjust", [dict(use_mean=True), dict(subtract_edges=True, edge_size=300),
                                    dict(use_mean=True, subtract_edges=True, edge_size=-250),
                                    dict(subtract_edges=True, savgol_window_size=31, savgol_poly_deg=7),
                                    dict(use_mean=True, savgol_window_size=101, savgol_poly_deg=10)],
                         ids=["mean", "edges", "mean-edges", "edges-31-7", "mean-101-10"])
def test_genome_driver_general_path(rec, dev, adjust):
    """``multi_wps_genome(adjust=...)`` with ``use_mean`` / ``subtract_edges``: the int32 WPS in HBM through
    ``adjust_segments`` with a ``skip_short`` plan, on two contigs with intervals too short for the filters."""
    import torch
    from finaletoolkit_b200 import distributed as FD
    from finaletoolkit_b200.device import AdjustPlan, WpsPlan, adjust_segments, savgol_tables
    from finaletoolkit_b200.io.fragments import FragmentTable
    from finaletoolkit_b200.synth import synth_fragments
    sizes = {"a": 40_000, "b": 25_000}
    table = FragmentTable({c: synth_fragments(n, 12_000, i, seed_base=5151) for i, (c, n) in enumerate(sizes.items())})
    w = 1000
    adj = dict(median_window_size=w, **adjust)
    m, d = adj.get("savgol_window_size", 21), adj.get("savgol_poly_deg", 2)
    sites = {"a": (np.array([0, 5000, 6100, 9000, 21_000]), np.array([4000, 6000, 6200, 20_000, 21_000 + w + m])),
             "b": (np.array([100, 3000, 12_000]), np.array([1100 + m - 1, 11_000, 24_000]))}
    res, _, _ = FD.multi_wps_genome(table, list(sizes.items()), sites, 5000, 120, 120, 180, 30, adjust=adj, device=dev,
                                    contigs=list(sizes))
    k = kinds(rec)                                                     # the general path ran
    assert (("hist", True, bool(adj.get("subtract_edges"))) in k) == bool(adj.get("use_mean"))
    assert (("edge_shift",) in k) == bool(adj.get("subtract_edges"))
    for c, n in sizes.items():
        r = res[c]
        s, e = sites[c]
        plan = WpsPlan(s, e, n, 180, dev)
        wps = plan.run(table.device(c, dev))
        assert torch.equal(r.wps, wps)
        lens = np.diff(plan.offsets)
        ap = AdjustPlan(lens, w, True, m, d, dev, skip_short=True)
        assert np.array_equal(r.adj_offsets, ap.out_off) and np.array_equal(r.adj_segments, np.flatnonzero(ap.n_out))
        assert (ap.n_out == 0).any() and (ap.n_out > 0).any()
        ref, _ = adjust_segments(wps, None, plan=ap, **adj)
        assert torch.equal(r.adjusted, ref), c
        # the values: the unsmoothed series against its bound, the smoothed one against the exact hat matrix
        pre_plan = AdjustPlan(lens, w, False, m, d, dev, skip_short=True)
        pre, _ = adjust_segments(wps, None, plan=pre_plan, **{**adj, "savgol": False})
        pre, got, wh = pre.cpu().numpy(), r.adjusted.cpu().numpy(), wps.cpu().numpy().astype(np.float64)
        shifts = gpu_shift(wh, lens, adj.get("edge_size", 500), dev) if adj.get("subtract_edges") else np.zeros(len(lens))
        for i in np.flatnonzero(ap.n_out):
            xi = wh[plan.offsets[i]: plan.offsets[i + 1]]
            p = pre[pre_plan.out_off[i]: pre_plan.out_off[i + 1]]
            if adj.get("use_mean"):
                check_mean(p, xi, w, mean_bound(xi, w, shifts[i]), (c, i))
            else:
                assert np.array_equal(p, median_ref(xi, w, shifts[i])), (c, i)
            check_smoothed(got[ap.out_off[i]: ap.out_off[i + 1]], p, m, d, savgol_tables(m, d), (c, i))


# ---------------------------------------------------------------------------------------------- coverage
def test_every_instantiation_was_reached(request):
    """The cases above launched every kernel instantiation (skipped when only some of them ran)."""
    ran = {it.originalname for it in request.session.items if it.module is request.module}
    tests = {name for name in vars(request.module) if name.startswith("test_")}
    if ran != tests:
        pytest.skip("only part of the module ran")
    missing = ALL - REACHED
    assert not missing, sorted(missing, key=str)
