"""Plain numpy restatement of the WPS periodogram (``wps_spectrum`` / ``device.spectrum_segments``, DESIGN.md 4.12).

For a series x of N values with mean mu and every integer period P:
    I(P) = |sum_{n<N} (x[n] - mu) exp(-2 pi i (n mod P) / P)|^2 / N
as the direct sum over n, with the phase reduced to n mod P, in fp64 (int32 values are exact in fp64).  An empty
series gives a row of NaN."""
import numpy as np


def spectrum(x, min_period, max_period):
    x = np.asarray(x, np.float64)
    N = x.size
    if N == 0:
        return np.full(max_period - min_period + 1, np.nan)
    xc = x - x.mean()
    n = np.arange(N)
    return np.array([abs(np.dot(xc, np.exp(-2j * np.pi * (n % P) / P))) ** 2 / N
                     for P in range(min_period, max_period + 1)])


def bound(x):
    """The allowed error of every I(P) of x: 1e-10 * max(1, sum (x - mu)^2)."""
    x = np.asarray(x, np.float64)
    return 1e-10 * max(1.0, float(np.sum((x - x.mean()) ** 2))) if x.size else 0.0


def check_row(got, x, min_period, max_period):
    """``got`` (one row) against the direct sum of ``x``."""
    exp = spectrum(x, min_period, max_period)
    got = np.asarray(got, np.float64)
    assert got.shape == exp.shape
    if np.asarray(x).size == 0:
        assert np.isnan(got).all()
        return
    err = np.abs(got - exp)
    assert np.isfinite(got).all() and float(err.max()) <= bound(x), (float(err.max()), bound(x))


def text(intervals, n, periods, intensity):
    """The TSV ``wps_spectrum`` writes."""
    head = "contig\tstart\tstop\tname\tn\t" + "\t".join(f"p{p}" for p in periods) + "\n"
    return head + "".join(f"{c}\t{s}\t{e}\t{name}\t{int(k)}\t" + "\t".join(repr(float(v)) for v in row) + "\n"
                          for (c, s, e, name), k, row in zip(intervals, n, intensity))
