"""Exact Savitzky-Golay arithmetic: the least-squares hat matrix in rationals and a rounding-error check.

``exact_hat(m, d)``: the hat matrix of a degree-``d`` least-squares polynomial fit on the ``m`` points
``-m//2 .. m//2``, ``H = A (A^T A)^-1 A^T`` with ``A`` the integer Vandermonde matrix.  The normal equations are
solved exactly (Gauss-Jordan elimination in Fractions), so ``H = N / den`` with integer ``N``.  Row ``m//2``
is the interior stencil, rows ``0 .. m//2 - 1`` / ``m//2 + 1 ..`` the mode='interp' edge fits of the first / last
``m`` samples - the three tables ``device.savgol_tables`` returns.

``check_smoothed``: a smoothed series against ``H`` applied exactly to the series it smoothed (the doubles scaled
to integers over one power-of-two denominator, so every ``sum H[row] . x`` is an exact rational)."""
from fractions import Fraction
from functools import lru_cache
from math import gcd

import numpy as np

EPS = float(np.finfo(np.float64).eps)
# a table entry of a correct construction is within this many ulp of max |H| (tests/test_host_logic.py checks the
# tables over every window <= 127 and degree <= 20 against it)
TABLE_ULPS = 16


@lru_cache(maxsize=None)
def exact_hat(m: int, d: int):
    """``(N, den)``: ``N`` an m x m numpy object array of Python ints, ``H = N / den`` exactly (``den > 0``)."""
    assert m >= 1 and m % 2 == 1 and 0 <= d < m
    if d == m - 1:                      # A is square and invertible: the fit interpolates, H = I
        return np.eye(m, dtype=np.int64).astype(object), 1
    h = m // 2
    pos = list(range(-h, h + 1))
    p = d + 1
    # (A^T A)^-1 by Gauss-Jordan elimination in Fractions (A^T A is positive definite: no pivoting needed)
    M = [[Fraction(sum(x ** (r + c) for x in pos)) for c in range(p)] + [Fraction(int(r == c)) for c in range(p)]
         for r in range(p)]
    for k in range(p):
        piv = M[k][k]
        assert piv > 0
        M[k] = [v / piv for v in M[k]]
        for i in range(p):
            if i != k and M[i][k] != 0:
                f = M[i][k]
                M[i] = [a - f * b for a, b in zip(M[i], M[k])]
    inv = [row[p:] for row in M]
    den = 1
    for row in inv:
        for v in row:
            den = den * v.denominator // gcd(den, v.denominator)
    G = np.array([[int(v * den) for v in row] for row in inv], dtype=object)   # (A^T A)^-1 = G / den
    A = np.array([[x ** k for k in range(p)] for x in pos], dtype=object)      # m x p Vandermonde, integers
    N = A.dot(G).dot(A.T)
    g = 0
    for v in N.flat:
        g = gcd(g, int(v))
    g = gcd(g, den)
    return N // g, den // g


def hat_float(m: int, d: int) -> np.ndarray:
    """``H`` rounded entry by entry to the nearest double (Python's int / int is correctly rounded)."""
    N, den = exact_hat(m, d)
    return np.array([[v / den for v in row] for row in N], dtype=np.float64)


def _scaled(x):
    """Doubles ``x`` as ``(P, K)``: Python ints with ``x_i = P_i / K`` exactly, ``K`` a power of two."""
    ratios = [float(v).as_integer_ratio() for v in x]
    K = max(q for _, q in ratios) if ratios else 1
    return np.array([p * (K // q) for p, q in ratios], dtype=object), K


def table_rounding(table: np.ndarray, N_rows, den: int) -> np.ndarray:
    """``|table - H|`` entry by entry (rounded to double, then up by one part in 1e9: an upper bound)."""
    out = np.empty(table.shape, np.float64)
    for idx in np.ndindex(table.shape):
        out[idx] = float(abs(Fraction(float(table[idx])) - Fraction(int(N_rows[idx]), den)))
    return out * (1 + 1e-9)


_ROUNDING = {}


def _tables_rounding(m: int, d: int, coef, first, last):
    """``table_rounding`` of the three tables, cached by their bytes; each entry must be within ``TABLE_ULPS`` ulp of
    ``max |H|`` of exact: the bound of ``check_smoothed`` allows a table its rounding, not a different filter."""
    key = (m, d, coef.tobytes(), first.tobytes(), last.tobytes())
    if key not in _ROUNDING:
        N, den = exact_hat(m, d)
        h = m // 2
        r = (table_rounding(coef, N[h], den), table_rounding(first, N[:h], den), table_rounding(last, N[h + 1:], den))
        scale = max(abs(int(v)) for v in N.flat) / den
        worst = max(float(t.max()) if t.size else 0.0 for t in r)
        assert worst <= TABLE_ULPS * EPS * scale * (1 + 1e-6), ((m, d), "table off the exact filter", worst / (EPS * scale))
        _ROUNDING[key] = r
    return _ROUNDING[key]


def check_smoothed(got, x, m: int, d: int, tables, tag=""):
    """``got``: one segment's smoothed output, ``x``: the series it smoothed (same length ``n >= m``), ``tables``:
    the ``(coef, edge_first, edge_last)`` fp64 tables the kernel applied.

    Output ``j`` is a dot product of ``m`` doubles: ``t . x_w`` with ``t`` the table row (interior: ``coef``, the
    first / last ``m//2`` outputs: the edge rows) and ``x_w`` the ``m`` samples it covers (``x[j-m//2 : j+m//2+1]``,
    or the first / last ``m`` samples).  The exact value is ``H_row . x_w``.  The bound is derived from

        |fl(t . x_w) - H_row . x_w| <= |fl(t . x_w) - t . x_w| + |(t - H_row) . x_w|
                                    <= gamma_m * sum |t_i x_i| + sum |t_i - H_i| |x_i|,

    with ``gamma_m = m u / (1 - m u) < m * eps`` (``u = eps / 2``) the standard bound of an m-term fp64 dot product
    accumulated in any order, with or without fused multiply-adds.  The second term is the table's own rounding: every
    table entry must be within ``TABLE_ULPS`` ulp of ``max |H|`` of exact, or the check fails whatever the output.  It also covers the exact sliding-moment path,
    whose result is the exact ``a S0 + b M2`` (an integer below 2^53) times the rounded constant ``0.5 / den``: two
    roundings, ``<= 2 u |y| <= m eps sum |c_i x_i|``.  The bound is evaluated in fp64 and widened by one part in 1e6,
    far more than that evaluation's own rounding.

    Non-finite samples: an output whose ``x_w`` holds a NaN must be NaN, every other output is checked as above."""
    got = np.asarray(got, np.float64)
    x = np.asarray(x, np.float64)
    n, h = x.size, m // 2
    assert got.size == n and n >= m, (tag, got.size, n, m)
    N, den = exact_hat(m, d)
    coef, first, last = (np.asarray(t, np.float64) for t in tables)
    # window start and table row of every output
    j = np.arange(n)
    start = np.clip(j - h, 0, n - m)
    nan = np.isnan(x)
    cnan = np.concatenate([[0], np.cumsum(nan)])
    want_nan = (cnan[start + m] - cnan[start]) > 0
    assert np.array_equal(np.isnan(got), want_nan), (tag, "NaN pattern", np.flatnonzero(np.isnan(got) != want_nan)[:8])
    assert not np.isinf(x).any(), tag                                   # the bound below is for finite series
    xz = np.where(nan, 0.0, x)
    P, K = _scaled(xz)
    ax = np.abs(xz)
    d_coef, d_first, d_last = _tables_rounding(m, d, coef, first, last)
    # interior
    if n > 2 * h:
        num = np.correlate(P, N[h], "valid")                               # (n - 2h,) exact numerators / (den K)
        mag = np.correlate(ax, np.abs(coef), "valid")
        dmag = np.correlate(ax, d_coef, "valid")
        for k in range(n - 2 * h):
            jj = k + h
            if want_nan[jj]:
                continue
            _assert_close(got[jj], int(num[k]), den * K, m * EPS * mag[k] + dmag[k], (tag, "interior", jj))
    # edge fits
    for rows, Nrows, d_rows, base, js in ((first, N[:h], d_first, 0, range(h)),
                                          (last, N[h + 1:], d_last, n - m, range(n - h, n))):
        for r, jj in enumerate(js):
            if want_nan[jj]:
                continue
            seg = slice(base, base + m)
            num = int(np.dot(Nrows[r], P[seg]))
            lim = m * EPS * float(np.abs(rows[r]) @ ax[seg]) + float(d_rows[r] @ ax[seg])
            _assert_close(got[jj], num, den * K, lim, (tag, "edge", jj))


def _assert_close(g, num: int, q: int, lim: float, tag):
    """``|g - num / q| <= lim * (1 + 1e-6)``, decided in integers."""
    gp, gq = float(g).as_integer_ratio()
    lp, lq = float(lim * (1 + 1e-6)).as_integer_ratio()
    err = abs(gp * q - num * gq)                                           # |g - y| * q * gq
    assert err * lq <= lp * q * gq, (tag, float(g), num / q, lim)
