"""``ftk_wps_plan_tiles`` (the host tile planner behind ``WpsPlan``) at the top of the int32 coordinate range.

A contig may be up to 2^31 - 1 bases long (BAM headers allow it), and ``distributed.GenomeShard`` places contigs
near that ceiling in its virtual coordinate space.  The planner computes in int64 and writes int32 tiles: a midpoint
window ``E + max_len`` must clamp to the contig instead of wrapping, and bounds past int32 must be refused.
Runs without a GPU: the planner is host code in the shared library."""
from ctypes import POINTER, c_int32, c_int64

import numpy as np
import pytest

I32_MAX = 2 ** 31 - 1
TILE = 5119          # FTK_WPS_TILE
FTK_E_RANGE = -3


def _plan(starts, stops, chrom_size, max_len, count_only=False):
    """(return code, tiles dict or None) of ``ftk_wps_plan_tiles``."""
    from finaletoolkit_b200._lib import lib
    s = np.ascontiguousarray(starts, np.int64)
    e = np.ascontiguousarray(stops, np.int64)
    off = np.zeros(len(s) + 1, np.int64)
    np.cumsum(np.maximum(e - s, 0), out=off[1:])
    i64p, i32p = POINTER(c_int64), POINTER(c_int32)
    p = lambda a, t: a.ctypes.data_as(POINTER(t))       # noqa: E731
    L = lib()
    n = L.ftk_wps_plan_tiles(p(s, c_int64), p(e, c_int64), p(off, c_int64), len(s), int(chrom_size), int(max_len),
                             i32p(), i32p(), i32p(), i32p(), i64p())
    if n < 0 or count_only:
        return int(n), None
    t = {k: np.full(n, -7, np.int32) for k in ("p0", "len", "mid_lo", "mid_hi")}
    t["out_off"] = np.full(n, -7, np.int64)
    rc = L.ftk_wps_plan_tiles(p(s, c_int64), p(e, c_int64), p(off, c_int64), len(s), int(chrom_size), int(max_len),
                              p(t["p0"], c_int32), p(t["len"], c_int32), p(t["mid_lo"], c_int32), p(t["mid_hi"], c_int32),
                              p(t["out_off"], c_int64))
    assert rc == n
    t["offsets"] = off
    return int(n), t


def _expected_tiles(S, E):
    """Tiles of one interval: equal pieces of at most FTK_WPS_TILE & ~3 positions, rounded up to a multiple of 4."""
    cap4 = TILE & ~3
    n = E - S
    pieces = -(-n // cap4)
    piece = -(-n // pieces)
    piece = (piece + 3) & ~3
    return [(S + k, min(piece, n - k)) for k in range(0, n, piece)]


def _check_cover(t, ivs, chrom_size, max_len):
    """Tiles cover every interval exactly once, in order, with the interval's clamped midpoint window."""
    k = 0
    for i, (S, E) in enumerate(ivs):
        exp = _expected_tiles(S, E)
        for j, (p0, ln) in enumerate(exp):
            assert (int(t["p0"][k]), int(t["len"][k])) == (p0, ln), (S, E, j)
            assert 0 < ln <= TILE
            assert int(t["mid_lo"][k]) == max(S - max_len, 0)
            assert int(t["mid_hi"][k]) == min(E + max_len, chrom_size)
            assert int(t["out_off"][k]) == int(t["offsets"][i]) + (p0 - S)
            k += 1
    assert k == len(t["p0"])


def test_interval_ending_at_the_int32_ceiling():
    """E = chrom_size = 2^31 - 1: mid_hi is 2^31 - 1 exactly, every tile field is positive (no wrap)."""
    c = I32_MAX
    ivs = [(c - 12_000, c - 5_000), (c - 5_000, c), (c - 1, c)]
    n, t = _plan([a for a, _ in ivs], [b for _, b in ivs], c, 180)
    assert n > 0
    _check_cover(t, ivs, c, 180)
    assert int(t["mid_hi"].max()) == c and int(t["mid_hi"].min()) > 0
    assert int(t["p0"][-1]) == c - 1 and int(t["len"][-1]) == 1
    assert int(t["p0"].astype(np.int64).max() + t["len"][np.argmax(t["p0"])]) == c


@pytest.mark.parametrize("max_len", [0, 1, 180, 600, 2 ** 30, I32_MAX])
def test_padded_window_clamps_instead_of_wrapping(max_len):
    """E + max_len > 2^31 - 1 clamps to the contig size; S - max_len < 0 clamps to 0."""
    c = I32_MAX
    ivs = [(0, 300), (c - 2 * TILE - 7, c - 50), (c - 50, c - 3)]
    n, t = _plan([a for a, _ in ivs], [b for _, b in ivs], c, max_len)
    _check_cover(t, ivs, c, max_len)
    assert (t["mid_hi"].astype(np.int64) >= t["mid_lo"]).all()
    # a contig shorter than the ceiling: the window clamps to its size, not to int32
    n, t = _plan([c - 10_000], [c - 5_000], c - 4_000, max_len)
    _check_cover(t, [(c - 10_000, c - 5_000)], c - 4_000, max_len)


@pytest.mark.parametrize("stop,chrom_size", [(2 ** 31, I32_MAX), (2 ** 31, 2 ** 31), (I32_MAX, 2 ** 31),
                                             (2 ** 32 + 5, I32_MAX), (10, 2 ** 40)])
def test_bounds_past_int32_are_refused(stop, chrom_size):
    rc, _ = _plan([stop - 100], [stop], chrom_size, 180, count_only=True)
    assert rc == FTK_E_RANGE
    with pytest.raises(Exception, match="ftk_wps_plan_tiles"):
        from finaletoolkit_b200.device import WpsPlan
        WpsPlan.host_tiles([stop - 100], [stop], chrom_size, 180)


def test_degenerate_interval_past_the_ceiling_is_skipped_not_refused():
    """E <= S owns no position (frag/_wps.py:145-152), whatever its bounds."""
    rc, _ = _plan([2 ** 31 + 10, 5], [2 ** 31 + 10, 5], I32_MAX, 180, count_only=True)
    assert rc == 0


@pytest.mark.parametrize("S,E", [(0, I32_MAX), (1, I32_MAX), (-(2 ** 30), I32_MAX)])
def test_interval_of_two_giga_bases_gets_the_right_tile_count(S, E):
    n, _ = _plan([S], [E], I32_MAX, 180, count_only=True)
    assert n == len(_expected_tiles(S, E))
    assert TILE * n >= E - S > (TILE - 4) * (n - 1)
