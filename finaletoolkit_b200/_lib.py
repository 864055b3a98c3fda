"""ctypes binding of ``libftk_b200.so`` (the C ABI in ``include/ftk_b200.h``).

The library is built in-tree by ``finaletoolkit_b200/csrc/build.py`` (nvcc,
sm_100a).  There is NO CPU fallback: if the shared library is missing or
fails to load, every compute entry point raises ``FtkLibraryError``.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_int64, c_uint8, c_uint32, c_void_p

__all__ = ["lib", "check", "FtkLibraryError", "FTK_NONE", "SO_PATH", "SYMBOLS"]

SO_PATH = os.environ.get("FTK_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libftk_b200.so")
FTK_NONE = -(2 ** 31)


class FtkLibraryError(RuntimeError):
    """libftk_b200.so is missing / failed to load, or a call returned an error."""


_i32p, _i64p, _u8p, _u32p, _f64p = (POINTER(c_int32), POINTER(c_int64), POINTER(c_uint8),
                                    POINTER(c_uint32), POINTER(c_double))
_P = c_void_p  # device pointers travel as integers

# name -> (restype, argtypes); must list every symbol include/ftk_b200.h declares
SYMBOLS = {
    "ftk_abi_version": (c_int, []),
    "ftk_error_string": (c_char_p, [c_int]),
    "ftk_last_cuda_error": (c_char_p, []),
    "ftk_pack_fragments_host": (c_int64, [_i32p, _i32p, _u8p, _u8p, c_int64, c_int32, _u32p, _i32p,
                                          _i32p, _i32p, _u8p, _u8p, c_int64, c_int32]),
    "ftk_unpack_fragments": (c_int, [_P, _P, _P, _P, _P, _P, c_int64, c_int64, _P, _P, _P, _P, c_int32, _P]),
    "ftk_length_stats_host": (c_int, [_i32p, _i32p, c_int64, c_int32, c_int32, c_int32, _f64p, _f64p, _f64p,
                                      _i64p, _i64p, _i64p, _f64p]),
    "ftk_wps_plan_tiles": (c_int64, [_i64p, _i64p, _i64p, c_int64, c_int64, c_int32,
                                     _i32p, _i32p, _i32p, _i32p, _i64p]),
    "ftk_wps_tile_ranges": (c_int, [_P, c_int64, _P, _P, c_int64, c_int32, c_int32, _P, _P]),
    "ftk_wps_tiles_i32": (c_int, [_P, _P, _P, c_int64, _P, _P, _P, _P, _P, c_int64,
                                  c_int32, c_int32, c_int32, c_int32, c_int32, _P, _P, _P]),
    "ftk_wps_tiles_i16": (c_int, [_P, _P, _P, c_int64, _P, _P, _P, _P, _P, c_int64,
                                  c_int32, c_int32, c_int32, c_int32, c_int32, _P, _P, _P, _P]),
    "ftk_wps_tiles_i8": (c_int, [_P, _P, _P, c_int64, _P, _P, _P, _P, _P, c_int64,
                                 c_int32, c_int32, c_int32, c_int32, c_int32, _P, _P, _P, _P]),
    "ftk_wps_cov_tile_ranges": (c_int, [_P, c_int64, _P, _P, c_int64, c_int32, c_int32, c_int32, c_int32, _P,
                                        _P, c_int64, _P, c_int64, _P]),
    "ftk_wps_cov_tiles": (c_int, [_P, _P, _P, c_int64, c_int32, _P, _P, _P, _P, _P, _P, c_int64,
                                  c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32,
                                  c_int32, _P, c_int32, _P, _P, _P, _P, _P]),
    "ftk_interval_hist_u64": (c_int, [_P, _P, _P, c_int64, c_int32, _P, _P, c_int64,
                                      c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32,
                                      _P, _P, _P, _P, _P]),
    "ftk_frag_lengths_i32": (c_int, [_P, _P, _P, c_int64, c_int32, c_int32, c_int32, c_int32,
                                     c_int32, c_int32, c_int32, _P, c_int64, _P, _P, _P]),
    "ftk_end_motif_hist_u64": (c_int, [_P, _P, _P, _P, c_int64, c_int32, _P, _P, c_int64,
                                       _P, _P, c_int64, c_int32, c_int32, c_int32, c_int32, c_int32,
                                       _P, _P, _P, _P]),
    "ftk_breakpoint_motif_hist_u64": (c_int, [_P, _P, _P, _P, c_int64, c_int32, _P, _P, c_int64,
                                              _P, _P, c_int64, c_int32, c_int32, c_int32, c_int32, c_int32,
                                              _P, _P, _P]),
    "ftk_delfi_windows_u64": (c_int, [_P, _P, _P, c_int64, c_int32, _P, _P, c_int64, _P, _P, c_int64,
                                      _P, _P, _P, _i32p, c_int32, c_int32, _P, _P, _P]),
    "ftk_agg_signal_f64": (c_int, [_P, c_int64, c_int64, c_int32, c_int32, _P, _P, _P]),
    "ftk_adjust_edge_shift_f64": (c_int, [_P, _P, c_int32, c_int32, _P, _P]),
    "ftk_adjust_wps_f64": (c_int, [_P, _P, _P, _P, _P, c_int32, c_int64, c_int32, c_int32, c_int32, _P, _P, _P]),
    "ftk_adjust_wps_generic_f64": (c_int, [_P, _P, _P, _P, _P, c_int32, _P, c_int64, c_int32, c_int32, c_int32,
                                           _P, _P, _P]),
    "ftk_savgol_f64": (c_int, [_P, _P, c_int32, c_int64, c_int32, _P, _P, _P, _P, _P]),
    "ftk_adjust_rank_f64": (c_int, [_P, c_int32, _P, _P, _P, c_int32, _P, _P, _P, c_int64, c_int32, c_int32,
                                    _P, _P, _P, c_int64, c_int64, c_int64, c_int32, c_int32, _P, _P, _P]),
    "ftk_cleavage_tiles_f64": (c_int, [_P, _P, _P, _P, c_int64, c_int32, _P, _P, _P, _P, _P, c_int64,
                                       c_int32, c_int32, c_int32, _P, _P, _P]),
    "ftk_depth_tiles_i32": (c_int, [_P, _P, _P, c_int64, c_int32, _P, _P, _P, _P, _P, c_int64,
                                    c_int32, c_int32, c_int32, c_int32, _P, _P, _P]),
    "ftk_gc_depth_tiles_f64": (c_int, [_P, _P, _P, c_int64, c_int32, _P, _P, c_int64, _P, _P, _P, _P, _P, c_int64,
                                       c_int32, c_int32, c_int32, c_int32, _P, c_int64, _P, _P, _P, _P]),
    "ftk_vplot_u64": (c_int, [_P, _P, _P, c_int64, c_int32, _P, _P, _P, c_int64, c_int32, c_int32, c_int32,
                              c_int32, c_int32, _P, _P, _P]),
    "ftk_ocf_u64": (c_int, [_P, _P, _P, c_int64, c_int32, _P, _P, _P, _P, c_int64, c_int32, c_int32, c_int32,
                            c_int32, c_int32, c_int32, _P, c_int32, c_int64, _P, _P, _P]),
    "ftk_gc_observed_u64": (c_int, [_P, _P, _P, c_int64, c_int32, _P, _P, c_int64, _P, _P, c_int64, c_int32, c_int32,
                                    c_int32, c_int32, _P, _P, _P]),
    "ftk_gc_expected_u64": (c_int, [_P, _P, c_int64, _P, _P, c_int64, c_int32, c_int32, c_int32, _P, _P]),
    "ftk_gc_weighted_intervals_f64": (c_int, [_P, _P, _P, c_int64, c_int32, _P, _P, c_int64, _P, _P, c_int64, c_int32,
                                              c_int32, c_int32, c_int32, _P, _P, _P, _P, _P]),
    "ftk_gc_weighted_sites_f64": (c_int, [_P, _P, _P, c_int64, c_int32, _P, _P, c_int64, _P, _P, _P, c_int64, c_int32,
                                          c_int32, c_int32, c_int32, c_int32, _P, _P, _P, _P, _P]),
    "ftk_spectrum_i32_f64": (c_int, [_P, _P, c_int64, c_int32, c_int32, _P, _P]),
    "ftk_spectrum_f64_f64": (c_int, [_P, _P, c_int64, c_int32, c_int32, _P, _P]),
    "ftk_fragfile_open": (c_void_p, [c_char_p, c_int32, _i32p]),
    "ftk_fragfile_open_slice": (c_void_p, [c_char_p, c_int64, c_int32, c_int64, c_int32, c_int32, c_int32, _i32p]),
    "ftk_bamfile_open": (c_void_p, [c_char_p, c_int32, _i32p]),
    "ftk_bamfile_fragments": (c_void_p, [c_void_p]),
    "ftk_bamfile_n_refs": (c_int32, [c_void_p]),
    "ftk_bamfile_ref_name": (c_char_p, [c_void_p, c_int32]),
    "ftk_bamfile_ref_length": (c_int64, [c_void_p, c_int32]),
    "ftk_bamfile_close": (None, [c_void_p]),
    "ftk_fragfile_is_bed6": (c_int32, [c_void_p]),
    "ftk_fragfile_skipped": (c_int64, [c_void_p]),
    "ftk_fragfile_n_contigs": (c_int32, [c_void_p]),
    "ftk_fragfile_contig_name": (c_char_p, [c_void_p, c_int32]),
    "ftk_fragfile_contig_count": (c_int64, [c_void_p, c_int32]),
    "ftk_fragfile_copy": (c_int, [c_void_p, c_int32, _i32p, _i32p, _u8p, _u8p]),
    "ftk_fragfile_copy_read1": (c_int, [c_void_p, c_int32, _i32p, _i32p]),
    "ftk_fragfile_close": (None, [c_void_p]),
    "ftk_zlib_compress_batch": (c_int, [_u8p, _i64p, c_int64, c_int32, c_int32, _u8p, _i64p, _i64p]),
    "ftk_format_bedgraph_i64": (c_int64, [c_char_p, c_int64, _i64p, c_int64, c_int32, c_void_p, c_int64]),
    "ftk_gzip_compress_batch": (c_int, [_u8p, _i64p, c_int64, c_int32, c_int32, _u8p, _i64p, _i64p]),
    "ftk_zlib_uncompress_batch": (c_int, [_u8p, _i64p, _i64p, c_int64, c_int32, _u8p, _i64p, _i64p]),
}

_lib = None


def lib():
    """Load (once) and return the ctypes handle; raise loudly if unavailable."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise FtkLibraryError(
                f"{SO_PATH} not found. Build it with `python -m finaletoolkit_b200.csrc.build` "
                "(nvcc, sm_100a). finaletoolkit_b200 has no CPU fallback.")
        try:
            h = ctypes.CDLL(SO_PATH)
        except OSError as e:  # pragma: no cover
            raise FtkLibraryError(f"cannot load {SO_PATH}: {e}") from e
        for name, (res, args) in SYMBOLS.items():
            try:
                fn = getattr(h, name)
            except AttributeError as e:
                raise FtkLibraryError(f"{SO_PATH} does not export {name}; rebuild it") from e
            fn.restype = res
            fn.argtypes = args
        _lib = h
    return _lib


def check(code: int, what: str = "") -> None:
    """Raise ``FtkLibraryError`` for a negative return code."""
    if code < 0:
        h = lib()
        msg = h.ftk_error_string(int(code)).decode()
        cuda = h.ftk_last_cuda_error().decode()
        raise FtkLibraryError(f"{what or 'libftk_b200'} failed: {msg}" + (f" [{cuda}]" if cuda else ""))
