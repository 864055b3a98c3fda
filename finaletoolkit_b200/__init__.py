"""finaletoolkit_b200 - B200-native (sm_100a CUDA) implementation of FinaleToolkit's
per-fragment interval-feature hot path, behind the reference's own Python API.

Flat namespace resolved lazily like the reference's (finaletoolkit/__init__.py:49-128):
``finaletoolkit_b200.wps``, ``.multi_wps``, ``.adjust_wps``, ``.coverage``, ...
Importing the package needs neither CUDA nor torch; calling a feature without a CUDA
device / libftk_b200.so raises ``FtkLibraryError`` (there is no CPU fallback).
"""
from __future__ import annotations

__version__ = "0.1.0"

_SUBMODULES = ("cli", "frag", "genome", "io", "utils", "device", "synth", "exceptions", "sharding")

_EXPORTS = {
    "frag_length": ("frag", "frag_length"), "frag_length_bins": ("frag", "frag_length_bins"),
    "frag_length_intervals": ("frag", "frag_length_intervals"),
    "coverage": ("frag", "coverage"), "single_coverage": ("frag", "single_coverage"),
    "wps": ("frag", "wps"), "multi_wps": ("frag", "multi_wps"), "adjust_wps": ("frag", "adjust_wps"),
    "cleavage_profile": ("frag", "cleavage_profile"), "multi_cleavage_profile": ("frag", "multi_cleavage_profile"),
    "coverage_profile": ("frag", "coverage_profile"), "multi_coverage_profile": ("frag", "multi_coverage_profile"),
    "vplot": ("frag", "vplot"), "gc_bias": ("frag", "gc_bias"), "GCBias": ("frag", "GCBias"),
    "read_gc_bias": ("frag", "read_gc_bias"), "gc_corrected_coverage": ("frag", "gc_corrected_coverage"),
    "gc_corrected_profile": ("frag", "gc_corrected_profile"), "GCCoverageResult": ("frag", "GCCoverageResult"),
    "GCSiteProfile": ("frag", "GCSiteProfile"), "wps_spectrum": ("frag", "wps_spectrum"),
    "WpsSpectrum": ("frag", "WpsSpectrum"),
    "end_motifs": ("frag", "end_motifs"), "region_end_motifs": ("frag", "region_end_motifs"),
    "interval_end_motifs": ("frag", "interval_end_motifs"),
    "EndMotifFreqs": ("frag", "EndMotifFreqs"), "EndMotifsIntervals": ("frag", "EndMotifsIntervals"),
    "delfi": ("frag", "delfi"), "delfi_gc_correct": ("frag", "delfi_gc_correct"),
    "delfi_merge_bins": ("frag", "delfi_merge_bins"), "trim_coverage": ("frag", "trim_coverage"),
    "breakpoint_motifs": ("frag", "breakpoint_motifs"), "region_breakpoint_motifs": ("frag", "region_breakpoint_motifs"),
    "interval_breakpoint_motifs": ("frag", "interval_breakpoint_motifs"),
    "BreakpointMotifFreqs": ("frag", "BreakpointMotifFreqs"),
    "BreakpointMotifsIntervals": ("frag", "BreakpointMotifsIntervals"),
    "frag_generator": ("utils", "frag_generator"), "frag_array": ("utils", "frag_array"),
    "frags_in_region": ("utils", "frags_in_region"), "get_intervals": ("utils", "get_intervals"),
    "gen_kmers": ("utils", "gen_kmers"), "reverse_complement": ("utils", "reverse_complement"),
    "chrom_sizes_to_dict": ("utils", "chrom_sizes_to_dict"), "chrom_sizes_to_list": ("utils", "chrom_sizes_to_list"),
    "agg_bw": ("utils", "agg_bw"), "overlaps": ("utils", "overlaps"),
    "GenomeGaps": ("genome", "GenomeGaps"), "ContigGaps": ("genome", "ContigGaps"),
    "ReferenceWrapper": ("io", "ReferenceWrapper"), "AlignmentWrapper": ("io", "AlignmentWrapper"),
    "Fragment": ("io", "Fragment"),
    # the exception hierarchy is part of the flat namespace too (finaletoolkit/__init__.py:30-40)
    "FinaleToolkitError": ("exceptions", "FinaleToolkitError"), "InvalidInputError": ("exceptions", "InvalidInputError"),
    "UnsupportedFormatError": ("exceptions", "UnsupportedFormatError"),
    "MissingReferenceError": ("exceptions", "MissingReferenceError"), "MissingIndexError": ("exceptions", "MissingIndexError"),
    "ContigNotFoundError": ("exceptions", "ContigNotFoundError"), "ContigMismatchError": ("exceptions", "ContigMismatchError"),
    "OutOfBoundsError": ("exceptions", "OutOfBoundsError"),
}
_ALIASES = {"end_motif": "end_motifs", "breakpoint_motif": "breakpoint_motifs"}


def __getattr__(name: str):
    import importlib
    if name in _SUBMODULES:
        return importlib.import_module(f".{name}", __name__)
    target = _ALIASES.get(name, name)
    if target in _EXPORTS:
        sub, attr = _EXPORTS[target]
        value = getattr(importlib.import_module(f".{sub}", __name__), attr)
        globals()[name] = value
        return value
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")


def __dir__():
    return sorted(set(globals()) | set(_SUBMODULES) | set(_EXPORTS) | set(_ALIASES))
