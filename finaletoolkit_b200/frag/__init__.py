"""Fragmentation feature extractors of the B200 hot path (names as in finaletoolkit.frag)."""
from ._frag_length import frag_length, frag_length_bins, frag_length_intervals, FragLengthStats
from ._coverage import coverage, single_coverage, CoverageResult
from ._wps import wps
from ._multi_wps import multi_wps
from ._adjust_wps import adjust_wps
from ._cleavage_profile import cleavage_profile, multi_cleavage_profile
from ._coverage_profile import coverage_profile, multi_coverage_profile
from ._vplot import vplot
from ._ocf import OcfResult, ocf
from ._gc_bias import GCBias, gc_bias, read_gc_bias
from ._gc_correct import GCCoverageResult, GCSiteProfile, gc_corrected_coverage, gc_corrected_profile
from ._gc_coverage_profile import gc_corrected_coverage_profile, multi_gc_corrected_coverage_profile
from ._wps_spectrum import WpsSpectrum, wps_spectrum
from ._end_motifs import (EndMotifFreqs, EndMotifsIntervals, region_end_motifs, end_motifs,
                          interval_end_motifs)
from ._delfi import delfi, delfi_gc_correct, delfi_merge_bins, trim_coverage
from ._breakpoint_motifs import (BreakpointMotifFreqs, BreakpointMotifsIntervals, region_breakpoint_motifs,
                                 breakpoint_motifs, interval_breakpoint_motifs)

__all__ = ["frag_length", "frag_length_bins", "frag_length_intervals", "FragLengthStats", "coverage",
           "single_coverage", "CoverageResult", "wps", "multi_wps", "adjust_wps", "cleavage_profile",
           "multi_cleavage_profile", "coverage_profile", "multi_coverage_profile", "vplot", "ocf", "OcfResult", "gc_bias", "GCBias", "read_gc_bias",
           "gc_corrected_coverage", "gc_corrected_profile", "GCCoverageResult", "GCSiteProfile",
           "gc_corrected_coverage_profile", "multi_gc_corrected_coverage_profile", "wps_spectrum",
           "WpsSpectrum", "EndMotifFreqs",
           "EndMotifsIntervals", "region_end_motifs", "end_motifs", "interval_end_motifs", "BreakpointMotifFreqs",
           "BreakpointMotifsIntervals", "region_breakpoint_motifs", "breakpoint_motifs",
           "interval_breakpoint_motifs", "delfi", "delfi_gc_correct", "delfi_merge_bins", "trim_coverage"]
