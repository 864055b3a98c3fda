"""`python -m finaletoolkit_b200.cli <subcommand>`: the hot-path subset of the reference CLI.

Table-driven Click group.  For every in-scope subcommand the flag spellings, parameter names
(== the Python kwarg names, reference cli/_args.py:17-19) and defaults are those of the reference
(cli/commands/__init__.py:87-640); dispatch filters the parameters by the target's signature like
cli/_dispatch.py:96-118 and expands ``--strand`` into both_strands / negative_strand
(cli/_dispatch.py:25-36).  Out-of-scope subcommands (delfi, breakpoint motifs, filter-file, agg-bw,
gap-bed) are not registered.  ``EXTRA_COMMANDS``, ``SITE_COMMANDS``, ``BIAS_COMMANDS``, ``CORRECTION_COMMANDS``,
``GC_TRACK_COMMANDS``, ``SPECTRUM_COMMANDS`` and ``ORIENTATION_COMMANDS`` hold the subcommands this package adds
(coverage-profile, vplot, gc-bias, gc-corrected-coverage / gc-corrected-profile, gc-corrected-coverage-profile,
wps-spectrum, ocf).
"""
from __future__ import annotations

import importlib
import inspect

import click

# (flags..., param name, click kwargs)
def _opt(*flags, **kw):
    return ("opt", flags, kw)


def _arg(name, **kw):
    return ("arg", (name,), kw)


_INPUT = _arg("input_file", metavar="INPUT")
_REF = _opt("-r", "--reference", "reference_file", metavar="FASTA", default=None,
            help="FASTA reference genome. Required for CRAM input.")
_THREADS = _opt("-t", "--threads", "workers", metavar="N", default=1, show_default=True, type=int,
                help="Accepted for compatibility (one process per GPU).")
_VERBOSE = _opt("-v", "--verbose", "verbose", count=True, default=0, help="Increase verbosity.")
_POLICY = _opt("-p", "--intersect-policy", "intersect_policy", type=click.Choice(["midpoint", "any"]),
               default="midpoint", show_default=True, help="'midpoint' or 'any' overlap.")
_STRAND = _opt("--strand", "strand", type=click.Choice(["both", "forward", "reverse"]), default="both",
               show_default=True, help="Fragment strand(s) for end motifs.")


def _out(help_):
    return _opt("-o", "--output", "output_file", metavar="PATH", default="-", show_default=True,
                help=f"{help_} Pass '-' to write to standard output (stdout).")


def _mapq(d):
    return _opt("-q", "--min-mapq", "quality_threshold", metavar="MAPQ", default=d, show_default=True, type=int,
                help="Minimum mapping quality (MAPQ).")


def _minlen(d):
    return _opt("--min-length", "min_length", metavar="BP", default=d, type=int, help="Minimum fragment length.")


def _maxlen(d):
    return _opt("--max-length", "max_length", metavar="BP", default=d, type=int, help="Maximum fragment length.")


def _k(d):
    return _opt("-k", "--kmer-length", "k", metavar="K", default=d, show_default=True, type=int, help="k-mer length.")


_SEP = _opt("-s", "--sep", "sep", default="\t", help="Field separator. Default is a tab.")
_HEADER = _opt("--header", "header", default=0, show_default=True, type=int, help="Header rows to ignore.")

# name -> (module, function, help, params)
COMMANDS = {
    "coverage": ("finaletoolkit_b200.frag", "coverage", "Fragment coverage over BED intervals.", [
        _INPUT, _arg("interval_file", metavar="REGIONS"), _REF, _out("BED file of coverage values."),
        _opt("-n", "--normalize", "normalize", is_flag=True, help="Normalize by total coverage."),
        _opt("--scale-factor", "scale_factor", metavar="X", default=1.0, show_default=True, type=float,
             help="Scale factor for coverage values."),
        _minlen(0), _maxlen(None), _POLICY, _mapq(30), _THREADS, _VERBOSE]),
    "frag-length-bins": ("finaletoolkit_b200.frag", "frag_length_bins", "Fragment lengths grouped into bins.", [
        _INPUT, _REF, _opt("-c", "--contig", "contig", type=str, help="Contig to select fragments from."),
        _opt("-S", "--start", "start", type=int, help="0-based start."),
        _opt("-E", "--stop", "stop", type=int, help="1-based stop."),
        _minlen(0), _maxlen(None), _POLICY,
        _opt("--bin-size", "bin_size", metavar="BP", type=int, default=1, show_default=True, help="Bin width."),
        _out("TSV of binned fragment lengths."),
        _opt("--summary-stats", "summary_stats", is_flag=True, help="Append summary statistics as comments."),
        _opt("--short-threshold", "short_fraction", metavar="BP", default=None, type=int,
             help="Include a short fraction (fragments <= this length)."),
        _opt("--histogram", "histogram_path", metavar="PNG", default=None, help="(unsupported) histogram PNG."),
        _mapq(30), _VERBOSE]),
    "frag-length-intervals": ("finaletoolkit_b200.frag", "frag_length_intervals",
                              "Fragment-length statistics over BED intervals.", [
        _INPUT, _arg("interval_file", metavar="REGIONS"), _REF, _minlen(0), _maxlen(None), _POLICY,
        _out("BED file of fragment-length statistics."),
        _opt("--short-threshold", "short_reads", metavar="BP", default=150, show_default=True, type=int,
             help="Short-fragment length cutoff."),
        _mapq(30), _THREADS, _VERBOSE]),
    "wps": ("finaletoolkit_b200.frag", "multi_wps", "Windowed Protection Score (WPS) over BED sites.", [
        _INPUT, _arg("site_bed", metavar="REGIONS"), _REF,
        _opt("--chrom-sizes", "chrom_sizes", metavar="CHROM_SIZES", help="A .chrom.sizes file."),
        _out("bigWig file of WPS results."),
        _opt("-i", "--interval-size", "interval_size", metavar="BP", default=5000, show_default=True, type=int,
             help="Window size centred on each site."),
        _opt("-W", "--window-size", "window_size", metavar="BP", default=120, show_default=True, type=int,
             help="WPS sliding-window size."),
        _minlen(120), _maxlen(180), _mapq(30), _THREADS, _VERBOSE]),
    "cleavage-profile": ("finaletoolkit_b200.frag", "multi_cleavage_profile", "Cleavage proportion over BED intervals.", [
        _INPUT, _arg("interval_file", metavar="REGIONS"), _arg("chrom_sizes", metavar="CHROM_SIZES"), _REF,
        _out("bigWig file of cleavage proportion."), _minlen(0), _maxlen(None), _mapq(20),
        _opt("--pad-left", "left", metavar="BP", default=0, show_default=True, type=int,
             help="Base pairs to subtract from each start coordinate."),
        _opt("--pad-right", "right", metavar="BP", default=0, show_default=True, type=int,
             help="Base pairs to add to each stop coordinate."),
        _THREADS, _VERBOSE]),
    "adjust-wps": ("finaletoolkit_b200.frag", "adjust_wps", "Median-filter + Savitzky-Golay adjust raw WPS.", [
        _arg("input_file", metavar="INPUT"), _arg("interval_file", metavar="REGIONS"),
        _arg("chrom_sizes", metavar="CHROM_SIZES"), _out("bigWig file of adjusted WPS."),
        _opt("-i", "--interval-size", "interval_size", metavar="BP", default=5000, show_default=True, type=int),
        _opt("-m", "--median-window-size", "median_window_size", metavar="BP", default=1000, show_default=True, type=int),
        _opt("--savgol-window-size", "savgol_window_size", metavar="BP", default=21, show_default=True, type=int),
        _opt("--savgol-poly-deg", "savgol_poly_deg", metavar="DEG", default=2, show_default=True, type=int),
        _opt("--savgol/--no-savgol", "savgol", default=True, help="Apply Savitzky-Golay filtering. On by default."),
        _opt("--mean", "mean", is_flag=True, help="Mean filter instead of median."),
        _opt("--subtract-edges", "subtract_edges", is_flag=True, help="Subtract the mean of the interval edges."),
        _opt("--edge-size", "edge_size", metavar="BP", default=500, show_default=True, type=int),
        _THREADS, _VERBOSE]),
    "end-motifs": ("finaletoolkit_b200.frag", "end_motifs", "Genome-wide 5' end-motif k-mer frequencies.", [
        _INPUT, _arg("refseq_file", metavar="REFERENCE"), _k(4), _minlen(50), _maxlen(None), _STRAND,
        _out("TSV of k-mer frequencies."), _mapq(20), _THREADS, _VERBOSE]),
    "interval-end-motifs": ("finaletoolkit_b200.frag", "interval_end_motifs", "End-motif counts per BED interval.", [
        _INPUT, _arg("refseq_file", metavar="REFERENCE"), _arg("intervals", metavar="REGIONS"), _k(4), _minlen(50),
        _maxlen(None), _STRAND, _out("TSV or CSV of end-motif frequencies."), _mapq(20), _THREADS, _VERBOSE]),
    "delfi": ("finaletoolkit_b200.frag", "delfi", "DELFI short/long fragment counts, ratio and GC content per bin.", [
        _INPUT, _arg("chrom_sizes", metavar="CHROM_SIZES"), _arg("reference_file", metavar="REFERENCE"),
        _arg("bins_file", metavar="BINS"),
        _opt("-b", "--blacklist", "blacklist_file", metavar="BED", help="BED file of regions to ignore."),
        _opt("-g", "--gap-file", "gap_file", metavar="GAPS",
             help="BED4 of telomere/centromere/short_arm annotations."),
        _out("Output file (.bed, .bed.gz, .tsv, or .csv)."),
        _opt("--no-gc-correct", "no_gc_correct", is_flag=True, default=False, help="Skip GC correction."),
        _opt("--remove-nocov/--no-remove-nocov", "remove_nocov", default=True,
             help="Remove the two hg19 regions with no coverage."),
        _opt("--merge-bins/--no-merge-bins", "merge_bins", default=True, help="Merge input bins to 5Mb."),
        _opt("--merge-size", "window_size", metavar="BP", default=5000000, show_default=True, type=int,
             help="Target size of merged genomic intervals."),
        _mapq(30), _THREADS, _VERBOSE]),
    "agg-bw": ("finaletoolkit_b200.utils", "agg_bw", "Strand-aware aggregate of a bigWig signal over BED6 intervals.", [
        _arg("input_file", metavar="INPUT"), _arg("interval_file", metavar="REGIONS"),
        _out("Wiggle file of the aggregate signal over the input intervals."),
        _opt("-m", "--median-window-size", "median_window_size", metavar="BP", default=1, show_default=True, type=int,
             help="Median filter window used upstream (120 replicates Snyder et al.)."),
        _opt("--mean", "mean", is_flag=True, help="Mean instead of sum."), _VERBOSE]),
    "breakpoint-motifs": ("finaletoolkit_b200.frag", "breakpoint_motifs", "Genome-wide breakpoint-motif k-mer frequencies.", [
        _INPUT, _arg("refseq_file", metavar="REFERENCE"), _k(6), _minlen(50), _maxlen(None), _STRAND,
        _out("TSV of k-mer frequencies."), _mapq(20), _THREADS, _VERBOSE]),
    "interval-breakpoint-motifs": ("finaletoolkit_b200.frag", "interval_breakpoint_motifs",
                                   "Breakpoint-motif counts per BED interval.", [
        _INPUT, _arg("refseq_file", metavar="REFERENCE"), _arg("intervals", metavar="REGIONS"), _k(6), _minlen(50),
        _maxlen(None), _STRAND, _out("TSV or CSV of breakpoint-motif frequencies."), _mapq(20), _THREADS, _VERBOSE]),
    "mds": ("finaletoolkit_b200.frag._end_motifs", "_cli_mds", "Motif diversity score from k-mer frequencies.", [
        _arg("file_path", metavar="INPUT", required=False, default="-"), _SEP, _HEADER]),
    "regional-mds": ("finaletoolkit_b200.frag._end_motifs", "_cli_regional_mds", "Regional MDS for each region.", [
        _arg("file_path", metavar="INPUT", required=False, default="-"), _arg("file_out", metavar="OUTPUT"), _SEP,
        _HEADER, _opt("--miller-madow", "miller_madow", is_flag=True, default=False,
                      help="Apply the Miller-Madow bias correction.")]),
}

# subcommands with no reference counterpart, kept apart from the reference's command table
EXTRA_COMMANDS = {
    "coverage-profile": ("finaletoolkit_b200.frag", "multi_coverage_profile",
                         "Per-base fragment depth (or fragment-midpoint count) over BED intervals.", [
        _INPUT, _arg("interval_file", metavar="REGIONS"), _arg("chrom_sizes", metavar="CHROM_SIZES"), _REF,
        _out("bigWig or gzipped bedGraph of per-base depth."), _minlen(None), _maxlen(None), _mapq(30),
        _opt("--pad-left", "left", metavar="BP", default=0, show_default=True, type=int,
             help="Base pairs to subtract from each start coordinate."),
        _opt("--pad-right", "right", metavar="BP", default=0, show_default=True, type=int,
             help="Base pairs to add to each stop coordinate."),
        _opt("--midpoint", "midpoint", is_flag=True, help="Count fragment midpoints instead of spanned bases."),
        _opt("--scale-factor", "scale_factor", metavar="X", default=1.0, show_default=True, type=float,
             help="Scale factor for depth values."),
        _opt("-n", "--normalize", "normalize", is_flag=True,
             help="Divide the scale factor by the number of passing fragments in the file."),
        _THREADS, _VERBOSE]),
}

# site-aggregate subcommands added here, in their own table so COMMANDS / EXTRA_COMMANDS keep their exact sets
SITE_COMMANDS = {
    "vplot": ("finaletoolkit_b200.frag", "vplot",
              "Fragment-length x midpoint-offset counts (V-plot) summed over BED sites.", [
        _INPUT, _arg("site_bed", metavar="SITES"), _REF, _out("TSV (or .tsv.gz) of the V-plot matrix."),
        _opt("--flank", "flank", metavar="BP", default=1000, show_default=True, type=int,
             help="Largest midpoint offset from a site centre."),
        _opt("--min-length", "min_length", metavar="BP", default=0, show_default=True, type=int,
             help="Minimum fragment length (first row)."),
        _opt("--max-length", "max_length", metavar="BP", default=500, show_default=True, type=int,
             help="Maximum fragment length (last row)."),
        _mapq(30), _THREADS, _VERBOSE]),
}

# bias-measurement subcommands added here, in their own table for the same reason
BIAS_COMMANDS = {
    "gc-bias": ("finaletoolkit_b200.frag", "gc_bias",
                "Observed and expected fragment counts by length and G+C content, and their ratio.", [
        _INPUT, _arg("refseq_file", metavar="REFERENCE"),
        _opt("--regions", "interval_file", metavar="BED", default=None,
             help="BED of regions to count in (default: every contig the input and the reference share)."),
        _REF, _out("TSV (or .tsv.gz) of counts and ratios by length and G+C bases."),
        _opt("--min-length", "min_length", metavar="BP", default=50, show_default=True, type=int,
             help="Minimum fragment length (first row)."),
        _opt("--max-length", "max_length", metavar="BP", default=500, show_default=True, type=int,
             help="Maximum fragment length (last row, at most 1024)."),
        _mapq(30), _THREADS, _VERBOSE]),
}

# subcommands that apply the GC model, in their own table for the same reason
_GC_MODEL = [
    _opt("--gc-bias", "gc_bias", metavar="TSV", default=None,
         help="GC model: a gc-bias table (default: fit one on INPUT first)."),
    _opt("--gc-regions", "gc_regions", metavar="BED", default=None,
         help="Regions to fit the GC model over (default: every contig the input and the reference share)."),
    _opt("--min-length", "min_length", metavar="BP", default=None, type=int,
         help="Minimum fragment length (default: the model's; 50 when fitting)."),
    _opt("--max-length", "max_length", metavar="BP", default=None, type=int,
         help="Maximum fragment length (default: the model's; 500 when fitting)."),
]
CORRECTION_COMMANDS = {
    "gc-corrected-coverage": ("finaletoolkit_b200.frag", "gc_corrected_coverage",
                              "Plain and GC-corrected fragment-midpoint counts over BED intervals.", [
        _INPUT, _arg("refseq_file", metavar="REFERENCE"), _arg("interval_file", metavar="REGIONS"), _REF,
        _out("TSV (or .tsv.gz) of plain and GC-corrected counts per interval."), *_GC_MODEL,
        _mapq(30), _THREADS, _VERBOSE]),
    "gc-corrected-profile": ("finaletoolkit_b200.frag", "gc_corrected_profile",
                             "Plain and GC-corrected fragment-midpoint profiles summed over BED sites.", [
        _INPUT, _arg("refseq_file", metavar="REFERENCE"), _arg("site_bed", metavar="SITES"), _REF,
        _out("TSV (or .tsv.gz) of plain and GC-corrected counts by midpoint offset."),
        _opt("--flank", "flank", metavar="BP", default=1000, show_default=True, type=int,
             help="Largest midpoint offset from a site centre."),
        *_GC_MODEL, _mapq(30), _THREADS, _VERBOSE]),
}

# GC-corrected per-base tracks, in their own table for the same reason
GC_TRACK_COMMANDS = {
    "gc-corrected-coverage-profile": ("finaletoolkit_b200.frag", "multi_gc_corrected_coverage_profile",
                                      "Per-base GC-corrected fragment depth (or fragment-midpoint sum) over BED "
                                      "intervals.", [
        _INPUT, _arg("refseq_file", metavar="REFERENCE"), _arg("interval_file", metavar="REGIONS"),
        _arg("chrom_sizes", metavar="CHROM_SIZES"), _REF,
        _out("bigWig or gzipped bedGraph of per-base GC-corrected depth."), *_GC_MODEL, _mapq(30),
        _opt("--pad-left", "left", metavar="BP", default=0, show_default=True, type=int,
             help="Base pairs to subtract from each start coordinate."),
        _opt("--pad-right", "right", metavar="BP", default=0, show_default=True, type=int,
             help="Base pairs to add to each stop coordinate."),
        _opt("--midpoint", "midpoint", is_flag=True, help="Sum at fragment midpoints instead of spanned bases."),
        _opt("--scale-factor", "scale_factor", metavar="X", default=1.0, show_default=True, type=float,
             help="Scale factor for depth values."),
        _opt("-n", "--normalize", "normalize", is_flag=True,
             help="Divide the scale factor by the number of passing fragments in the file."),
        _THREADS, _VERBOSE]),
}

# subcommands that transform WPS further, in their own table for the same reason
SPECTRUM_COMMANDS = {
    "wps-spectrum": ("finaletoolkit_b200.frag", "wps_spectrum",
                     "Periodograms of the (adjusted) WPS of BED windows at integer periods (nucleosome repeat).", [
        _INPUT, _arg("site_bed", metavar="REGIONS"), _REF,
        _opt("--chrom-sizes", "chrom_sizes", metavar="CHROM_SIZES", help="A .chrom.sizes file."),
        _out("TSV (or .tsv.gz) of one periodogram per BED row."),
        _opt("--min-period", "min_period", metavar="BP", default=120, show_default=True, type=int,
             help="Shortest period (at least 2)."),
        _opt("--max-period", "max_period", metavar="BP", default=280, show_default=True, type=int,
             help="Longest period (at most 1024)."),
        _opt("--adjust/--no-adjust", "adjust", default=True,
             help="Median-filter + Savitzky-Golay adjust the WPS first. On by default."),
        _opt("-m", "--median-window-size", "median_window_size", metavar="BP", default=1000, show_default=True,
             type=int),
        _opt("--savgol/--no-savgol", "savgol", default=True, help="Apply Savitzky-Golay filtering. On by default."),
        _opt("--savgol-window-size", "savgol_window_size", metavar="BP", default=21, show_default=True, type=int),
        _opt("--savgol-poly-deg", "savgol_poly_deg", metavar="DEG", default=2, show_default=True, type=int),
        _opt("-W", "--window-size", "window_size", metavar="BP", default=120, show_default=True, type=int,
             help="WPS sliding-window size."),
        _minlen(120), _maxlen(180), _mapq(30), _THREADS, _VERBOSE]),
}

# fragment-end orientation subcommands, in their own table for the same reason
ORIENTATION_COMMANDS = {
    "ocf": ("finaletoolkit_b200.frag", "ocf",
            "Orientation-aware fragment end profiles (OCF) summed over the sites of each BED file.", [
        _INPUT, _arg("site_beds", metavar="SITES", nargs=-1, required=True), _REF,
        _out("TSV (or .tsv.gz) of the OCF value of each site set."),
        _opt("--profiles", "profile_file", metavar="PATH", default=None,
             help="TSV (or .tsv.gz) of the upstream and downstream end counts of each site set."),
        _opt("--flank", "flank", metavar="BP", default=1000, show_default=True, type=int,
             help="Largest end offset from a site centre (at most 8192)."),
        _opt("--peak-offset", "peak_offset", metavar="BP", default=60, show_default=True, type=int,
             help="Centre of the OCF peak windows."),
        _opt("--peak-width", "peak_width", metavar="BP", default=20, show_default=True, type=int,
             help="Width of the OCF peak windows."),
        _minlen(None), _maxlen(None), _mapq(30), _THREADS, _VERBOSE]),
}


def run(module: str, func: str, params: dict):
    """Import the target lazily, translate --strand, keep only the kwargs it accepts, call it."""
    params = dict(params)
    strand = params.pop("strand", None)
    if strand is not None:
        params["both_strands"] = strand == "both"
        params["negative_strand"] = strand == "reverse"
    target = getattr(importlib.import_module(module), func)
    accepted = inspect.signature(target).parameters
    return target(**{k: v for k, v in params.items() if k in accepted})


def _make(name, module, func, help_, spec):
    def callback(**params):
        run(module, func, params)

    cmd = callback
    for kind, names, kw in reversed(spec):
        cmd = (click.argument(*names, **kw) if kind == "arg" else click.option(*names, **kw))(cmd)
    return click.command(name, help=help_)(cmd)


@click.group(context_settings={"help_option_names": ["-h", "--help"]})
def main_cli():
    """finaletoolkit_b200: the B200-native hot path of FinaleToolkit."""


for _name, (_module, _func, _help, _spec) in {**COMMANDS, **EXTRA_COMMANDS, **SITE_COMMANDS, **BIAS_COMMANDS,
                                              **CORRECTION_COMMANDS, **GC_TRACK_COMMANDS, **SPECTRUM_COMMANDS,
                                              **ORIENTATION_COMMANDS}.items():
    main_cli.add_command(_make(_name, _module, _func, _help, _spec))


if __name__ == "__main__":
    main_cli()
