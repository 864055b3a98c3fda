/*
 * ftk_b200.h - C ABI of the B200-native FinaleToolkit hot path.
 *
 * FinaleToolkit (the reference, /root/reference/src/finaletoolkit) has no FFI:
 * its seam is the Python function layer.  This header is the array-level seam
 * a maintainer would bind (ctypes, see INTEGRATION.md) in place of the
 * reference's per-interval Python/numba loops.  Each entry point cites the
 * reference code it replaces.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch types.
 *   - `*_dev` pointers are DEVICE pointers; `*_host` are host pointers.
 *   - All device entry points are asynchronous on `stream` (a cudaStream_t
 *     passed as void*), allocate nothing, and keep no global state.
 *   - Return 0 on success, a negative FTK_E_* code otherwise
 *     (ftk_error_string() describes it).  No exceptions cross the ABI.
 *   - Fragments of ONE contig, sorted ascending by start (the order of a
 *     tabix-indexed .frag.gz), as columns: start,stop int32; mapq,strand uint8.
 *     Coordinates are 0-based half-open and must fit int32.
 *   - FTK_NONE stands for Python None (unbounded) in length / region bounds.
 */
#ifndef FTK_B200_H
#define FTK_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FTK_ABI_VERSION 2
#define FTK_NONE INT32_MIN

#define FTK_OK 0
#define FTK_E_INVALID -1   /* bad argument (null pointer, negative size, ...) */
#define FTK_E_CUDA -2      /* a CUDA runtime call or launch failed            */
#define FTK_E_RANGE -3     /* a size exceeds what the kernel supports         */
#define FTK_E_IO -4        /* file unreadable or not valid (b)gzip            */

/* `pooled` modes of ftk_interval_hist_u64 */
#define FTK_POOL_NONE 0       /* counts and histogram rows per interval            */
#define FTK_POOL_ALL 1        /* counts and histogram pooled into row 0            */
#define FTK_POOL_HIST_ONLY 2  /* counts per interval, ONE pooled histogram (row 0) */

#define FTK_POLICY_MIDPOINT 0
#define FTK_POLICY_ANY 1

/* Positions per WPS tile (one CTA).  Intervals longer than this are split. */
#define FTK_WPS_TILE 5119 /* 5120 smem slots minus one guard slot for odd windows */

typedef void *ftk_stream_t; /* cudaStream_t */

int ftk_abi_version(void);
const char *ftk_error_string(int code);
/* last CUDA error text recorded by this library on the calling thread ("" if none) */
const char *ftk_last_cuda_error(void);

/* ------------------------------------------------- packed fragment columns
 * Wire format host -> HBM, replacing the per-interval text stream of io/alignment.py:270-302 /
 * utils/_frag_generator.py:124-130 (PCIe is the end-to-end limit: 3.06 - 4.06 B per fragment instead of 10).
 *   words[i]  = dstart | length << 11 | strand << 23 | mapq << 24   (uint32; dstart = start[i] - start[i-1],
 *               0 for the first fragment of a block; dstart < 2048, length < 4096)
 *   anchors[b] = start of the first fragment of block b (FTK_PACK_BLOCK fragments), or -1 - r when the
 *               block does not fit the fields: its rows are then stored verbatim as raw block r
 *               (raw_*[r * FTK_PACK_BLOCK ...]).  Lossless for any int32 columns.
 * words holds n_blocks * FTK_PACK_BLOCK entries (zero padded), n_blocks = ceil(n / FTK_PACK_BLOCK). */
#define FTK_PACK_BLOCK 64

/* record_bytes = 4: the 32-bit records above (words: 64 per block).  record_bytes = 3: 24-bit records
 * dstart (6 bits) | length << 6 (9 bits) | strand << 15 | mapq << 16, stored back to back (48 words per
 * block, 3.0625 B per fragment); a block with a gap >= 64 bp or a fragment >= 512 bp escapes to the raw
 * columns.  Same anchors, same raw columns, same losslessness.
 * Host (decoder side), multi-threaded (threads <= 0: all cores).  Returns the number of raw blocks.
 * With words_host == NULL only counts them (so the caller can size the raw columns);
 * FTK_E_RANGE if raw_capacity_blocks is too small.  mapq_host / strand_host may be NULL (255 / 0). */
int64_t ftk_pack_fragments_host(const int32_t *start_host, const int32_t *stop_host, const uint8_t *mapq_host,
                                const uint8_t *strand_host, int64_t n, int32_t threads,
                                uint32_t *words_host, int32_t *anchors_host,
                                int32_t *raw_start_host, int32_t *raw_stop_host, uint8_t *raw_mapq_host,
                                uint8_t *raw_strand_host, int64_t raw_capacity_blocks, int32_t record_bytes);

/* Device: words / anchors (of the first block to unpack; a slice of a contig may start at any block
 * boundary) + the contig's raw columns -> int32 start / stop, uint8 mapq / strand (either may be NULL)
 * of n fragments.  start_dev / stop_dev / words_dev must be 8-byte aligned. */
int ftk_unpack_fragments(const uint32_t *words_dev, const int32_t *anchors_dev,
                         const int32_t *raw_start_dev, const int32_t *raw_stop_dev,
                         const uint8_t *raw_mapq_dev, const uint8_t *raw_strand_dev, int64_t n_raw_blocks,
                         int64_t n, int32_t *start_dev, int32_t *stop_dev, uint8_t *mapq_dev, uint8_t *strand_dev,
                         int32_t record_bytes, ftk_stream_t stream);

/* ------------------------------------------------- per-interval length statistics (host)
 * frag_length_intervals' statistics (frag/_frag_length.py:156-172, :204-238) for n_rows intervals at
 * once from the rows ftk_interval_hist_u64 produced (hist narrowed to int32, first_seen as is): mean,
 * the reference's off-by-one median, stdev accumulated in the dict's first-seen order with the same
 * libm pow() calls CPython makes, min, max, count, fraction of lengths <= short_reads.  Empty rows get
 * -1 in every field.  Host, multi-threaded (threads <= 0: all cores). */
int ftk_length_stats_host(const int32_t *hist_host, const int32_t *first_seen_host, int64_t n_rows,
                          int32_t n_bins, int32_t short_reads, int32_t threads,
                          double *mean, double *median, double *stdev, int64_t *vmin, int64_t *vmax,
                          int64_t *count, double *frac_short);

/* ------------------------------------------------------------------ WPS
 * Replaces the per-position loop of wps() - frag/_wps.py:176-188 calling the
 * numba kernel _single_nt_wps (frag/_wps.py:25-53) - and the per-interval
 * fragment selection frag_array(..., start=minimum, stop=maximum) of
 * frag/_wps.py:156-169 (mapq filter io/alignment.py:291; inclusive length
 * filter and midpoint policy utils/_frag_generator.py:117-123).
 *
 * Work unit = tile: positions [p0, p0+len) of one interval, len <= FTK_WPS_TILE.
 * A fragment takes part in a tile iff mapq >= min_mapq, min_len <= L <= max_len
 * and mid_lo <= (start+stop)/2 < mid_hi, where [mid_lo, mid_hi) is the
 * interval's padded fetch window [max(S-max_len,0), min(E+max_len,chrom_size)).
 * out[tile_out_off + (c - p0)] = WPS at position c, int32 (the reference's
 * int64 column; abs(WPS) <= local depth).
 */

/* Host helper: expand intervals into tiles.  Pass NULL outputs to count only.
 * Returns the number of tiles (>= 0) or a negative error code.
 * ivl_out_off[k] = offset of interval k's first position in `out`. */
int64_t ftk_wps_plan_tiles(const int64_t *ivl_start, const int64_t *ivl_stop,
                           const int64_t *ivl_out_off, int64_t n_ivl,
                           int64_t chrom_size, int32_t max_len,
                           int32_t *tile_p0, int32_t *tile_len,
                           int32_t *tile_mid_lo, int32_t *tile_mid_hi,
                           int64_t *tile_out_off);

/* Per-tile fragment index ranges (binary search over the sorted starts) into
 * scratch_dev: int64[2 * n_tiles].  Called implicitly by ftk_wps_tiles_i32
 * unless ranges_ready != 0. */
int ftk_wps_tile_ranges(const int32_t *frag_start_dev, int64_t n_frag,
                        const int32_t *tile_p0_dev, const int32_t *tile_len_dev, int64_t n_tiles,
                        int32_t window_size, int32_t max_len, int64_t *scratch_dev,
                        ftk_stream_t stream);

int ftk_wps_tiles_i32(const int32_t *frag_start_dev, const int32_t *frag_stop_dev,
                      const uint8_t *frag_mapq_dev /* NULL = no mapq filter */, int64_t n_frag,
                      const int32_t *tile_p0_dev, const int32_t *tile_len_dev,
                      const int32_t *tile_mid_lo_dev, const int32_t *tile_mid_hi_dev,
                      const int64_t *tile_out_off_dev, int64_t n_tiles,
                      int32_t window_size, int32_t min_len, int32_t max_len, int32_t min_mapq,
                      int32_t ranges_ready, int64_t *scratch_dev, int32_t *out_dev,
                      ftk_stream_t stream);

/* Same as ftk_wps_tiles_i32 with int16 scores: halves the device->host bytes of the
 * end-to-end path.  *overflow_flag_dev (caller zeroes it) is OR-ed with 1 if any score
 * does not fit int16 (needs a > 32767-fold pile-up); the caller then reruns in int32. */
int ftk_wps_tiles_i16(const int32_t *frag_start_dev, const int32_t *frag_stop_dev,
                      const uint8_t *frag_mapq_dev, int64_t n_frag,
                      const int32_t *tile_p0_dev, const int32_t *tile_len_dev,
                      const int32_t *tile_mid_lo_dev, const int32_t *tile_mid_hi_dev,
                      const int64_t *tile_out_off_dev, int64_t n_tiles,
                      int32_t window_size, int32_t min_len, int32_t max_len, int32_t min_mapq,
                      int32_t ranges_ready, int64_t *scratch_dev, int16_t *out_dev,
                      int32_t *overflow_flag_dev, ftk_stream_t stream);

/* Same, scores as int8 (a quarter of the int32 bytes device->host).  Exact whenever every |WPS| <= 127
 * (local depth below 128, the case for ordinary whole-genome coverage); otherwise *overflow_flag_dev
 * is set and the caller reruns with ftk_wps_tiles_i16 / _i32. */
int ftk_wps_tiles_i8(const int32_t *frag_start_dev, const int32_t *frag_stop_dev,
                      const uint8_t *frag_mapq_dev, int64_t n_frag,
                      const int32_t *tile_p0_dev, const int32_t *tile_len_dev,
                      const int32_t *tile_mid_lo_dev, const int32_t *tile_mid_hi_dev,
                      const int64_t *tile_out_off_dev, int64_t n_tiles,
                      int32_t window_size, int32_t min_len, int32_t max_len, int32_t min_mapq,
                      int32_t ranges_ready, int64_t *scratch_dev, int8_t *out_dev,
                      int32_t *overflow_flag_dev, ftk_stream_t stream);

/* Fused pass: WPS + per-interval coverage counts + ONE pooled length histogram in a single sweep
 * over the fragments (the three reference loops frag/_wps.py:176-188, frag/_coverage.py:117-130 with
 * intersect_policy="midpoint", frag/_frag_length.py:147-153 over the same intervals).
 * tile_ivl_dev[t] = index of the interval tile t belongs to, with bit 31 set on the interval's FIRST tile.  counts_dev[ivl] (uint64, ACCUMULATED,
 * caller zeroes) += fragments with mapq >= cov_min_mapq, cov_min_len <= L <= cov_max_len (FTK_NONE =
 * unbounded) whose midpoint lies in the interval; hist_dev[L] (uint64[n_bins], ACCUMULATED) += 1 for
 * each counted fragment with L < n_bins (n_bins = 0: no histogram, hist_dev may be NULL).
 * max_frag_len = longest fragment of the contig (bounds the candidate search).
 * out_kind: 0 = int32 scores, 1 = int16, 2 = int8 (overflow protocol of ftk_wps_tiles_i16/_i8;
 * overflow_flag_dev may be NULL for int32).  scratch_dev: int64[2 * n_tiles] = the per-tile fragment
 * ranges of ftk_wps_cov_tile_ranges (wider on the left than ftk_wps_tile_ranges': every fragment whose
 * midpoint can fall into the tile); computed here unless ranges_ready != 0.
 * Every interval is an independent stream (overlapping intervals each count their own fragments,
 * and the pooled histogram gains one entry per (interval, fragment) pair like the reference's loop). */
/* zero_counts_dev / zero_hist_dev (may be NULL with a zero length): accumulators this prepass also
 * clears (n_counts / n_hist uint64 entries), so that a step is two launches. */
int ftk_wps_cov_tile_ranges(const int32_t *frag_start_dev, int64_t n_frag,
                            const int32_t *tile_p0_dev, const int32_t *tile_len_dev, int64_t n_tiles,
                            int32_t window_size, int32_t max_len, int32_t cov_max_len, int32_t max_frag_len,
                            int64_t *scratch_dev, uint64_t *zero_counts_dev, int64_t n_counts,
                            uint64_t *zero_hist_dev, int64_t n_hist, ftk_stream_t stream);

int ftk_wps_cov_tiles(const int32_t *frag_start_dev, const int32_t *frag_stop_dev,
                      const uint8_t *frag_mapq_dev, int64_t n_frag, int32_t max_frag_len,
                      const int32_t *tile_p0_dev, const int32_t *tile_len_dev,
                      const int32_t *tile_mid_lo_dev, const int32_t *tile_mid_hi_dev,
                      const int64_t *tile_out_off_dev, const int32_t *tile_ivl_dev, int64_t n_tiles,
                      int32_t window_size, int32_t min_len, int32_t max_len, int32_t min_mapq,
                      int32_t cov_min_len, int32_t cov_max_len, int32_t cov_min_mapq, int32_t n_bins,
                      int32_t ranges_ready, int64_t *scratch_dev, int32_t out_kind, void *out_dev, int32_t *overflow_flag_dev,
                      uint64_t *counts_dev, uint64_t *hist_dev, ftk_stream_t stream);

/* ------------------------------------------- coverage / fragment lengths
 * Fragment stream of a region (S, E) - FTK_NONE = None - exactly as the
 * reference builds it: tabix overlap rows (io/alignment.py:270-302:
 * stop > S and start < E, mapq >= min_mapq), inclusive length filter and
 * intersect policy (utils/_frag_generator.py:21-55,117-123).
 *
 * ftk_interval_hist_u64 replaces, per interval,
 *   - single_coverage's counting loop, frag/_coverage.py:117-130  -> counts
 *   - _distribution_from_gen, frag/_frag_length.py:147-153        -> hist (+ first_seen)
 * counts[row] += number of stream fragments; hist[row*n_bins + L] += 1 for
 * L < n_bins; first_seen[row*n_bins + L] = min fragment index with that
 * length (the dict's first-insertion order, which the reference's fp sums
 * follow, frag/_frag_length.py:213-217).  row = interval index, or 0 when
 * pooled (FTK_POOL_*: FTK_POOL_HIST_ONLY keeps per-interval counts and pools only
 * the histogram - coverage + length distribution in one pass).  Outputs are ACCUMULATED: the caller zeroes counts/hist and fills
 * first_seen with INT32_MAX.  n_bins == 0: counts only (hist/first_seen NULL).
 * Each interval is processed by `splits` CTAs.  scratch_dev: int64[2*n_ivl].
 * max_frag_len = max(stop-start) over the contig (bounds the left halo).
 */
int ftk_interval_hist_u64(const int32_t *frag_start_dev, const int32_t *frag_stop_dev,
                          const uint8_t *frag_mapq_dev, int64_t n_frag, int32_t max_frag_len,
                          const int32_t *ivl_start_dev, const int32_t *ivl_stop_dev, int64_t n_ivl,
                          int32_t policy, int32_t min_len, int32_t max_len, int32_t min_mapq,
                          int32_t n_bins, int32_t pooled, int32_t splits,
                          int64_t *scratch_dev, uint64_t *counts_dev, uint64_t *hist_dev,
                          int32_t *first_seen_dev, ftk_stream_t stream);

/* frag_length(): lengths (stop-start) of the stream of one region in stream
 * order, frag/_frag_length.py:290-308.  out_dev must hold n_frag int32;
 * *n_out_dev receives the count.  scratch_dev: int64[scratch_len],
 * scratch_len >= 2 + nb + (nb+1)/2 with nb = ceil(n_frag/1024) + 1. */
int ftk_frag_lengths_i32(const int32_t *frag_start_dev, const int32_t *frag_stop_dev,
                         const uint8_t *frag_mapq_dev, int64_t n_frag, int32_t max_frag_len,
                         int32_t region_start, int32_t region_stop, int32_t policy,
                         int32_t min_len, int32_t max_len, int32_t min_mapq,
                         int64_t *scratch_dev, int64_t scratch_len, int32_t *out_dev,
                         int64_t *n_out_dev, ftk_stream_t stream);

/* ------------------------------------------------------------ end motifs
 * Replaces the per-fragment loop of region_end_motifs, frag/_end_motifs.py:115-179
 * (and its Pool drivers frag/_motif_common.py:580-610, 633-687).
 * seq_words_dev: 2 bits per base, base i in bits 2*(i%16).. of word i/16, codes
 * A0 C1 G2 T3; nmask_words_dev: 1 bit per base (bit i%32 of word i/32), set for
 * N.  Both padded with >= 2 spare words.  counts[row*4^k + index] += 1 with
 * index in itertools.product("ACGT") order (utils/utils.py:388-410); row =
 * interval, or 0 when `pooled`.  strand_mode 0 = both strands, 1 = forward only,
 * 2 = negative only.  *error_flag_dev is OR-ed with 1 when the reference would
 * raise RuntimeError (reverse k-mer out of bounds, frag/_end_motifs.py:144-151).
 * 1 <= k <= 12.  scratch_dev: int64[2*n_ivl]. */
int ftk_end_motif_hist_u64(const int32_t *frag_start_dev, const int32_t *frag_stop_dev,
                           const uint8_t *frag_mapq_dev, const uint8_t *frag_strand_dev,
                           int64_t n_frag, int32_t max_frag_len,
                           const uint32_t *seq_words_dev, const uint32_t *nmask_words_dev,
                           int64_t contig_len,
                           const int32_t *ivl_start_dev, const int32_t *ivl_stop_dev, int64_t n_ivl,
                           int32_t k, int32_t strand_mode, int32_t min_mapq,
                           int32_t pooled, int32_t splits,
                           int64_t *scratch_dev, uint64_t *counts_dev, int32_t *error_flag_dev,
                           ftk_stream_t stream);

/* Breakpoint motifs: the per-fragment loop of region_breakpoint_motifs,
 * frag/_breakpoint_motifs.py:120-186 (k-mers centred on the two breakpoints, h = k/2:
 * forward ref[fs-h, fs+h), reverse revcomp(ref[fe-h, fe+h))).  Same operands, layout,
 * strand_mode and scratch as ftk_end_motif_hist_u64.  Fragments with fs-h < 0 or
 * fs+h >= contig_len are skipped, an out-of-bounds reverse window skips that end only, and
 * an odd k never counts anything (the reference's "length discrepancy" branch); there is no
 * error path. */
int ftk_breakpoint_motif_hist_u64(const int32_t *frag_start_dev, const int32_t *frag_stop_dev,
                                  const uint8_t *frag_mapq_dev, const uint8_t *frag_strand_dev,
                                  int64_t n_frag, int32_t max_frag_len,
                                  const uint32_t *seq_words_dev, const uint32_t *nmask_words_dev,
                                  int64_t contig_len,
                                  const int32_t *ivl_start_dev, const int32_t *ivl_stop_dev,
                                  int64_t n_ivl, int32_t k, int32_t strand_mode, int32_t min_mapq,
                                  int32_t pooled, int32_t splits,
                                  int64_t *scratch_dev, uint64_t *counts_dev, ftk_stream_t stream);

/* ----------------------------------------------------------- DELFI windows
 * Replaces the per-fragment loop + GC count of _delfi_single_window, frag/_delfi.py:404-511 (run
 * once per 100 kb bin by the Pool at frag/_delfi.py:283-294) for all bins of one contig.
 * counts_dev: uint64[n_win][4] = {short (100..150), long (151..220), num_frags, G+C bases};
 * all four columns are accumulated (zero them first); column 3 only when seq_words_dev is given
 * (bins that are not valid reference intervals add 0, :472-482).
 * Fragment filter: tabix overlap with the bin, mapq >= min_mapq, 100 <= L <= 220, midpoint in the
 * bin, not inside a blacklist region, not in_tcmere (genome/gaps.py:226-248).
 * Blacklist: bl_off_dev int32[n_win+1] indexes bl_start_dev/bl_stop_dev, the regions contained in
 * each bin (frag/_delfi.py:110-127); NULL = no blacklist.
 * gaps5_host (HOST pointer, or NULL = no gap track for the contig): {centromere start, centromere
 * stop, n_telomeres, max telomere start, min telomere stop}.
 * seq/nmask layout as for ftk_end_motif_hist_u64.  scratch_dev: int64[2*n_win]. */
int ftk_delfi_windows_u64(const int32_t *frag_start_dev, const int32_t *frag_stop_dev,
                          const uint8_t *frag_mapq_dev, int64_t n_frag, int32_t max_frag_len,
                          const uint32_t *seq_words_dev, const uint32_t *nmask_words_dev,
                          int64_t contig_len,
                          const int32_t *win_start_dev, const int32_t *win_stop_dev, int64_t n_win,
                          const int32_t *bl_off_dev, const int32_t *bl_start_dev,
                          const int32_t *bl_stop_dev, const int32_t *gaps5_host,
                          int32_t min_mapq, int32_t splits,
                          int64_t *scratch_dev, uint64_t *counts_dev, ftk_stream_t stream);

/* ------------------------------------------------------------- agg_bw
 * Replaces the accumulation loop of agg_bw, utils/_agg_bw.py:84-123.  signal_dev: float32
 * [n_seg][row_len], one row per accepted interval (the bigWig values of [start, stop), NaN where
 * uncovered); strand_dev: int8 per row, +1 = '+', -1 = '-' (row is flipped), 0 = skipped.
 * out_dev[p] = sum over rows in order of row[trim_lo + p] ('+') or row[trim_lo + out_len-1-p] ('-'),
 * NaN as 0, accumulated in fp64 in row order (bit-identical to the reference's running sum).
 * trim_lo = median_window_size // 2, out_len = stop - start - median_window_size. */
int ftk_agg_signal_f64(const float *signal_dev, int64_t n_seg, int64_t row_len, int32_t trim_lo,
                       int32_t out_len, const int8_t *strand_dev, double *out_dev, ftk_stream_t stream);

/* ------------------------------------------------------------ adjust_wps
 * Replaces _local_filter/_running_stat (frag/_adjust_wps.py:25-45) and the
 * scipy.signal.savgol_filter call (frag/_adjust_wps.py:135-138) inside
 * _single_adjust_wps (frag/_adjust_wps.py:63-163).
 *
 * x_dev: raw WPS samples (float32, as a bigWig stores them) of n_seg contiguous
 * segments; segment s = x[seg_off[s] .. seg_off[s+1]) with n_s samples and
 * n_s - w outputs written to out[seg_out_off[s] ..] (float64):
 *   adj[j] = (x[j+w/2]-shift) - stat((x-shift)[j:j+w]),  stat = median | mean
 * Work is cut into runs of run_len outputs: seg_run_off[s] = first run of
 * segment s (prefix sum of ceil((n_s-w)/run_len)), n_runs in total.
 * ftk_adjust_wps_f64 writes adj (the median/mean-subtracted series) and is the fast
 * path (integer-valued samples whose local range fits a 256-wide window); runs it
 * cannot handle are flagged in fallback_dev[run] and must be redone with
 * ftk_adjust_wps_generic_f64 (any float input; scratch_dev: float[n_list * w]).
 * ftk_savgol_f64 then applies savgol_filter(adj, sg_w, deg, mode='interp') per
 * segment (out != adj) from the sg_w interior coefficients and the two
 * (sg_w/2 x sg_w) edge-fit matrices.  w even, 2 <= w <= 32767; sg_w odd <= 127.
 * seg_shift_dev: per-segment constant to subtract (NULL = 0), e.g. from
 * ftk_adjust_edge_shift_f64 = mean(mean(x[:edge]), mean(x[-edge:]))
 * (subtract_edges, frag/_adjust_wps.py:119-123), with Python's slice semantics for any edge: 0 or a
 * negative edge that empties a slice gives NaN. */
int ftk_adjust_edge_shift_f64(const float *x_dev, const int64_t *seg_off_dev, int32_t n_seg,
                              int32_t edge_size, double *shift_dev, ftk_stream_t stream);

int ftk_adjust_wps_f64(const float *x_dev, const int64_t *seg_off_dev, const int64_t *seg_out_off_dev,
                       const int64_t *seg_run_off_dev, const double *seg_shift_dev, int32_t n_seg,
                       int64_t n_runs, int32_t w, int32_t use_mean, int32_t run_len,
                       double *adj_out_dev, uint8_t *fallback_dev, ftk_stream_t stream);

int ftk_adjust_wps_generic_f64(const float *x_dev, const int64_t *seg_off_dev, const int64_t *seg_out_off_dev,
                               const int64_t *seg_run_off_dev, const double *seg_shift_dev, int32_t n_seg,
                               const int64_t *run_list_dev, int64_t n_list, int32_t w,
                               int32_t use_mean, int32_t run_len, double *adj_out_dev,
                               float *scratch_dev, ftk_stream_t stream);

int ftk_savgol_f64(const double *adj_dev, const int64_t *seg_out_off_dev, int32_t n_seg, int64_t n_total,
                   int32_t sg_w, const double *coef_dev, const double *edge_first_dev,
                   const double *edge_last_dev, double *out_dev, ftk_stream_t stream);

/* Fused running-median adjust + Savitzky-Golay for integer-valued input (raw WPS), one CTA per tile:
 * rank bitmaps in shared memory instead of per-thread sliding histograms, the adjusted series never
 * leaves the SM (frag/_adjust_wps.py:25-45 _local_filter(median) + :131-138 savgol_filter in ONE kernel).
 * x_dev: float32 (x_kind 0, bigWig values) or int32 (x_kind 1, device-resident WPS) samples of all
 * segments back to back.  Tiles are planned by the caller: tile t covers outputs
 * [tile_t0[t], tile_t0[t] + tile_n[t]) of segment tile_seg[t]; a_cap / s_cap = the largest number of
 * adjusted values / samples any tile needs (outputs +- sg_w/2 clipped to the segment, + w samples).
 * sg_w = 0: no smoothing (out = adjusted series).  seg_shift_dev NULL = no subtract_edges.
 * tile_flag_dev[t] (uint8, zeroed here) is set for tiles that could not be handled (non-integer or
 * |x| > 32000 samples, value spread beyond the searched bands): the caller redoes those through
 * ftk_adjust_wps_f64 / ftk_adjust_wps_generic_f64 + ftk_savgol_f64.
 * sg_num_a, sg_num_b, sg_den (sg_den > 0, no subtract_edges): the interior Savitzky-Golay coefficients as the
 * exact rationals c_i = (sg_num_a + sg_num_b * i^2) / sg_den, i = -sg_w/2 .. sg_w/2 (polynomial degree <= 3:
 * degree 0/1 = (1, 0, sg_w); degree 2/3 = (S4, -S2, sg_w * S4 - S2^2) with S2 = sum i^2, S4 = sum i^4).  The
 * smoothing then runs as exact integer sliding moments of 2 * adjusted (O(1) per output) and is rounded once;
 * it differs from the fp64 stencil of coef_dev (used when sg_den == 0, and by the fallback path) only by that
 * stencil's own rounding (~1e-16 x sum |c_i x_i|).  Without smoothing the results are identical to the fallback path. */
int ftk_adjust_rank_f64(const void *x_dev, int32_t x_kind, const int64_t *seg_off_dev,
                        const int64_t *seg_out_off_dev, const double *seg_shift_dev, int32_t n_seg,
                        const int32_t *tile_seg_dev, const int32_t *tile_t0_dev, const int32_t *tile_n_dev,
                        int64_t n_tiles, int32_t median_window, int32_t sg_w, const double *coef_dev,
                        const double *edge_first_dev, const double *edge_last_dev,
                        int64_t sg_num_a, int64_t sg_num_b, int64_t sg_den, int32_t a_cap, int32_t s_cap,
                        double *out_dev, uint8_t *tile_flag_dev, ftk_stream_t stream);

/* ------------------------------------------------------- cleavage profile
 * Replaces _coverage_and_ends + the proportion step of cleavage_profile
 * (frag/_cleavage_profile.py:33-90, 190-217).  Tiles as for WPS (ftk_wps_plan_tiles with
 * max_len = 0 gives tile_mid_lo/hi = the interval [start, stop), passed here as
 * tile_ivl_lo/hi): a fragment takes part in a tile iff mapq >= min_mapq, min_len <= L <= max_len
 * (FTK_NONE = unbounded) and stop > ivl_lo and start < ivl_hi (frag_array(...,"any")).
 * out[tile_out_off + (p - p0)] = depth(p) ? ends(p) / depth(p) * 100 : 0 (float64), ends = start
 * of '+' fragments / stop of '-' fragments (frag_strand NULL = all '+').
 * scratch_dev: int64[2 * n_tiles]. */
int ftk_cleavage_tiles_f64(const int32_t *frag_start_dev, const int32_t *frag_stop_dev,
                           const uint8_t *frag_mapq_dev, const uint8_t *frag_strand_dev,
                           int64_t n_frag, int32_t max_frag_len,
                           const int32_t *tile_p0_dev, const int32_t *tile_len_dev,
                           const int32_t *tile_ivl_lo_dev, const int32_t *tile_ivl_hi_dev,
                           const int64_t *tile_out_off_dev, int64_t n_tiles,
                           int32_t min_len, int32_t max_len, int32_t min_mapq,
                           int64_t *scratch_dev, double *out_dev, ftk_stream_t stream);

/* ------------------------------------------------------ per-base fragment depth
 * The depth track of coverage_profile: the coverage array of _coverage_and_ends
 * (frag/_cleavage_profile.py:33-90) as its own output, or the fragment-midpoint count.  Same tile
 * table and fragment filter as ftk_cleavage_tiles_f64 (mapq >= min_mapq, min_len <= L <= max_len,
 * FTK_NONE = unbounded); no strand column is read.
 * midpoint == 0: out[tile_out_off + (p - p0)] = #{passing fragments with start <= p < stop}
 * midpoint != 0: out[tile_out_off + (p - p0)] = #{passing fragments with (start + stop) / 2 == p}
 * (int32).  A fragment of length >= 1 that covers, or is centred on, a position overlaps that
 * position's interval, so tile_ivl_lo/hi are validated but never read.  The one exception is a
 * zero-length fragment (start == stop, passing only with min_len <= 0): midpoint mode counts it at
 * start by the definition above, also at an interval's first position, where the "any" overlap
 * test (stop > ivl_lo) of ftk_cleavage_tiles_f64 would drop it.  Span mode never counts it.
 * scratch_dev: int64[2 * n_tiles]. */
int ftk_depth_tiles_i32(const int32_t *frag_start_dev, const int32_t *frag_stop_dev,
                        const uint8_t *frag_mapq_dev, int64_t n_frag, int32_t max_frag_len,
                        const int32_t *tile_p0_dev, const int32_t *tile_len_dev,
                        const int32_t *tile_ivl_lo_dev, const int32_t *tile_ivl_hi_dev,
                        const int64_t *tile_out_off_dev, int64_t n_tiles,
                        int32_t min_len, int32_t max_len, int32_t min_mapq, int32_t midpoint,
                        int64_t *scratch_dev, int32_t *out_dev, ftk_stream_t stream);

/* ---------------------------------------------------------------- V-plot
 * Site-centred fragment V-plot: a fragment-length x midpoint-offset count matrix summed over sites.
 * Site k has the window [win_lo[k], win_hi[k]) = [c - flank, c + flank + 1) around its centre c (the
 * kernel reads c = win_lo[k] + flank; win_hi only bounds the candidate search) and is flipped when
 * site_flip[k] != 0 ('-' strand).  A fragment passes when mapq >= min_mapq and min_len <= L <= max_len,
 * L = stop - start; its midpoint is m = (start + stop) / 2 and its offset d = m - c (flipped: c - m).
 * For every site and every passing fragment with |d| <= flank:
 *   out[(L - min_len) * (2 * flank + 1) + d + flank] += 1
 * so a fragment counts once per site whose window holds its midpoint (duplicate sites count again).
 * out_dev: uint64[(max_len - min_len + 1) * (2 * flank + 1)], ACCUMULATED (the caller zeroes it).
 * Each site's candidate range is split into `splits` slices, one warp each.  scratch_dev: int64[2*n_sites].
 * max_frag_len = max(stop - start) over the contig.  0 <= min_len <= max_len, 0 <= flank <= FTK_VPLOT_MAX_FLANK,
 * at most FTK_VPLOT_MAX_CELLS cells; n_sites == 0 or n_frag == 0 returns 0 without a launch. */
#define FTK_VPLOT_MAX_FLANK (1 << 20)
#define FTK_VPLOT_MAX_CELLS (1 << 27)
int ftk_vplot_u64(const int32_t *frag_start_dev, const int32_t *frag_stop_dev, const uint8_t *frag_mapq_dev,
                  int64_t n_frag, int32_t max_frag_len, const int32_t *win_lo_dev, const int32_t *win_hi_dev,
                  const uint8_t *site_flip_dev, int64_t n_sites, int32_t flank, int32_t min_len, int32_t max_len,
                  int32_t min_mapq, int32_t splits, int64_t *scratch_dev, uint64_t *out_dev, ftk_stream_t stream);

/* ---------------------------------------------------------------- OCF end profiles
 * Orientation-aware fragment end profiles (Sun et al. 2019): upstream- and downstream-end offset counts
 * around sites, summed over the sites of each of n_sets site sets.  Site k has the window of ftk_vplot_u64
 * ([win_lo[k], win_hi[k]) = [c - flank, c + flank + 1), c = win_lo[k] + flank), is flipped when
 * site_flip[k] != 0 and belongs to set site_set[k] (0 <= site_set[k] < n_sets).  A fragment [s, e) passes when
 * mapq >= min_mapq, L = e - s >= 1 and min_len <= L <= max_len (FTK_NONE = unbounded).  Its upstream end
 * offset is x_U = s - c and its downstream one x_D = (e - 1) - c (flipped: x_U = c - (e - 1), x_D = c - s).
 * For every site of set k and every passing fragment, each end independently:
 *   out[(2 k + 0) * (2 * flank + 1) + x_U + flank] += 1  when |x_U| <= flank
 *   out[(2 k + 1) * (2 * flank + 1) + x_D + flank] += 1  when |x_D| <= flank
 * out_dev: uint64[n_sets][2][2 * flank + 1], ACCUMULATED (the caller zeroes it).
 * Work split: each site's candidate range is split into `splits` slices, unit u = site * splits + slice is one
 * warp, and CTA b (of n_cta) takes the units [cta_bounds_dev[b], cta_bounds_dev[b + 1]) (int32[n_cta + 1]),
 * which must all belong to one set: sort the sites by set.  A CTA counts in shared memory and adds its counts
 * to out_dev before the candidate fragments it has taken since the last such flush pass flush_every
 * (1 <= flush_every <= 2^32 - 1; 2^32 - 1 flushes only when a 32-bit counter could overflow).
 * scratch_dev: int64[2 * n_sites].  max_frag_len = max(stop - start) over the contig.  0 <= flank <=
 * FTK_OCF_MAX_FLANK, at most FTK_OCF_MAX_CELLS cells, n_sites * splits <= INT32_MAX; n_sites == 0 or
 * n_frag == 0 returns 0 without a launch. */
#define FTK_OCF_MAX_FLANK 8192
#define FTK_OCF_MAX_CELLS (1 << 27)
int ftk_ocf_u64(const int32_t *frag_start_dev, const int32_t *frag_stop_dev, const uint8_t *frag_mapq_dev,
                int64_t n_frag, int32_t max_frag_len, const int32_t *win_lo_dev, const int32_t *win_hi_dev,
                const uint8_t *site_flip_dev, const int32_t *site_set_dev, int64_t n_sites, int32_t n_sets,
                int32_t flank, int32_t min_len, int32_t max_len, int32_t min_mapq, int32_t splits,
                const int32_t *cta_bounds_dev, int32_t n_cta, int64_t flush_every, int64_t *scratch_dev,
                uint64_t *out_dev, ftk_stream_t stream);

/* ---------------------------------------------------------------- GC bias
 * Fragment-level GC model (Benjamini & Speed 2012): fragment counts by (length, G+C bases), observed over the
 * sample's fragments and expected over every placement a fragment of that length could take.
 * A placement [p, p + L) of one contig counts when p >= 0, p + L <= contig_len, its midpoint p + L / 2 lies in
 * a region [reg_start[k], reg_stop[k]) and none of its bases is N; its G/C count g is the number of C or G
 * bases in it.  Each counting placement adds
 *   out[(L - min_len) * (max_len + 1) + g] += 1
 *   ftk_gc_observed_u64: one placement per fragment with mapq >= min_mapq and min_len <= L <= max_len,
 *                        L = stop - start (the midpoint is (start + stop) / 2);
 *   ftk_gc_expected_u64: one placement per (p, L) with min_len <= L <= max_len.
 * seq_words_dev / nmask_words_dev: the contig packed as synth.pack_twobit does (2 bits per base, A0 C1 G2 T3,
 * N bit mask, two spare words of padding; seq_words_dev 8-byte aligned).  1 <= min_len <= max_len <=
 * FTK_GC_MAX_LENGTH, contig_len <= INT32_MAX.  out_dev: uint64[(max_len - min_len + 1) * (max_len + 1)],
 * ACCUMULATED (the caller zeroes it).
 * Observed: regions sorted, disjoint and clipped to [0, contig_len]; each region's candidate range is split
 * into `splits` slices, one warp each; scratch_dev: int64[2 * n_reg]; max_frag_len = max(stop - start) over
 * the contig.  n_reg == 0 or n_frag == 0 returns 0 without a launch.
 * Expected: a table of midpoint tiles [tile_lo[t], tile_hi[t]), each inside one region, disjoint, at most
 * tile_cap <= FTK_GC_MAX_TILE midpoints long; one CTA per (tile, 32 consecutive lengths).  n_tiles == 0
 * returns 0 without a launch. */
#define FTK_GC_MAX_LENGTH 1024
#define FTK_GC_MAX_TILE 16384
int ftk_gc_observed_u64(const int32_t *frag_start_dev, const int32_t *frag_stop_dev, const uint8_t *frag_mapq_dev,
                        int64_t n_frag, int32_t max_frag_len, const uint32_t *seq_words_dev,
                        const uint32_t *nmask_words_dev, int64_t contig_len, const int32_t *reg_start_dev,
                        const int32_t *reg_stop_dev, int64_t n_reg, int32_t min_len, int32_t max_len,
                        int32_t min_mapq, int32_t splits, int64_t *scratch_dev, uint64_t *out_dev,
                        ftk_stream_t stream);
int ftk_gc_expected_u64(const uint32_t *seq_words_dev, const uint32_t *nmask_words_dev, int64_t contig_len,
                        const int32_t *tile_lo_dev, const int32_t *tile_hi_dev, int64_t n_tiles, int32_t tile_cap,
                        int32_t min_len, int32_t max_len, uint64_t *out_dev, ftk_stream_t stream);

/* ---------------------------------------------------------------- GC-corrected counts
 * The GC model applied: weights_dev is a float64 table of the GC-bias matrices' shape, read as
 * weights[(L - min_len) * (max_len + 1) + g] (typically 1 / ratio, 0 where the ratio is undefined).  A fragment
 * is selected when mapq >= min_mapq, min_len <= L <= max_len (L = stop - start) and its midpoint
 * m = (start + stop) / 2 passes the unit's position test.  Every selected fragment adds 1 to a count; it also
 * adds weights[L - min_len, g] to a corrected sum when start >= 0, stop <= contig_len and none of its bases is N
 * (the placement rule of ftk_gc_observed_u64; g = its C/G bases).  The reference, lengths and fragments are as
 * for ftk_gc_observed_u64.  Outputs are ACCUMULATED (the caller zeroes them); each unit's candidate range is split
 * into `splits` slices, one warp each; n_units == 0 or n_frag == 0 returns 0 without a launch.
 *   ftk_gc_weighted_intervals_f64: interval k is [ivl_start[k], ivl_stop[k]) (FTK_NONE = unbounded; overlapping and
 *     unsorted intervals are fine), test ivl_start <= m < ivl_stop; out_count_dev uint64[n_ivl],
 *     out_corrected_dev fp64[n_ivl].  scratch_dev: int64[2 * n_ivl + 2 * n_ivl * splits] (candidate ranges, then
 *     one partial count and sum per (interval, slice)).  The partials are reduced in a fixed order, so the result
 *     is bit-identical run to run for the same `splits`.
 *   ftk_gc_weighted_sites_f64: the windows of ftk_vplot_u64 ([c - flank, c + flank + 1), flipped when
 *     site_flip[k] != 0), test |d| <= flank with d = m - c (flipped: c - m); out_count_dev uint64[2 * flank + 1]
 *     and out_corrected_dev fp64[2 * flank + 1] at d + flank, summed over the sites (fp64 atomics: the order of
 *     the corrected sums varies between runs).  scratch_dev: int64[2 * n_sites]; flank <= FTK_VPLOT_MAX_FLANK. */
int ftk_gc_weighted_intervals_f64(const int32_t *frag_start_dev, const int32_t *frag_stop_dev,
                                  const uint8_t *frag_mapq_dev, int64_t n_frag, int32_t max_frag_len,
                                  const uint32_t *seq_words_dev, const uint32_t *nmask_words_dev, int64_t contig_len,
                                  const int32_t *ivl_start_dev, const int32_t *ivl_stop_dev, int64_t n_ivl,
                                  int32_t min_len, int32_t max_len, int32_t min_mapq, int32_t splits,
                                  int64_t *scratch_dev, const double *weights_dev, uint64_t *out_count_dev,
                                  double *out_corrected_dev, ftk_stream_t stream);
int ftk_gc_weighted_sites_f64(const int32_t *frag_start_dev, const int32_t *frag_stop_dev,
                              const uint8_t *frag_mapq_dev, int64_t n_frag, int32_t max_frag_len,
                              const uint32_t *seq_words_dev, const uint32_t *nmask_words_dev, int64_t contig_len,
                              const int32_t *win_lo_dev, const int32_t *win_hi_dev, const uint8_t *site_flip_dev,
                              int64_t n_sites, int32_t flank, int32_t min_len, int32_t max_len, int32_t min_mapq,
                              int32_t splits, int64_t *scratch_dev, const double *weights_dev,
                              uint64_t *out_count_dev, double *out_corrected_dev, ftk_stream_t stream);

/* ---------------------------------------------------------------- GC-corrected depth tracks
 * The per-base depth of ftk_depth_tiles_i32 (same tile table, scratch and midpoint switch) with the GC model
 * applied.  weights_dev: int64 of the GC-bias matrices' shape, the weights quantised to units of 2^-32
 * (Q = rint(W * 2^32)), read as weights[(L - min_len) * (max_len + 1) + g]; max_weight = max(Q), 0 <= max_weight <
 * FTK_GC_DEPTH_MAX_WEIGHT.  A fragment passes when mapq >= min_mapq and min_len <= L <= max_len (1 <= min_len <=
 * max_len <= FTK_GC_MAX_LENGTH, no FTK_NONE); its weight is Q[L - min_len, g] when start >= 0, stop <= contig_len and
 * no base of it is N (g = its C/G bases, the placement rule of ftk_gc_observed_u64), else 0.
 * midpoint == 0: S(p) = sum of the weights of passing fragments with start <= p < stop
 * midpoint != 0: S(p) = sum of the weights of passing fragments with (start + stop) / 2 == p
 * out[tile_out_off + (p - p0)] = (double)S(p) * 2^-32 (fp64; S is summed in int64, so the result is exact below 2^53
 * units and bit-identical between runs and batchings).  Every partial sum of a tile is bounded by its candidate
 * fragments times max_weight; a tile where that bound exceeds INT64_MAX ORs 1 into *overflow_dev (int32, zeroed by
 * the caller) and writes none of its positions.  seq_words_dev / nmask_words_dev: the packed contig of
 * ftk_gc_observed_u64; out_dev 8-byte aligned.  n_tiles == 0 returns 0 without a launch. */
#define FTK_GC_DEPTH_MAX_WEIGHT (INT64_C(1) << 62)
int ftk_gc_depth_tiles_f64(const int32_t *frag_start_dev, const int32_t *frag_stop_dev,
                           const uint8_t *frag_mapq_dev, int64_t n_frag, int32_t max_frag_len,
                           const uint32_t *seq_words_dev, const uint32_t *nmask_words_dev, int64_t contig_len,
                           const int32_t *tile_p0_dev, const int32_t *tile_len_dev,
                           const int32_t *tile_ivl_lo_dev, const int32_t *tile_ivl_hi_dev,
                           const int64_t *tile_out_off_dev, int64_t n_tiles,
                           int32_t min_len, int32_t max_len, int32_t min_mapq, int32_t midpoint,
                           const int64_t *weights_dev, int64_t max_weight, int64_t *scratch_dev,
                           int32_t *overflow_dev, double *out_dev, ftk_stream_t stream);

/* ---------------------------------------------------------------- periodicity spectra
 * Segment s is x_dev[offsets_dev[s] .. offsets_dev[s + 1]) (int64 offsets, segments back to back; N values,
 * mean mu).  For every integer period P in [min_period, max_period]:
 *   X(P) = sum_{n<N} (x[n] - mu) * exp(-2 pi i (n mod P) / P),  out_dev[s * n_periods + P - min_period] = |X(P)|^2 / N
 * (n_periods = max_period - min_period + 1; fp64).  The per-residue folds sum_{n = r mod P} x[n] are exact int64
 * sums for int32 input and fp64 sums for fp64 input.  An empty segment gives a row of NaN.  No atomics: the output
 * is bit-identical from run to run, and a segment's row does not depend on the other segments of the call.
 * 2 <= min_period <= max_period <= FTK_SPECTRUM_MAX_PERIOD; n_seg == 0 returns 0 without a launch (replaces the
 * bigWig export + host FFT of Snyder et al. 2016's gene-body WPS periodograms). */
#define FTK_SPECTRUM_MAX_PERIOD 1024
int ftk_spectrum_i32_f64(const int32_t *x_dev, const int64_t *offsets_dev, int64_t n_seg, int32_t min_period,
                         int32_t max_period, double *out_dev, ftk_stream_t stream);
int ftk_spectrum_f64_f64(const double *x_dev, const int64_t *offsets_dev, int64_t n_seg, int32_t min_period,
                         int32_t max_period, double *out_dev, ftk_stream_t stream);

/* ------------------------------------------------- fragment file decode (host)
 * Multi-threaded decode of a BGZF / gzip fragment file into per-contig columns; replaces the
 * per-interval pysam.TabixFile.fetch text stream of io/alignment.py:270-302 (5-column FinaleDB
 * layout or BED6, malformed rows skipped, '+' in the strand field = forward) with one pass.
 * Host pointers only; no CUDA involved.  n_threads < 1 = all hardware threads.
 * ftk_fragfile_open returns NULL and sets *err (FTK_E_IO / FTK_E_INVALID) on failure.
 * ftk_fragfile_copy fills caller buffers (pinned or pageable) of ftk_fragfile_contig_count
 * elements, rows in file order. */
void *ftk_fragfile_open(const char *path, int32_t n_threads, int32_t *err);
/* Same, for the part of a tabix-indexed file between two virtual offsets (coffset = file offset of a
 * BGZF block, uoffset = byte inside its inflated text): what pysam.TabixFile.fetch(contig) reads
 * through the .tbi index (io/alignment.py:270-279), here one contig's whole block range in one
 * parallel pass.  bed6 = the column layout detected on the file's first data line. */
void *ftk_fragfile_open_slice(const char *path, int64_t coffset_beg, int32_t uoffset_beg,
                              int64_t coffset_end, int32_t uoffset_end, int32_t bed6,
                              int32_t n_threads, int32_t *err);
/* BAM -> fragment columns: AlignmentWrapper._fetch_sam + _read_is_low_quality (io/alignment.py:60-71,
 * 242-268; the mapq test stays a kernel predicate) on a streamed, multi-threaded BGZF inflate - no
 * htslib.  ftk_bamfile_fragments returns a handle for the ftk_fragfile_* accessors (owned by the
 * BAM handle: do not close it separately); ftk_bamfile_n_refs / _ref_name / _ref_length expose the
 * header's @SQ table (AlignmentWrapper._chroms, :126-127). */
void *ftk_bamfile_open(const char *path, int32_t n_threads, int32_t *err);
void *ftk_bamfile_fragments(void *bam_handle);
int32_t ftk_bamfile_n_refs(void *bam_handle);
const char *ftk_bamfile_ref_name(void *bam_handle, int32_t i);
int64_t ftk_bamfile_ref_length(void *bam_handle, int32_t i);
void ftk_bamfile_close(void *bam_handle);
int32_t ftk_fragfile_is_bed6(void *handle);
int64_t ftk_fragfile_skipped(void *handle);
int32_t ftk_fragfile_n_contigs(void *handle);
const char *ftk_fragfile_contig_name(void *handle, int32_t i);
int64_t ftk_fragfile_contig_count(void *handle, int32_t i);
int ftk_fragfile_copy(void *handle, int32_t i, int32_t *start_host, int32_t *stop_host,
                      uint8_t *mapq_host, uint8_t *strand_host);
/* BAM-derived handles only: the reference span [pos, bam_endpos) of READ 1 of every fragment, rows as in
 * ftk_fragfile_copy.  An indexed BAM fetch selects READS overlapping the region before the fragment is
 * built (io/alignment.py:242-247: `for read in self._handle.fetch(contig, start, stop)`), so the host side
 * needs these two columns to make the same selection (FragmentTable.fetched).  Returns 0 = copied,
 * 1 = the handle carries no read-1 columns (fragment files), < 0 = error. */
int ftk_fragfile_copy_read1(void *handle, int32_t i, int32_t *r1_start_host, int32_t *r1_end_host);
void ftk_fragfile_close(void *handle);

/* ------------------------------------------------- bigWig section codec (host)
 * bigWig data sections are independent zlib streams (one per <= 65535 items), which the
 * reference compresses / inflates one at a time inside pyBigWig's addEntries / intervals
 * (frag/_multi_wps.py:300-325, frag/_adjust_wps.py:80-105,275-291).  These two calls run a
 * whole batch of sections on n_threads host threads (n_threads < 1 = all hardware threads).
 * Host pointers only; no CUDA involved.
 *   compress:   member i = in[in_off[i] .. in_off[i+1]) -> written at out + out_off[i]; the slot
 *               out_off[i+1] - out_off[i] must be >= zlib's compressBound(len) (len + len/1000 +
 *               64 is enough); out_size[i] receives the compressed size.
 *   uncompress: member i = in[in_off[i] .. in_off[i] + in_size[i]) -> out + out_off[i], slot
 *               out_off[i+1] - out_off[i]; out_size[i] receives the inflated size.
 * Return 0, FTK_E_INVALID (bad arguments / slot too small) or FTK_E_IO (corrupt stream). */
int ftk_zlib_compress_batch(const uint8_t *in, const int64_t *in_off, int64_t n, int32_t level,
                            int32_t n_threads, uint8_t *out, const int64_t *out_off,
                            int64_t *out_size);
int ftk_zlib_uncompress_batch(const uint8_t *in, const int64_t *in_off, const int64_t *in_size,
                              int64_t n, int32_t n_threads, uint8_t *out, const int64_t *out_off,
                              int64_t *out_size);

/* ------------------------------------------------- text outputs (host)
 * bedGraph lines `contig\tpos\tpos+1\tscore\n` for n consecutive positions from `start`, the text
 * multi_wps writes one f-string at a time (frag/_multi_wps.py:328-341).  With out_host == NULL the
 * call returns the byte count; otherwise it fills out_host (out_cap >= that count) on n_threads
 * threads and returns the bytes written, or FTK_E_INVALID. */
int64_t ftk_format_bedgraph_i64(const char *contig, int64_t start, const int64_t *scores_host, int64_t n,
                                int32_t n_threads, char *out_host, int64_t out_cap);
/* gzip (RFC 1952) members of independent chunks, laid out like ftk_zlib_compress_batch (slot >= the
 * zlib deflateBound of a gzip stream: len + len/1000 + 64 is enough).  Concatenated members form one
 * valid .gz file - the multi-threaded stand-in for the reference's gzip.open(path, "wt") writers
 * (frag/_multi_wps.py:328-341, frag/_cleavage_profile.py:392-405). */
int ftk_gzip_compress_batch(const uint8_t *in, const int64_t *in_off, int64_t n, int32_t level,
                            int32_t n_threads, uint8_t *out, const int64_t *out_off,
                            int64_t *out_size);

#ifdef __cplusplus
}
#endif
#endif /* FTK_B200_H */
