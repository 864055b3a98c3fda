// Site-centred fragment V-plot: a (fragment length x midpoint offset) count matrix summed over sites.
//
// For every site (centre c, optionally flipped) and every passing fragment (mapq >= min_mapq,
// min_len <= L <= max_len, L = stop - start) whose midpoint m = (start + stop) / 2 lies within flank of c,
// out[(L - min_len) * (2 * flank + 1) + d + flank] += 1 with d = m - c ('-' sites: c - m).
//
// Each (site, split) pair is one WARP streaming a contiguous slice of the site's candidate range with 128-bit
// loads (the layout of interval_count_warp_kernel: eight independent warps per CTA).  Matching fragments go
// to the matrix with one 64-bit global RED each: the matrix (601 x 2001 x 8 B = 9.6 MB at the defaults) stays
// in L2, a per-CTA shared-memory copy could not hold it, and the cells a warp hits at once are distinct, so
// warp aggregation would buy nothing.
// Roofline: HBM, 9 B per candidate fragment (start, stop, mapq) - or the L2 RED rate when most candidates
// match (DESIGN.md 4.9).
#include "ftk_common.cuh"

namespace ftk {

constexpr int kVplotThreads = 256;
constexpr int kVplotUnroll = 4;

__device__ __forceinline__ void red_global_inc_u64(unsigned long long *p) {
    asm volatile("red.global.add.u64 [%0], %1;" :: "l"(p), "l"(1ull) : "memory");
}

__global__ void __launch_bounds__(kVplotThreads)
vplot_warp_kernel(const int32_t *__restrict__ frag_start, const int32_t *__restrict__ frag_stop,
                  const uint8_t *__restrict__ frag_mapq, const int32_t *__restrict__ win_lo,
                  const uint8_t *__restrict__ site_flip, const int64_t *__restrict__ ranges, int flank,
                  int min_len, int max_len, int min_mapq, int splits, int64_t n_units,
                  unsigned long long *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t unit = (int64_t)blockIdx.x * (kVplotThreads / 32) + (threadIdx.x >> 5);
    if (unit >= n_units) return;
    const int64_t site = unit / splits;
    const int split = (int)(unit % splits);
    const int c = __ldg(win_lo + site) + flank;           // the window is [c - flank, c + flank + 1)
    const bool flip = __ldg(site_flip + site) != 0;
    int64_t lo, hi;
    slice_of(ranges, site, split, splits, lo, hi);

    const unsigned len_span = (unsigned)(max_len - min_len);
    const unsigned width = 2u * (unsigned)flank;              // d + flank in [0, width]
    const int64_t row = 2 * (int64_t)flank + 1;
    auto visit = [&](int fs, int fe, int q, int, int) {
        const int L = fe - fs;                                // the sentinel (L = -1) fails the length test
        const int m = fs + (L >> 1);
        const int64_t d = flip ? (int64_t)c - m : (int64_t)m - c;
        const bool ok = ((unsigned)(L - min_len) <= len_span) & (q >= min_mapq) & ((uint64_t)(d + flank) <= width);
        if (ok) red_global_inc_u64(out + (int64_t)(L - min_len) * row + (d + flank));
    };
    stream_fragments<32, kVplotUnroll>(FragCols{frag_start, frag_stop, frag_mapq, nullptr}, lo, hi, lane, visit);
}

}  // namespace ftk

using namespace ftk;

extern "C" int ftk_vplot_u64(const int32_t *frag_start, const int32_t *frag_stop, const uint8_t *frag_mapq,
                             int64_t n_frag, int32_t max_frag_len, const int32_t *win_lo, const int32_t *win_hi,
                             const uint8_t *site_flip, int64_t n_sites, int32_t flank, int32_t min_len,
                             int32_t max_len, int32_t min_mapq, int32_t splits, int64_t *scratch, uint64_t *out,
                             ftk_stream_t stream_) {
    if (n_sites == 0) return FTK_OK;
    if (n_frag < 0 || n_sites < 0 || flank < 0 || splits < 1 || min_len < 0 || max_len < min_len) return FTK_E_INVALID;
    if (!win_lo || !win_hi || !site_flip || !scratch || !out) return FTK_E_INVALID;
    if (n_frag > 0 && (!frag_start || !frag_stop)) return FTK_E_INVALID;
    if (flank > FTK_VPLOT_MAX_FLANK) return FTK_E_RANGE;
    if (((int64_t)max_len - min_len + 1) * (2 * (int64_t)flank + 1) > FTK_VPLOT_MAX_CELLS) return FTK_E_RANGE;
    if (n_sites > INT32_MAX / 2 || n_sites * (int64_t)splits > INT32_MAX) return FTK_E_RANGE;
    if (n_frag == 0) return FTK_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    // start >= m - L/2 >= c - flank - max/2 and start <= m <= c + flank: a superset of the fragments that can count
    const int reach = (max_frag_len < max_len ? (max_frag_len < 0 ? 0 : max_frag_len) : max_len) >> 1;
    const int rc = launch_candidate_ranges(frag_start, n_frag, win_lo, win_hi, false, n_sites, reach, 0, scratch, stream);
    if (rc != FTK_OK) return rc;
    const int64_t n_units = n_sites * (int64_t)splits;
    const int per_cta = kVplotThreads / 32;
    vplot_warp_kernel<<<(unsigned)((n_units + per_cta - 1) / per_cta), kVplotThreads, 0, stream>>>(
        frag_start, frag_stop, frag_mapq, win_lo, site_flip, scratch, flank, min_len, max_len, min_mapq, splits, n_units,
        reinterpret_cast<unsigned long long *>(out));
    FTK_CHECK_LAUNCH("vplot_warp_kernel");
    return FTK_OK;
}
