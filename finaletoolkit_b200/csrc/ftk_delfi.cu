// DELFI window counts + GC content on sm_100a.
//
// Replaces the per-fragment loop and the str.count GC pass of _delfi_single_window
// (frag/_delfi.py:404-511), which the reference runs once per 100 kb bin in a process pool
// (frag/_delfi.py:283-294).  One launch handles every bin of a contig:
//   stream   : tabix overlap with the bin (fe > ws, fs < we), mapq >= q          (:437)
//   length   : 100 <= L <= 220                                                   (:442-443)
//   midpoint : ws <= (fs+fe)//2 < we                                             (:445-447)
//   blacklist: dropped when start AND stop both lie in [r0, r1) of one blacklist region that is
//              itself contained in the bin (frag/_delfi.py:110-127, :449-457)
//   gaps     : dropped when the fragment overlaps the centromere, or overlaps EVERY telomere
//              (ContigGaps.in_tcmere, genome/gaps.py:226-248 - the `all` is the reference's)
//   short    : L < 151, long: L >= 151, num_frags = short + long                  (:462-467)
// and a second kernel counts G + C bases of each bin in the 2-bit packed contig (:470-484).
// The arm / NOARM decision and the NaN conventions stay on the host.
// Roofline: HBM, 9 B per candidate fragment (start, stop, mapq) + 0.375 B per bin base.
#include "ftk_common.cuh"

namespace ftk {

constexpr int kDelfiThreads = 256;

struct DelfiGaps { int use, c0, c1, has_telo, t0_max, t1_min; };

__global__ void __launch_bounds__(kDelfiThreads)
delfi_count_kernel(const int32_t *__restrict__ frag_start, const int32_t *__restrict__ frag_stop,
                   const uint8_t *__restrict__ frag_mapq,
                   const int32_t *__restrict__ win_start, const int32_t *__restrict__ win_stop,
                   const int64_t *__restrict__ ranges,
                   const int32_t *__restrict__ bl_off, const int32_t *__restrict__ bl_start,
                   const int32_t *__restrict__ bl_stop, DelfiGaps gaps, int min_mapq, int splits,
                   unsigned long long *__restrict__ counts /* [n_win][4] */) {
    const int tid = threadIdx.x;
    const int64_t win = blockIdx.x / splits;
    const int split = blockIdx.x % splits;
    const int S = win_start[win], E = win_stop[win];
    const int b_lo = bl_off ? bl_off[win] : 0, b_hi = bl_off ? bl_off[win + 1] : 0;
    int64_t lo, hi;
    slice_of(ranges, win, split, splits, lo, hi);

    int n_short = 0, n_long = 0;
    // One fragment, branch-free: every test of frag/_delfi.py:437-470 is a predicate (the tabix overlap
    // `stop > S and start < E` is implied by 100 <= length and the midpoint lying in [S, E)).  Only the
    // blacklist walk (a bin's own CSR list, nearly always empty) branches.
    const unsigned span = E > S ? (unsigned)(E - S) : 0u;
    auto visit = [&](int fs, int fe, int q, int, int) {
        const int len = fe - fs;
        const int mid = (int)(((int64_t)fs + fe) >> 1);   // floor, like Python's //
        bool pass = (q >= min_mapq) & ((unsigned)(len - 100) <= 120u) & ((unsigned)(mid - S) < span);
        if (gaps.use) {
            const bool in_c = (fe > gaps.c0) & (fs < gaps.c1);
            const bool in_t = gaps.has_telo & (fe > gaps.t0_max) & (fs < gaps.t1_min);
            pass = pass & !(in_c | in_t);
        }
        if (b_hi > b_lo && pass) {
            for (int b = b_lo; b < b_hi; ++b) {
                const int r0 = __ldg(bl_start + b), r1 = __ldg(bl_stop + b);
                if (fs >= r0 && fs < r1 && fe >= r0 && fe < r1) { pass = false; break; }
            }
        }
        const int is_long = len >= 151;
        n_long += pass & is_long;
        n_short += pass & !is_long;
    };
    stream_fragments<kDelfiThreads, 2>(FragCols{frag_start, frag_stop, frag_mapq, nullptr}, lo, hi, tid, visit);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        n_short += __shfl_down_sync(0xffffffffu, n_short, o);
        n_long += __shfl_down_sync(0xffffffffu, n_long, o);
    }
    if ((tid & 31) == 0) {
        if (n_short) atomicAdd(&counts[win * 4 + 0], (unsigned long long)n_short);
        if (n_long) atomicAdd(&counts[win * 4 + 1], (unsigned long long)n_long);
        if (n_short + n_long) atomicAdd(&counts[win * 4 + 2], (unsigned long long)(n_short + n_long));
    }
}

// bit i of a 16-bit mask -> bit 2i
__device__ __forceinline__ uint32_t spread16(uint32_t x) {
    x &= 0xffffu;
    x = (x | (x << 8)) & 0x00ff00ffu;
    x = (x | (x << 4)) & 0x0f0f0f0fu;
    x = (x | (x << 2)) & 0x33333333u;
    x = (x | (x << 1)) & 0x55555555u;
    return x;
}

// kGcWarps warps per bin (a 100-kb bin is 37.5 KB of packed contig: one warp per bin left the chip at
// ~1 TB/s), each striding over the bin's words and adding its partial with one atomic: G/C bases (codes
// 1, 2 <=> bit0 ^ bit1) that are not N, in [ws, we) clipped to the contig.  Bins that are not valid
// reference intervals count 0 (frag/_delfi.py:472-482).  counts[][3] accumulates (caller zeroes).
constexpr int kGcWarps = 8;
__global__ void __launch_bounds__(kDelfiThreads)
delfi_gc_kernel(const uint32_t *__restrict__ seq, const uint32_t *__restrict__ nmask, int64_t contig_len,
                const int32_t *__restrict__ win_start, const int32_t *__restrict__ win_stop, int64_t n_win,
                unsigned long long *__restrict__ counts) {
    const int64_t gwarp = ((int64_t)blockIdx.x * kDelfiThreads + threadIdx.x) >> 5;
    const int64_t win = gwarp / kGcWarps;
    const int part = (int)(gwarp % kGcWarps);
    const int lane = threadIdx.x & 31;
    if (win >= n_win) return;
    const int64_t S = win_start[win], E = win_stop[win];
    // valid_interval (utils/validation.py:146-166): 0 <= start < len, 0 <= stop <= len
    const bool valid = S >= 0 && S < contig_len && E >= 0 && E <= contig_len && S <= E;
    int n = 0;
    if (valid) {
        const int64_t w0 = S >> 4, w1 = (E + 15) >> 4;   // 16-base words
        for (int64_t w = w0 + part * 32 + lane; w < w1; w += 32 * kGcWarps) {
            const uint32_t x = __ldg(seq + w);
            uint32_t gc = (x ^ (x >> 1)) & 0x55555555u;
            const uint32_t nm = __ldg(nmask + (w >> 1)) >> ((w & 1) * 16);
            gc &= ~spread16(nm);
            const int64_t base0 = w << 4;
            if (base0 < S) gc &= ~0u << (2 * (int)(S - base0));
            if (base0 + 16 > E) {
                const int keep = (int)(E - base0);               // 0 < keep < 16
                gc &= (keep >= 16) ? ~0u : ((1u << (2 * keep)) - 1u);
            }
            n += __popc(gc);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n += __shfl_down_sync(0xffffffffu, n, o);
    if (lane == 0 && n) atomicAdd(&counts[win * 4 + 3], (unsigned long long)n);
}

}  // namespace ftk

using namespace ftk;

extern "C" int ftk_delfi_windows_u64(const int32_t *frag_start, const int32_t *frag_stop,
                                     const uint8_t *frag_mapq, int64_t n_frag, int32_t max_frag_len,
                                     const uint32_t *seq_words, const uint32_t *nmask_words, int64_t contig_len,
                                     const int32_t *win_start, const int32_t *win_stop, int64_t n_win,
                                     const int32_t *bl_off, const int32_t *bl_start, const int32_t *bl_stop,
                                     const int32_t *gaps5, int32_t min_mapq, int32_t splits,
                                     int64_t *scratch, uint64_t *counts, ftk_stream_t stream_) {
    if (n_win == 0) return FTK_OK;
    if (n_frag < 0 || n_win < 0 || splits < 1) return FTK_E_INVALID;
    if (!win_start || !win_stop || !scratch || !counts) return FTK_E_INVALID;
    if (n_frag > 0 && (!frag_start || !frag_stop)) return FTK_E_INVALID;
    if (bl_off && (!bl_start || !bl_stop)) return FTK_E_INVALID;
    if ((seq_words == nullptr) != (nmask_words == nullptr)) return FTK_E_INVALID;
    if (n_win * (int64_t)splits > INT32_MAX) return FTK_E_RANGE;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    DelfiGaps g = {0, 0, 0, 0, 0, 0};
    if (gaps5) {   // host array: centromere start, stop, n_telomeres, max telomere start, min telomere stop
        g.use = 1; g.c0 = gaps5[0]; g.c1 = gaps5[1]; g.has_telo = gaps5[2] > 0; g.t0_max = gaps5[3]; g.t1_min = gaps5[4];
    }
    const int rc = launch_candidate_ranges(frag_start, n_frag, win_start, win_stop, false, n_win,
                                           max_frag_len < 0 ? 0 : max_frag_len, 0, scratch, stream);
    if (rc != FTK_OK) return rc;
    auto *c = reinterpret_cast<unsigned long long *>(counts);
    delfi_count_kernel<<<(unsigned)(n_win * splits), kDelfiThreads, 0, stream>>>(
        frag_start, frag_stop, frag_mapq, win_start, win_stop, scratch, bl_off, bl_start, bl_stop, g,
        min_mapq, splits, c);
    FTK_CHECK_LAUNCH("delfi_count_kernel");
    if (seq_words) {
        const int64_t threads = n_win * 32 * kGcWarps;
        delfi_gc_kernel<<<(unsigned)((threads + kDelfiThreads - 1) / kDelfiThreads), kDelfiThreads, 0, stream>>>(
            seq_words, nmask_words, contig_len, win_start, win_stop, n_win, c);
        FTK_CHECK_LAUNCH("delfi_gc_kernel");
    }
    return FTK_OK;
}
