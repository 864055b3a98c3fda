// 5' end-motif k-mer histograms on sm_100a.
//
// Replaces the per-fragment loop of region_end_motifs (frag/_end_motifs.py:115-179):
// two py2bit sequence() calls + a dict increment per fragment become two 64-bit
// window reads of a 2-bit packed contig (L2-resident: chr1 = 62 MB + 31 MB N-mask)
// and shared-memory-privatised histogram atomics.
//   forward k-mer : ref[fs, fs+k)              index = sum code_j * 4^(k-1-j)
//   reverse k-mer : revcomp(ref[fe-k, fe))     (utils/utils.py:413-437)
//   k-mers containing N are skipped (frag/_end_motifs.py:133,142)
//   forward window out of bounds -> fragment skipped entirely (:135-136)
//   reverse window out of bounds -> RuntimeError in the reference (:144-151):
//       reported through *error_flag, the host raises.
// Membership is tabix overlap only - no length filter, no midpoint policy
// (frag/_end_motifs.py:115-120, SURVEY quirk 8).
// Index order = itertools.product("ACGT") (utils/utils.py:388-410): A0 C1 G2 T3.
// Breakpoint motifs (region_breakpoint_motifs, frag/_breakpoint_motifs.py:53-196) are the same
// kernel with windows centred on the two breakpoints, h = k/2:
//   fragment skipped when fs-h < 0 or fs+h >= contig_len (:125-133)
//   forward k-mer : ref[fs-h, fs+h)            reverse : revcomp(ref[fe-h, fe+h))
//   reverse window out of bounds -> that end is skipped (OutOfBoundsError is a ValueError, :186)
//   odd k: every window has 2h != k bases -> "length discrepancy" -> nothing is ever counted
// Roofline: HBM, 10 B per candidate fragment (start, stop, mapq, strand) + 2 x 2 B
// of packed reference per end served from L2.
#include <type_traits>

#include "ftk_common.cuh"

namespace ftk {

constexpr int kMotifThreads = 256;
constexpr int kMotifSmemBins = 4096;  // k <= 6 privatised in shared memory


// 2k-bit window starting at base `pos` (base i at bits 2*(i%16) of word i/16): one funnel shift
// over two consecutive words; k <= 12, so 24 bits at a shift <= 30 always fit.
__device__ __forceinline__ uint32_t window2(const uint32_t *__restrict__ seq, int pos, uint32_t mask2k) {
    const int w = pos >> 4;
    return __funnelshift_r(__ldg(seq + w), __ldg(seq + w + 1), (pos & 15) * 2) & mask2k;
}
__device__ __forceinline__ bool has_n(const uint32_t *__restrict__ nmask, int pos, uint32_t maskk) {
    const int w = pos >> 5;
    return (__funnelshift_r(__ldg(nmask + w), __ldg(nmask + w + 1), pos & 31) & maskk) != 0u;
}
// reverse the order of the k 2-bit digits of x (first base becomes the most significant digit)
__device__ __forceinline__ uint32_t digit_reverse(uint32_t x, int k) {
    x = __brev(x);
    x = ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
    return x >> (32 - 2 * k);
}

// Fragments are fetched four per lane with 128-bit loads (two vectors = eight fragments in flight per
// thread); the k-mer windows are read from the L2-resident packed contig.  (A variant that staged the
// contig span of every 4096-fragment sub-chunk in shared memory was measured in round 2 and lost:
// 0.59 ms against 0.39 ms - the staging serialises bounds -> span -> fragments behind two barriers
// per sub-chunk and its 75 registers cut the residency to three CTAs per SM.)
//
// What keeps the per-fragment instruction count down (the kernel is issue-bound, not DRAM-bound):
//   * K and the strand mode are template parameters for the common cases (masks, shifts and the
//     mode tests fold away instead of being rematerialised under the 40-register budget);
//   * N runs are rare and long (telomeres, centromere, assembly gaps), so every CTA first ORs the
//     N-mask words of the span its fragment slice can touch - two loads per thread - and, when that is
//     zero, runs the loop instantiated without the per-end N test (two loads + four operations less
//     per end: 296 -> 251 us with the batch below, 216 us without it);
//   * the next vector of a thread is loaded while the current one is processed, the lines two
//     iterations ahead are pulled into L2, slices are 16 K fragments (the per-CTA chain ranges ->
//     slice bounds -> N pre-scan -> first fragments is paid once per slice).
// Measured and dropped: handling the four fragments of a vector together, branch-free, with all
// sixteen window words requested before the first k-mer is formed (251 us against 216 us for the
// plain per-fragment loop: the predicated form executes the atomics' address arithmetic for every
// lane); a second histogram for raw-bit forward k-mers (328 us); bank-interleaved replicas.
template <int K>
struct MotifK {
    int k_rt;
    __device__ __forceinline__ int k() const { return K ? K : k_rt; }
    __device__ __forceinline__ uint32_t mask2k() const { return (1u << (2 * k())) - 1u; }
    __device__ __forceinline__ uint32_t maskk() const { return (1u << k()) - 1u; }
};

#ifndef FTK_MOTIF_CTAS
#define FTK_MOTIF_CTAS 5
#endif
constexpr int kMotifCtasPerSm = FTK_MOTIF_CTAS;   // 5 or 6 CTAs per SM measure the same (213-217 us); 8 is slower
constexpr int kMotifNScanWords = 8192;      // longest span (in 32-base mask words) a CTA pre-scans for N

template <int K, int MODE, bool SMEM, bool BREAKPOINT>
__global__ void __launch_bounds__(kMotifThreads, kMotifCtasPerSm)
end_motif_kernel(const int32_t *__restrict__ frag_start, const int32_t *__restrict__ frag_stop,
                 const uint8_t *__restrict__ frag_mapq, const uint8_t *__restrict__ frag_strand,
                 const uint32_t *__restrict__ seq, const uint32_t *__restrict__ nmask, int64_t contig_len,
                 const int32_t *__restrict__ ivl_start, const int32_t *__restrict__ ivl_stop,
                 const int64_t *__restrict__ ranges, int k, int strand_mode, int min_mapq, int max_frag_len,
                 int pooled, int splits, unsigned long long *__restrict__ counts,
                 int32_t *__restrict__ error_flag) {
    // ONE histogram for both ends, indexed like the reference's table (forward k-mers digit-reversed per
    // fragment).  Measured alternatives that lost: a second histogram holding the forward k-mers under their
    // raw window bits, re-indexed at the flush (saves the digit reversal, 328 us against 252 us for k = 4 -
    // not understood: same number of atomics, fewer instructions); 4 / 8 / 16 bank-interleaved replicas (no
    // change).  The cost that remains is the shared-memory atomic unit itself (DESIGN.md §4.1).
    __shared__ int s_cnt[SMEM ? (K ? (1 << (2 * K)) : kMotifSmemBins) : 1];
    const int tid = threadIdx.x;
    MotifK<K> KK{k};
    const int n_bins = 1 << (2 * KK.k());
    const int64_t ivl = blockIdx.x / splits;
    const int split = blockIdx.x % splits;
    unsigned long long *__restrict__ row = counts + (pooled ? 0 : ivl * (int64_t)n_bins);
    int64_t lo, hi;
    slice_of(ranges, ivl, split, splits, lo, hi);
    if (hi <= lo) return;

    const int S = ivl_start[ivl], E = ivl_stop[ivl];
    const int len32 = (int)min(contig_len, (int64_t)INT32_MAX);     // 32-bit everything inside the slice
    const int mode = (MODE < 3) ? MODE : strand_mode;
    const int kk = KK.k();
    const uint32_t mask2k = KK.mask2k(), maskk = KK.maskk();

    // the slice is widened to a 16-byte boundary on the left so that every lane loads 4 fragments per
    // 128-bit load; the (at most three) fragments left of lo get stop = INT32_MIN and fail the overlap test
    const int64_t lo_al = lo & ~(int64_t)3;
    const int skip = (int)(lo - lo_al);
    const int cnt = (int)(hi - lo_al);
    const int nvec = cnt >> 2;
    const int4 *__restrict__ vs = reinterpret_cast<const int4 *>(frag_start + lo_al);
    const int4 *__restrict__ ve = reinterpret_cast<const int4 *>(frag_stop + lo_al);
    const uchar4 *__restrict__ vq = reinterpret_cast<const uchar4 *>(frag_mapq ? frag_mapq + lo_al : nullptr);
    const uchar4 *__restrict__ vd = reinterpret_cast<const uchar4 *>(frag_strand ? frag_strand + lo_al : nullptr);
    auto load = [&](int v, int4 &s4, int4 &e4, uchar4 &q4, uchar4 &d4) {
        if (v < nvec) {
            s4 = __ldcs(vs + v); e4 = __ldcs(ve + v);
            q4 = vq ? __ldcs(vq + v) : make_uchar4(255, 255, 255, 255);
            d4 = vd ? __ldcs(vd + v) : make_uchar4(1, 1, 1, 1);
        } else {
            s4 = make_int4(0, 0, 0, 0); e4 = make_int4(INT32_MIN, INT32_MIN, INT32_MIN, INT32_MIN);
            q4 = make_uchar4(0, 0, 0, 0); d4 = make_uchar4(1, 1, 1, 1);
        }
    };
    // the first vector of every thread is requested before the N pre-scan so that the two overlap
    int4 s_c, e_c;
    uchar4 q_c, d_c;
    load(tid, s_c, e_c, q_c, d_c);
    if (tid == 0 && skip) {
        e_c.x = INT32_MIN;
        if (skip > 1) e_c.y = INT32_MIN;
        if (skip > 2) e_c.z = INT32_MIN;
    }

    // does the span this slice can touch hold any N?  (start-sorted: first start .. last start + longest fragment)
    int any_n = 1;
    {
        const int64_t p_lo = max((int64_t)__ldg(frag_start + lo) - kk, (int64_t)0);
        const int64_t p_hi = min((int64_t)__ldg(frag_start + hi - 1) + max_frag_len + 2 * kk, (int64_t)len32);
        const int64_t w_lo = p_lo >> 5, w_hi = (p_hi >> 5) + 1;     // has_n reads words w and w + 1
        unsigned acc = 0;
        if (p_hi >= p_lo && w_hi - w_lo < kMotifNScanWords) {
            for (int64_t w = w_lo + tid; w <= w_hi; w += kMotifThreads) acc |= __ldg(nmask + w);
        } else {
            acc = 1u;
        }
        if (SMEM) for (int b = tid; b < n_bins; b += kMotifThreads) s_cnt[b] = 0;
        any_n = __syncthreads_or(acc != 0u);
    }

    // The shared histograms are addressed through their 32-bit shared-window address and bumped with
    // red.shared: left to itself the compiler re-derives that address per atomic (S2R SR_CgaCtaId + LEA
    // in the hot loop - measured 3x slower than the whole rest of the loop).
    uint32_t s_base = 0u;
    if (SMEM) {     // laundered through an opaque move so that it is computed once and kept in a register
        const uint32_t a = static_cast<uint32_t>(__cvta_generic_to_shared(s_cnt));
        asm volatile("mov.b32 %0, %1;" : "=r"(s_base) : "r"(a));
    }
    auto bump_s = [&](uint32_t byte_off) {
        asm volatile("red.shared.add.u32 [%0], 1;" :: "r"(s_base + byte_off) : "memory");
    };
    auto stream = [&](auto ncheck_tag) {
        constexpr bool NCHECK = decltype(ncheck_tag)::value;
        auto fwd = [&](int pos) {      // k-mer read 5'->3' on the forward strand starting at pos
            if (NCHECK && has_n(nmask, pos, maskk)) return;
            const uint32_t wbits = window2(seq, pos, mask2k);
            if (SMEM) bump_s(digit_reverse(wbits, kk) << 2);
            else atomicAdd(&row[digit_reverse(wbits, kk)], 1ull);
        };
        auto rev = [&](int pos) {      // reverse complement of ref[pos, pos + k)
            if (NCHECK && has_n(nmask, pos, maskk)) return;
            const uint32_t idx = (~window2(seq, pos, mask2k)) & mask2k;
            if (SMEM) bump_s(idx << 2);
            else atomicAdd(&row[idx], 1ull);
        };
        auto visit = [&](int fs, int fe, int q, int sd) {
            if (q < min_mapq || !(fe > S && fs < E)) return;
            if (BREAKPOINT) {
                const int h = kk >> 1;
                if (fs < h || fs >= len32 - h) return;                       // too close to a contig end
                if ((kk & 1) != 0) return;                                   // 2h != k: never counted
                if (mode == 0 || (mode == 1 && sd)) fwd(fs - h);
                if (mode != 1) {
                    if (fe < h || fe > len32 - h) return;                    // OutOfBoundsError -> skipped
                    rev(fe - h);
                }
                return;
            }
            if (mode == 1 && !sd) return;                // forward-only: '+' fragments only
            if (mode != 2) {
                if ((unsigned)fs > (unsigned)(len32 - kk)) return;           // fs < 0 or past the end: ValueError -> `continue`
                fwd(fs);
            }
            if (mode != 1) {
                if (fe < kk || fe > len32) {
                    if (mode == 0) atomicOr(error_flag, 1);                  // RuntimeError in the reference
                    return;
                }
                rev(fe - kk);
            }
        };
        // software pipeline: the next vector of the thread is in flight while the current one is turned
        // into window reads and atomics
        for (int v = tid; v < nvec; v += kMotifThreads) {
            int4 s_n, e_n;
            uchar4 q_n, d_n;
            if (v + 2 * kMotifThreads < nvec) {     // two iterations ahead: pull the lines into L2 (no registers held)
                asm volatile("prefetch.global.L2 [%0];" :: "l"(vs + v + 2 * kMotifThreads));
                asm volatile("prefetch.global.L2 [%0];" :: "l"(ve + v + 2 * kMotifThreads));
            }
            load(v + kMotifThreads, s_n, e_n, q_n, d_n);
            visit(s_c.x, e_c.x, q_c.x, d_c.x);
            visit(s_c.y, e_c.y, q_c.y, d_c.y);
            visit(s_c.z, e_c.z, q_c.z, d_c.z);
            visit(s_c.w, e_c.w, q_c.w, d_c.w);
            s_c = s_n; e_c = e_n; q_c = q_n; d_c = d_n;
        }
        {   // tail: at most 3 fragments
            const int i = nvec * 4 + tid;
            if (i < cnt && i >= skip)
                visit(__ldcs(frag_start + lo_al + i), __ldcs(frag_stop + lo_al + i),
                      frag_mapq ? (int)__ldcs(frag_mapq + lo_al + i) : 255,
                      frag_strand ? (int)__ldcs(frag_strand + lo_al + i) : 1);
        }
    };
    if (any_n) stream(std::true_type{});
    else stream(std::false_type{});
    if (SMEM) {
        __syncthreads();
        for (int b = tid; b < n_bins; b += kMotifThreads) {
            const int cr = s_cnt[b];
            if (cr) atomicAdd(&row[b], (unsigned long long)cr);
        }
    }
}

}  // namespace ftk

using namespace ftk;

template <bool BREAKPOINT>
static int motif_hist_launch(const int32_t *frag_start, const int32_t *frag_stop,
                             const uint8_t *frag_mapq, const uint8_t *frag_strand,
                             int64_t n_frag, int32_t max_frag_len,
                             const uint32_t *seq_words, const uint32_t *nmask_words, int64_t contig_len,
                             const int32_t *ivl_start, const int32_t *ivl_stop, int64_t n_ivl,
                             int32_t k, int32_t strand_mode, int32_t min_mapq,
                             int32_t pooled, int32_t splits,
                             int64_t *scratch, uint64_t *counts, int32_t *error_flag,
                             ftk_stream_t stream_) {
    if (n_ivl == 0) return FTK_OK;
    if (n_frag < 0 || n_ivl < 0 || splits < 1 || k < 1 || k > 12) return FTK_E_INVALID;
    if (strand_mode < 0 || strand_mode > 2) return FTK_E_INVALID;
    if (!seq_words || !nmask_words || !ivl_start || !ivl_stop || !scratch || !counts) return FTK_E_INVALID;
    if (!BREAKPOINT && !error_flag) return FTK_E_INVALID;
    if (n_frag > 0 && (!frag_start || !frag_stop)) return FTK_E_INVALID;
    if (n_ivl * (int64_t)splits > INT32_MAX) return FTK_E_RANGE;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    // overlap: fe > S (=> fs > S - max_frag_len) and fs < E
    const int mfl = max_frag_len < 0 ? 0 : max_frag_len;
    const int rc = launch_candidate_ranges(frag_start, n_frag, ivl_start, ivl_stop, false, n_ivl, mfl, 0, scratch, stream);
    if (rc != FTK_OK) return rc;
    const unsigned grid = (unsigned)(n_ivl * splits);
    auto *c = reinterpret_cast<unsigned long long *>(counts);
#define FTK_MOTIF(K, MODE, SMEM)                                                                             \
    end_motif_kernel<K, MODE, SMEM, BREAKPOINT><<<grid, kMotifThreads, 0, stream>>>(                         \
        frag_start, frag_stop, frag_mapq, frag_strand, seq_words, nmask_words, contig_len, ivl_start,        \
        ivl_stop, scratch, k, strand_mode, min_mapq, mfl, pooled, splits, c, error_flag)
    // the common cases are compiled with K and the strand mode fixed; everything else takes the runtime variant
    if (k == 4 && strand_mode == 0) FTK_MOTIF(4, 0, true);
    else if (k == 6 && strand_mode == 0) FTK_MOTIF(6, 0, true);
    else if (k == 3 && strand_mode == 0) FTK_MOTIF(3, 0, true);
    else if (k == 5 && strand_mode == 0) FTK_MOTIF(5, 0, true);
    else if ((1 << (2 * k)) <= kMotifSmemBins) FTK_MOTIF(0, 3, true);
    else FTK_MOTIF(0, 3, false);
#undef FTK_MOTIF
    FTK_CHECK_LAUNCH("end_motif_kernel");
    return FTK_OK;
}

extern "C" int ftk_end_motif_hist_u64(const int32_t *frag_start, const int32_t *frag_stop,
                                      const uint8_t *frag_mapq, const uint8_t *frag_strand,
                                      int64_t n_frag, int32_t max_frag_len,
                                      const uint32_t *seq_words, const uint32_t *nmask_words,
                                      int64_t contig_len,
                                      const int32_t *ivl_start, const int32_t *ivl_stop, int64_t n_ivl,
                                      int32_t k, int32_t strand_mode, int32_t min_mapq,
                                      int32_t pooled, int32_t splits,
                                      int64_t *scratch, uint64_t *counts, int32_t *error_flag,
                                      ftk_stream_t stream_) {
    return motif_hist_launch<false>(frag_start, frag_stop, frag_mapq, frag_strand, n_frag, max_frag_len,
                                    seq_words, nmask_words, contig_len, ivl_start, ivl_stop, n_ivl, k,
                                    strand_mode, min_mapq, pooled, splits, scratch, counts, error_flag, stream_);
}

extern "C" int ftk_breakpoint_motif_hist_u64(const int32_t *frag_start, const int32_t *frag_stop,
                                             const uint8_t *frag_mapq, const uint8_t *frag_strand,
                                             int64_t n_frag, int32_t max_frag_len,
                                             const uint32_t *seq_words, const uint32_t *nmask_words,
                                             int64_t contig_len,
                                             const int32_t *ivl_start, const int32_t *ivl_stop, int64_t n_ivl,
                                             int32_t k, int32_t strand_mode, int32_t min_mapq,
                                             int32_t pooled, int32_t splits,
                                             int64_t *scratch, uint64_t *counts, ftk_stream_t stream_) {
    return motif_hist_launch<true>(frag_start, frag_stop, frag_mapq, frag_strand, n_frag, max_frag_len,
                                   seq_words, nmask_words, contig_len, ivl_start, ivl_stop, n_ivl, k,
                                   strand_mode, min_mapq, pooled, splits, scratch, counts, nullptr, stream_);
}
