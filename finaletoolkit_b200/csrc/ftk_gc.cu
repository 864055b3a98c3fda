// Fragment GC bias: observed and expected fragment counts by (length, G+C bases) on the 2-bit packed contig.
//
// A placement [p, p + L) counts when p >= 0, p + L <= contig_len, its midpoint p + L / 2 lies in a region and
// none of its bases is N; its key is (L - min_len, g) with g = G/C bases in [p, p + L).
//   observed: every passing fragment (mapq >= min_mapq, min_len <= L <= max_len) is one placement.
//   expected: every (p, L) with L in [min_len, max_len] is one placement.
// out[(L - min_len) * (max_len + 1) + g] += 1 in both kernels (DESIGN.md 4.10).
// weighted: the model applied; selected fragments counted per interval or by offset from a site centre, with their
// weights[(L - min_len) * (max_len + 1) + g] summed where g is defined (DESIGN.md 4.11).
//
// Packed layout (synth.pack_twobit): base i in bits 2(i%16) of seq word i/16 (A0 C1 G2 T3), its N flag in bit
// i%32 of nmask word i/32.  A 64-bit seq word k and nmask word k cover the same 32 bases, so every read here is
// one aligned 64-bit seq load + one 32-bit nmask load per 32 bases; G/C <=> bit0 ^ bit1 of a base's code.
#include "ftk_common.cuh"

namespace ftk {

constexpr int kGcThreads = 256;
constexpr int kGcObsUnroll = 4;
constexpr int kGcLanes = 32;   // lengths per expected CTA: lane l owns length Lb + l

__device__ __forceinline__ void red_global_add_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("red.global.add.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}

__device__ __forceinline__ uint64_t gc_bits64(uint64_t x) {   // bit 2j set <=> base j of the word is C or G
    return (x ^ (x >> 1)) & 0x5555555555555555ull;
}

// G/C bases g of [fs, fe) and whether any of its bases is N (0 <= fs < fe <= contig_len).  Walks the 32-base
// words of the span: the N flags OR-ed from the end-masked nmask words, G/C by popc of the end-masked 64-bit G/C
// bit pairs (a caller drops a fragment with an N before G/C of an N base could matter, so the G/C bits need no
// N mask).
struct GcWalk {
    int g;
    bool has_n;
};

__device__ __forceinline__ GcWalk gc_walk(const uint64_t *__restrict__ seq64, const uint32_t *__restrict__ nmask,
                                          int fs, int fe) {
    const int k0 = fs >> 5, k1 = (fe - 1) >> 5;
    int g = 0;
    uint32_t n = 0;
    for (int k = k0; k <= k1; ++k) {
        uint32_t sel = ~0u;
        if (k == k0) sel &= ~0u << (fs & 31);
        if (k == k1) sel &= ~0u >> (31 - ((fe - 1) & 31));
        uint64_t sel2 = ~0ull;                               // sel spread to the base pairs of the seq word
        if (k == k0) sel2 &= ~0ull << (2 * (fs & 31));
        if (k == k1) sel2 &= ~0ull >> (62 - 2 * ((fe - 1) & 31));
        n |= __ldg(nmask + k) & sel;
        g += __popcll(gc_bits64(__ldg(seq64 + k)) & sel2);
    }
    return GcWalk{g, n != 0};
}

// ------------------------------------------------------------------------------------------------ observed
// One WARP per (region, split) unit streams a slice of the region's candidate range (the layout of
// vplot_warp_kernel).  A passing fragment's lane walks its words (gc_walk), then one 64-bit global RED.
__global__ void __launch_bounds__(kGcThreads)
gc_observed_warp_kernel(const int32_t *__restrict__ frag_start, const int32_t *__restrict__ frag_stop,
                        const uint8_t *__restrict__ frag_mapq, const uint64_t *__restrict__ seq64,
                        const uint32_t *__restrict__ nmask, int64_t contig_len, const int32_t *__restrict__ reg_start,
                        const int32_t *__restrict__ reg_stop, const int64_t *__restrict__ ranges, int min_len,
                        int max_len, int min_mapq, int splits, int64_t n_units, unsigned long long *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t unit = (int64_t)blockIdx.x * (kGcThreads / 32) + (threadIdx.x >> 5);
    if (unit >= n_units) return;
    const int64_t reg = unit / splits;
    const int split = (int)(unit % splits);
    const int S = __ldg(reg_start + reg);
    const unsigned reg_len = (unsigned)(__ldg(reg_stop + reg) - S);
    int64_t lo, hi;
    slice_of(ranges, reg, split, splits, lo, hi);

    const unsigned len_span = (unsigned)(max_len - min_len);
    const int64_t row = (int64_t)max_len + 1;
    auto visit = [&](int fs, int fe, int q, int, int) {
        const int L = fe - fs;                                   // the sentinel (L = -1) fails the length test
        const int m = fs + (L >> 1);
        const bool ok = ((unsigned)(L - min_len) <= len_span) & (q >= min_mapq) & ((unsigned)(m - S) < reg_len) &
                        (fs >= 0) & ((int64_t)fe <= contig_len);
        if (!ok) return;
        const GcWalk w = gc_walk(seq64, nmask, fs, fe);
        if (!w.has_n) red_global_add_u64(out + (int64_t)(L - min_len) * row + w.g, 1ull);
    };
    stream_fragments<32, kGcObsUnroll>(FragCols{frag_start, frag_stop, frag_mapq, nullptr}, lo, hi, lane, visit);
}

// ------------------------------------------------------------------------------------------------ weighted
// The GC model applied (DESIGN.md 4.11).  A fragment is selected when mapq >= min_mapq, min_len <= L <= max_len
// and its midpoint m passes the unit's position test; it adds 1 to the count and, when it lies in the contig and
// touches no N (the placement rule of gc_observed), weights[(L - min_len) * (max_len + 1) + g] to the corrected sum.
// One WARP per (unit, split), as in gc_observed_warp_kernel.
//   SITES = false: unit = interval [S, E) (FTK_NONE = unbounded), test S <= m < E.  Each lane keeps a uint64
//     count and an fp64 sum; a fixed xor-shuffle tree reduces them and lane 0 writes the unit's partial, so the
//     result depends only on the launch shape (gc_weighted_combine_kernel adds the splits in order).
//   SITES = true: unit = site, centre c = win_lo + flank, d = m - c ('-' sites: c - m), test |d| <= flank; every
//     selected fragment is a 64-bit RED into count[d + flank] and an fp64 RED into corrected[d + flank].
__device__ __forceinline__ void red_global_add_f64(double *p, double v) {
    asm volatile("red.global.add.f64 [%0], %1;" :: "l"(p), "d"(v) : "memory");
}

template <bool SITES>
__global__ void __launch_bounds__(kGcThreads)
gc_weighted_warp_kernel(const int32_t *__restrict__ frag_start, const int32_t *__restrict__ frag_stop,
                        const uint8_t *__restrict__ frag_mapq, const uint64_t *__restrict__ seq64,
                        const uint32_t *__restrict__ nmask, int64_t contig_len, const int32_t *__restrict__ unit_lo,
                        const int32_t *__restrict__ unit_hi, const uint8_t *__restrict__ site_flip,
                        const int64_t *__restrict__ ranges, const double *__restrict__ weights, int flank, int min_len,
                        int max_len, int min_mapq, int splits, int64_t n_units,
                        unsigned long long *__restrict__ count, double *__restrict__ corrected) {
    const int lane = threadIdx.x & 31;
    const int64_t unit = (int64_t)blockIdx.x * (kGcThreads / 32) + (threadIdx.x >> 5);
    if (unit >= n_units) return;
    const int64_t k = unit / splits;
    const int split = (int)(unit % splits);
    int64_t lo, hi;
    slice_of(ranges, k, split, splits, lo, hi);
    // SITES: the window is [c - flank, c + flank + 1); intervals: m in [m_lo, m_last] (inclusive, so that an
    // unbounded stop admits a midpoint of 2^31 - 1)
    const int S = __ldg(unit_lo + k);
    const int c = S + flank;
    const bool flip = SITES && __ldg(site_flip + k) != 0;
    const int E = SITES ? 0 : __ldg(unit_hi + k);
    const int m_lo = (S == FTK_NONE) ? INT32_MIN : S;
    const int m_last = (E == FTK_NONE) ? INT32_MAX : E - 1;

    const unsigned len_span = (unsigned)(max_len - min_len);
    const unsigned width = 2u * (unsigned)flank;
    const int64_t row = (int64_t)max_len + 1;
    unsigned long long my_count = 0;
    double my_sum = 0.0;
    auto visit = [&](int fs, int fe, int q, int, int) {
        const int L = fe - fs;                                   // the sentinel (L = -1) fails the length test
        const int m = fs + (L >> 1);
        const int64_t d = flip ? (int64_t)c - m : (int64_t)m - c;
        const bool pos = SITES ? ((uint64_t)(d + flank) <= width) : ((m >= m_lo) & (m <= m_last));
        if (!(((unsigned)(L - min_len) <= len_span) & (q >= min_mapq) & pos)) return;
        double w = 0.0;
        const bool placed = (fs >= 0) & ((int64_t)fe <= contig_len);
        if (placed) {
            const GcWalk gw = gc_walk(seq64, nmask, fs, fe);
            if (!gw.has_n) w = __ldg(weights + (int64_t)(L - min_len) * row + gw.g);
        }
        if (SITES) {
            red_global_add_u64(count + (d + flank), 1ull);
            if (w != 0.0) red_global_add_f64(corrected + (d + flank), w);
        } else {
            ++my_count;
            my_sum += w;
        }
    };
    stream_fragments<32, kGcObsUnroll>(FragCols{frag_start, frag_stop, frag_mapq, nullptr}, lo, hi, lane, visit);
    if (SITES) return;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {                           // every lane ends with the same tree's result
        my_count += __shfl_xor_sync(0xffffffffu, my_count, o);
        my_sum += __shfl_xor_sync(0xffffffffu, my_sum, o);
    }
    if (lane == 0) {
        count[unit] = my_count;
        corrected[unit] = my_sum;
    }
}

// out_count[i] += the partial counts of interval i, out_corrected[i] += its partial sums, split 0 first.
__global__ void __launch_bounds__(kGcThreads)
gc_weighted_combine_kernel(const unsigned long long *__restrict__ part_count, const double *__restrict__ part_sum,
                           int64_t n_ivl, int splits, unsigned long long *__restrict__ out_count,
                           double *__restrict__ out_corrected) {
    const int64_t i = (int64_t)blockIdx.x * kGcThreads + threadIdx.x;
    if (i >= n_ivl) return;
    unsigned long long c = out_count[i];
    double w = out_corrected[i];
    for (int s = 0; s < splits; ++s) {
        c += part_count[i * splits + s];
        w += part_sum[i * splits + s];
    }
    out_count[i] = c;
    out_corrected[i] = w;
}

// ------------------------------------------------------------------------------------------------ expected
// A CTA per (tile of midpoints [m0, m1) inside one region, group of 32 lengths Lb .. Lb + 31).
//  1. Stage, for the bases [a0, a0 + span) that the group's placements touch, the packed prefix counts
//     P[i] = (G/C bases in [a0, a0 + i)) | (N bases in [a0, a0 + i)) << 16 in shared memory (span < 2^16, so
//     neither field overflows and P[e] - P[p] subtracts both fields at once).
//  2. Lane l owns L = Lb + l; the warps walk consecutive midpoints.  Placement (m, L) is [p, e) with
//     p = m - L / 2, e = p + L: g and the N test are two shared loads.  A lane counts a run of equal g in a
//     register and adds it to its histogram row with one shared RED when g changes or a placement is invalid.
//  3. The CTA flushes its nonzero bins with 64-bit global REDs.
struct GcExpSmem {
    uint32_t *P, *hist, *cgc, *cn, *cbase;
};

__host__ __device__ __forceinline__ int gc_exp_span_cap(int tile_cap, int max_len) {
    return tile_cap + max_len + 64;   // midpoints + halo + the alignment of a0 to a 32-base word
}

__host__ __device__ __forceinline__ size_t gc_exp_smem_bytes(int tile_cap, int max_len) {
    const int span = gc_exp_span_cap(tile_cap, max_len);
    const int nch = span / 32 + 1;
    return 4 * ((size_t)span + 1 + (size_t)kGcLanes * (max_len + 1) + 3 * (size_t)nch);
}

__global__ void __launch_bounds__(kGcThreads)
gc_expected_kernel(const uint64_t *__restrict__ seq64, const uint32_t *__restrict__ nmask, int64_t contig_len,
                   const int32_t *__restrict__ tile_lo, const int32_t *__restrict__ tile_hi, int tile_cap,
                   int min_len, int max_len, unsigned long long *__restrict__ out) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int span_cap = gc_exp_span_cap(tile_cap, max_len);
    const int nch_cap = span_cap / 32 + 1;
    const int stride = max_len + 1;
    uint32_t *P = smem;
    uint32_t *hist = P + span_cap + 1;
    uint32_t *cgc = hist + kGcLanes * stride, *cn = cgc + nch_cap, *cbase = cn + nch_cap;

    const int Lb = min_len + (int)blockIdx.y * kGcLanes;
    const int Lhi = min(Lb + kGcLanes - 1, max_len);
    const int64_t m0 = __ldg(tile_lo + blockIdx.x);
    const int64_t m1 = min((int64_t)__ldg(tile_hi + blockIdx.x), m0 + tile_cap);
    if (m1 <= m0) return;
    // bases [a0, top): the lowest p of the group down to the highest e (clipped to the contig)
    const int64_t a0 = max(m0 - (Lhi >> 1), (int64_t)0) & ~(int64_t)31;
    const int64_t top = min(m1 - 1 + (Lhi - (Lhi >> 1)), contig_len);
    const int span = (int)max(top - a0, (int64_t)0);
    const int nch = (span + 31) >> 5;
    const int rows_stride = Lhi + 1;   // bins this group can reach (g <= L <= Lhi)

    for (int i = tid; i < kGcLanes * rows_stride; i += kGcThreads) hist[i] = 0u;
    // per-word G/C and N bit masks of the span, and their block-wide exclusive prefix
    uint32_t carry = 0;
    __shared__ uint32_t warp_sum[kGcThreads / 32];
    for (int c0 = 0; c0 < nch; c0 += kGcThreads) {
        const int c = c0 + tid;
        uint32_t gmask = 0, nm = 0;
        if (c < nch) {
            const int64_t k = (a0 >> 5) + c;
            const uint64_t x = gc_bits64(__ldg(seq64 + k));
            nm = __ldg(nmask + k);
            uint32_t gm = 0;
#pragma unroll
            for (int j = 0; j < 32; ++j) gm |= (uint32_t)((x >> (2 * j)) & 1ull) << j;
            gmask = gm & ~nm;
            const int keep = span - 32 * c;                     // bases of this word inside the span
            if (keep < 32) { const uint32_t m = (1u << keep) - 1u; gmask &= m; nm &= m; }
            cgc[c] = gmask; cn[c] = nm;
        }
        const uint32_t v = (uint32_t)__popc(gmask) | ((uint32_t)__popc(nm) << 16);
        uint32_t incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) warp_sum[warp] = incl;
        __syncthreads();
        uint32_t before = carry, total = 0;
#pragma unroll
        for (int w = 0; w < kGcThreads / 32; ++w) {
            const uint32_t s = warp_sum[w];
            before += (w < warp) ? s : 0u;
            total += s;
        }
        if (c < nch) cbase[c] = before + incl - v;
        carry += total;
        __syncthreads();
    }
    for (int i = tid; i <= span; i += kGcThreads) {
        const int c = i >> 5, j = i & 31;
        if (c >= nch) { P[i] = carry; continue; }           // i == span on a word boundary: the total
        const uint32_t below = (1u << j) - 1u;
        P[i] = cbase[c] + (uint32_t)__popc(cgc[c] & below) + ((uint32_t)__popc(cn[c] & below) << 16);
    }
    __syncthreads();

    // walk the midpoints: warp w takes a contiguous share, lane l the length Lb + l
    const int L = Lb + lane;
    const bool lane_on = L <= Lhi;
    const int n_mid = (int)(m1 - m0);
    const int share = (n_mid + kGcThreads / 32 - 1) / (kGcThreads / 32);
    const int r0 = warp * share, r1 = min(n_mid, r0 + share);
    const int off = (int)(m0 - a0) - (L >> 1);                   // p - a0 of the warp's midpoint r: off + r
    const uint32_t row_addr = smem_addr_once(hist + lane * rows_stride);
    int cur = -1, run = 0;
    for (int r = r0; r < r1; ++r) {
        const int p = off + r, e = p + L;
        int g = -1;
        if (lane_on & (p >= 0) & (e <= span)) {                   // p >= 0 <=> placement start >= 0; e <= span <=> end <= contig_len
            const uint32_t d = P[e] - P[p];
            g = (d >> 16) ? -1 : (int)(d & 0xffffu);
        }
        if (g != cur) {
            if (cur >= 0) red_shared_add(row_addr + 4u * (uint32_t)cur, run);
            cur = g; run = 0;
        }
        ++run;
    }
    if (cur >= 0) red_shared_add(row_addr + 4u * (uint32_t)cur, run);
    __syncthreads();

    for (int i = tid; i < kGcLanes * rows_stride; i += kGcThreads) {
        const uint32_t h = hist[i];
        const int l = i / rows_stride, g = i - l * rows_stride;
        if (h) red_global_add_u64(out + (int64_t)(Lb + l - min_len) * stride + g, (unsigned long long)h);
    }
}

}  // namespace ftk

using namespace ftk;

static int gc_common_args(const uint32_t *seq_words, const uint32_t *nmask_words, int64_t contig_len, int32_t min_len,
                          int32_t max_len, const uint64_t *out) {
    if (!seq_words || !nmask_words || !out || contig_len < 0 || min_len < 1 || max_len < min_len) return FTK_E_INVALID;
    if (max_len > FTK_GC_MAX_LENGTH || contig_len > INT32_MAX) return FTK_E_RANGE;
    if ((reinterpret_cast<uintptr_t>(seq_words) & 7) != 0) return FTK_E_INVALID;   // read as 64-bit words
    return FTK_OK;
}

extern "C" int ftk_gc_observed_u64(const int32_t *frag_start, const int32_t *frag_stop, const uint8_t *frag_mapq,
                                   int64_t n_frag, int32_t max_frag_len, const uint32_t *seq_words,
                                   const uint32_t *nmask_words, int64_t contig_len, const int32_t *reg_start,
                                   const int32_t *reg_stop, int64_t n_reg, int32_t min_len, int32_t max_len,
                                   int32_t min_mapq, int32_t splits, int64_t *scratch, uint64_t *out,
                                   ftk_stream_t stream_) {
    if (n_reg == 0) return FTK_OK;
    if (n_frag < 0 || n_reg < 0 || splits < 1 || !reg_start || !reg_stop || !scratch) return FTK_E_INVALID;
    if (n_frag > 0 && (!frag_start || !frag_stop)) return FTK_E_INVALID;
    const int rc0 = gc_common_args(seq_words, nmask_words, contig_len, min_len, max_len, out);
    if (rc0 != FTK_OK) return rc0;
    if (n_reg > INT32_MAX / 2 || n_reg * (int64_t)splits > INT32_MAX) return FTK_E_RANGE;
    if (n_frag == 0) return FTK_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    // m in [S, E) and m = s + L/2 with L <= min(max_frag_len, max_len): S - reach <= s < E
    const int reach = (max_frag_len < max_len ? (max_frag_len < 0 ? 0 : max_frag_len) : max_len) >> 1;
    const int rc = launch_candidate_ranges(frag_start, n_frag, reg_start, reg_stop, false, n_reg, reach, 0, scratch, stream);
    if (rc != FTK_OK) return rc;
    const int64_t n_units = n_reg * (int64_t)splits;
    const int per_cta = kGcThreads / 32;
    gc_observed_warp_kernel<<<(unsigned)((n_units + per_cta - 1) / per_cta), kGcThreads, 0, stream>>>(
        frag_start, frag_stop, frag_mapq, reinterpret_cast<const uint64_t *>(seq_words), nmask_words, contig_len,
        reg_start, reg_stop, scratch, min_len, max_len, min_mapq, splits, n_units,
        reinterpret_cast<unsigned long long *>(out));
    FTK_CHECK_LAUNCH("gc_observed_warp_kernel");
    return FTK_OK;
}

static int gc_weighted_args(const int32_t *frag_start, const int32_t *frag_stop, int64_t n_frag,
                            const uint32_t *seq_words, const uint32_t *nmask_words, int64_t contig_len,
                            const int32_t *unit_lo, const int32_t *unit_hi, int64_t n_units, int32_t min_len,
                            int32_t max_len, int32_t splits, const int64_t *scratch, const double *weights,
                            const uint64_t *out_count, const double *out_corrected) {
    if (n_frag < 0 || n_units < 0 || splits < 1 || !unit_lo || !unit_hi || !scratch || !weights || !out_corrected)
        return FTK_E_INVALID;
    if (n_frag > 0 && (!frag_start || !frag_stop)) return FTK_E_INVALID;
    const int rc = gc_common_args(seq_words, nmask_words, contig_len, min_len, max_len, out_count);
    if (rc != FTK_OK) return rc;
    if (n_units > INT32_MAX / 2 || n_units * (int64_t)splits > INT32_MAX) return FTK_E_RANGE;
    return FTK_OK;
}

extern "C" int ftk_gc_weighted_intervals_f64(const int32_t *frag_start, const int32_t *frag_stop,
                                             const uint8_t *frag_mapq, int64_t n_frag, int32_t max_frag_len,
                                             const uint32_t *seq_words, const uint32_t *nmask_words,
                                             int64_t contig_len, const int32_t *ivl_start, const int32_t *ivl_stop,
                                             int64_t n_ivl, int32_t min_len, int32_t max_len, int32_t min_mapq,
                                             int32_t splits, int64_t *scratch, const double *weights,
                                             uint64_t *out_count, double *out_corrected, ftk_stream_t stream_) {
    if (n_ivl == 0) return FTK_OK;
    const int rc0 = gc_weighted_args(frag_start, frag_stop, n_frag, seq_words, nmask_words, contig_len, ivl_start,
                                     ivl_stop, n_ivl, min_len, max_len, splits, scratch, weights, out_count,
                                     out_corrected);
    if (rc0 != FTK_OK) return rc0;
    if (n_frag == 0) return FTK_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    // S <= m = s + L/2 < E with L <= min(max_frag_len, max_len): S - reach <= s < E
    const int reach = (max_frag_len < max_len ? (max_frag_len < 0 ? 0 : max_frag_len) : max_len) >> 1;
    const int rc = launch_candidate_ranges(frag_start, n_frag, ivl_start, ivl_stop, false, n_ivl, reach, 0, scratch, stream);
    if (rc != FTK_OK) return rc;
    const int64_t n_units = n_ivl * (int64_t)splits;
    auto *part_count = reinterpret_cast<unsigned long long *>(scratch + 2 * n_ivl);
    auto *part_sum = reinterpret_cast<double *>(scratch + 2 * n_ivl + n_units);
    const int per_cta = kGcThreads / 32;
    gc_weighted_warp_kernel<false><<<(unsigned)((n_units + per_cta - 1) / per_cta), kGcThreads, 0, stream>>>(
        frag_start, frag_stop, frag_mapq, reinterpret_cast<const uint64_t *>(seq_words), nmask_words, contig_len,
        ivl_start, ivl_stop, nullptr, scratch, weights, 0, min_len, max_len, min_mapq, splits, n_units, part_count,
        part_sum);
    FTK_CHECK_LAUNCH("gc_weighted_warp_kernel<false>");
    gc_weighted_combine_kernel<<<(unsigned)((n_ivl + kGcThreads - 1) / kGcThreads), kGcThreads, 0, stream>>>(
        part_count, part_sum, n_ivl, splits, reinterpret_cast<unsigned long long *>(out_count), out_corrected);
    FTK_CHECK_LAUNCH("gc_weighted_combine_kernel");
    return FTK_OK;
}

extern "C" int ftk_gc_weighted_sites_f64(const int32_t *frag_start, const int32_t *frag_stop, const uint8_t *frag_mapq,
                                         int64_t n_frag, int32_t max_frag_len, const uint32_t *seq_words,
                                         const uint32_t *nmask_words, int64_t contig_len, const int32_t *win_lo,
                                         const int32_t *win_hi, const uint8_t *site_flip, int64_t n_sites,
                                         int32_t flank, int32_t min_len, int32_t max_len, int32_t min_mapq,
                                         int32_t splits, int64_t *scratch, const double *weights,
                                         uint64_t *out_count, double *out_corrected, ftk_stream_t stream_) {
    if (n_sites == 0) return FTK_OK;
    if (flank < 0 || !site_flip) return FTK_E_INVALID;
    const int rc0 = gc_weighted_args(frag_start, frag_stop, n_frag, seq_words, nmask_words, contig_len, win_lo,
                                     win_hi, n_sites, min_len, max_len, splits, scratch, weights, out_count,
                                     out_corrected);
    if (rc0 != FTK_OK) return rc0;
    if (flank > FTK_VPLOT_MAX_FLANK) return FTK_E_RANGE;
    if (n_frag == 0) return FTK_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    // start >= m - L/2 >= c - flank - max/2 and start <= m <= c + flank (the reaches of ftk_vplot_u64)
    const int reach = (max_frag_len < max_len ? (max_frag_len < 0 ? 0 : max_frag_len) : max_len) >> 1;
    const int rc = launch_candidate_ranges(frag_start, n_frag, win_lo, win_hi, false, n_sites, reach, 0, scratch, stream);
    if (rc != FTK_OK) return rc;
    const int64_t n_units = n_sites * (int64_t)splits;
    const int per_cta = kGcThreads / 32;
    gc_weighted_warp_kernel<true><<<(unsigned)((n_units + per_cta - 1) / per_cta), kGcThreads, 0, stream>>>(
        frag_start, frag_stop, frag_mapq, reinterpret_cast<const uint64_t *>(seq_words), nmask_words, contig_len,
        win_lo, win_hi, site_flip, scratch, weights, flank, min_len, max_len, min_mapq, splits, n_units,
        reinterpret_cast<unsigned long long *>(out_count), out_corrected);
    FTK_CHECK_LAUNCH("gc_weighted_warp_kernel<true>");
    return FTK_OK;
}

extern "C" int ftk_gc_expected_u64(const uint32_t *seq_words, const uint32_t *nmask_words, int64_t contig_len,
                                   const int32_t *tile_lo, const int32_t *tile_hi, int64_t n_tiles, int32_t tile_cap,
                                   int32_t min_len, int32_t max_len, uint64_t *out, ftk_stream_t stream_) {
    if (n_tiles == 0) return FTK_OK;
    if (n_tiles < 0 || !tile_lo || !tile_hi || tile_cap < 1) return FTK_E_INVALID;
    const int rc0 = gc_common_args(seq_words, nmask_words, contig_len, min_len, max_len, out);
    if (rc0 != FTK_OK) return rc0;
    if (tile_cap > FTK_GC_MAX_TILE || n_tiles > INT32_MAX) return FTK_E_RANGE;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const size_t smem = gc_exp_smem_bytes(tile_cap, max_len);
    FTK_CUDA_TRY(cudaFuncSetAttribute(gc_expected_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const dim3 grid((unsigned)n_tiles, (unsigned)((max_len - min_len) / kGcLanes + 1));
    gc_expected_kernel<<<grid, kGcThreads, smem, stream>>>(reinterpret_cast<const uint64_t *>(seq_words), nmask_words,
                                                           contig_len, tile_lo, tile_hi, tile_cap, min_len, max_len,
                                                           reinterpret_cast<unsigned long long *>(out));
    FTK_CHECK_LAUNCH("gc_expected_kernel");
    return FTK_OK;
}
