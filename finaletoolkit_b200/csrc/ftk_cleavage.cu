// Cleavage profile (Zhou et al. 2022) and per-base fragment depth on sm_100a.
//
// Replaces _coverage_and_ends (frag/_cleavage_profile.py:33-90: np.add.at difference array +
// cumsum for depth, bincount of strand-selected ends) and the proportion step of
// cleavage_profile (frag/_cleavage_profile.py:190-217):
//   depth[p]  = #{fragments with start <= p < stop}       (start/stop clipped to the interval)
//   ends[p]   = #{'+' fragments with start == p} + #{'-' fragments with stop == p}
//   out[p]    = depth ? ends / depth * 100 : 0             (fp64, same operation order)
// over the fragments of frag_array(..., intersect_policy="any") for the interval: mapq >= q,
// inclusive length window, stop > interval_start and start < interval_stop.
// Same tile machinery as WPS: one CTA per <= 5120-position tile, events scattered with shared
// atomics into a difference array (+1 at start, -1 at stop, clamped onto the first slot /
// dropped past the last) and an end-count array, block prefix scan, fp64 store.
// Roofline: HBM, 10 B per candidate fragment (start, stop, mapq, strand) + 8 B per position.
// Measured and dropped in round 2: ONE packed array (ends * 65536 + depth difference in a word: two
// atomics per fragment instead of three, 20 KB instead of 40 KB per tile, WPS-style shuffle scan) -
// 905 us with direct 16-byte stores, 1.08 ms with the results staged through the array, against
// 827 us for the two-array form below; ATOMS.ADD vs ATOMS.POPC.INC makes no difference (834 / 839 us).
//
// The depth tracks of coverage_profile run the same tile body without the end counts:
//   span:     depth[p] = #{passing fragments with start <= p < stop}   (the depth above, int32)
//   midpoint: depth[p] = #{passing fragments with (start + stop) // 2 == p}
// No strand column is read, the tile keeps only the difference array (20 KB), the midpoint form
// skips the scan (its scattered counts are the answer) and positions leave as int32 in 16-byte
// streaming stores.  Roofline: HBM, 9 B per candidate fragment + 4 B per position.
//
// The GC-corrected depth tracks (gc_depth_tile_kernel) run the same tiles with each fragment weighted by the GC
// model: an int64 difference array and scan, a G/C walk of the packed contig per passing fragment, fp64 out.
#include "ftk_common.cuh"
#include "ftk_gc_walk.cuh"

namespace ftk {

constexpr int kClvThreads = 256;
constexpr int kClvCap = 5120;
constexpr int kClvPer = kClvCap / kClvThreads;   // 20 contiguous positions per thread

enum class ClvMode { kCleavage, kDepthSpan, kDepthMid };

// Store len int32 positions of the shared tile to dst (4-byte aligned) with coalesced 16-byte streaming stores:
// up to 3 leading positions reach a 16-byte boundary, up to 3 trail.
__device__ __forceinline__ void clv_store_i32(const int *stage, int *__restrict__ dst, int len, int tid) {
    const int head = min((int)(((16u - ((unsigned)reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u) >> 2), len);
    const int nvec = (len - head) >> 2, rest = len - head - 4 * nvec;
    int4 *__restrict__ vdst = reinterpret_cast<int4 *>(dst + head);
    if (head == 0) {
        for (int p = tid; p < nvec; p += kClvThreads) st_stream4(vdst + p, reinterpret_cast<const int4 *>(stage)[p]);
    } else {
        for (int p = tid; p < nvec; p += kClvThreads) {
            const int *s = stage + head + 4 * p;
            st_stream4(vdst + p, make_int4(s[0], s[1], s[2], s[3]));
        }
    }
    if (tid < head + rest) {
        const int p = tid < head ? tid : len - rest + (tid - head);
        dst[p] = stage[p];
    }
}

// One tile of the cleavage / depth kernels (one CTA of kClvThreads per tile).
template <ClvMode MODE, class OutT>
__device__ __forceinline__ void clv_tile_body(
        const int32_t *__restrict__ frag_start, const int32_t *__restrict__ frag_stop,
        const uint8_t *__restrict__ frag_mapq, const uint8_t *__restrict__ frag_strand,
        const int32_t *__restrict__ tile_p0, const int32_t *__restrict__ tile_len,
        const int32_t *__restrict__ tile_ivl_lo, const int32_t *__restrict__ tile_ivl_hi,
        const int64_t *__restrict__ tile_out_off, const int64_t *__restrict__ ranges,
        int min_len, int max_len, int min_mapq, OutT *__restrict__ out) {
    constexpr bool kEnds = MODE == ClvMode::kCleavage;
    __shared__ __align__(16) int DE[kEnds ? 2 * kClvCap : kClvCap];
    int *D = DE;              // depth difference array (midpoint depth: the counts themselves)
    int *E = DE + kClvCap;    // fragment-end counts (the pair is recycled as double[kClvCap] for the store)
    __shared__ int warp_tot[kClvThreads / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t tile = blockIdx.x;
    const int p0 = tile_p0[tile], len = tile_len[tile];
    // depth needs no interval bounds: a fragment covering (or centred on) a tile position overlaps its interval;
    // only a zero-length fragment at an interval's first position escapes that, and the midpoint definition counts it
    int ivl_lo = 0, ivl_hi = 0;
    if constexpr (kEnds) { ivl_lo = tile_ivl_lo[tile]; ivl_hi = tile_ivl_hi[tile]; }
    const int64_t lo = ranges[2 * tile], hi = ranges[2 * tile + 1];
    for (int i = tid; i < kClvCap / 4; i += kClvThreads) {
        reinterpret_cast<int4 *>(D)[i] = make_int4(0, 0, 0, 0);
        if constexpr (kEnds) reinterpret_cast<int4 *>(E)[i] = make_int4(0, 0, 0, 0);
    }
    __syncthreads();
    const uint32_t d_addr = smem_addr_once(D), e_addr = kEnds ? smem_addr_once(E) : 0u;
    auto visit = [&](int fs, int fe, int q, int sd, int) {
        const int L = fe - fs;
        if constexpr (kEnds) {
            // frag_array(..., "any") of the INTERVAL: tabix overlap + mapq + inclusive length window
            if (q < min_mapq || L < 0 || !frag_len_ok(L, min_len, max_len) || !(fe > ivl_lo && fs < ivl_hi)) return;
        } else {
            if (q < min_mapq || L < 0 || !frag_len_ok(L, min_len, max_len)) return;
        }
        const int s_idx = fs - p0, e_idx = fe - p0;
        if constexpr (MODE == ClvMode::kDepthMid) {
            const int m_idx = s_idx + (L >> 1);          // (start + stop) // 2 - p0 without int32 overflow
            if (m_idx >= 0 && m_idx < len) red_shared_inc(d_addr + 4u * (unsigned)m_idx);
        } else if (e_idx > 0 && s_idx < len) {          // covers at least one tile position
            red_shared_inc(d_addr + 4u * (unsigned)max(s_idx, 0));
            if (e_idx < len) red_shared_add(d_addr + 4u * (unsigned)e_idx, -1);
        }
        if constexpr (kEnds) {
            const int end_idx = sd ? s_idx : e_idx;
            if (end_idx >= 0 && end_idx < len) red_shared_inc(e_addr + 4u * (unsigned)end_idx);
        }
    };
    stream_fragments<kClvThreads, 2>(FragCols{frag_start, frag_stop, frag_mapq, frag_strand}, lo, hi, tid, visit);
    __syncthreads();
    if constexpr (MODE == ClvMode::kDepthMid) {
        clv_store_i32(D, out + tile_out_off[tile], len, tid);
        return;
    }
    // block prefix scan: each thread owns kClvPer contiguous positions (int4 loads, conflict-free)
    int d[kClvPer];
    const int base = tid * kClvPer;
#pragma unroll
    for (int j = 0; j < kClvPer / 4; ++j) {
        const int4 v = *reinterpret_cast<const int4 *>(&D[base + 4 * j]);
        d[4 * j] = v.x; d[4 * j + 1] = v.y; d[4 * j + 2] = v.z; d[4 * j + 3] = v.w;
    }
#pragma unroll
    for (int j = 1; j < kClvPer; ++j) d[j] += d[j - 1];
    int t = d[kClvPer - 1];
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, t, off);
        if (lane >= off) t += n;
    }
    if (lane == 31) warp_tot[warp] = t;
    __syncthreads();
    int offset = t - d[kClvPer - 1];
#pragma unroll
    for (int w = 0; w < kClvThreads / 32; ++w) offset += (w < warp) ? warp_tot[w] : 0;
    if constexpr (!kEnds) {
        // every thread rewrites only the kClvPer positions it read, so D is the depth stage in place
#pragma unroll
        for (int j = 0; j < kClvPer / 4; ++j)
            *reinterpret_cast<int4 *>(&D[base + 4 * j]) = make_int4(d[4 * j] + offset, d[4 * j + 1] + offset,
                                                                    d[4 * j + 2] + offset, d[4 * j + 3] + offset);
        __syncthreads();
        clv_store_i32(D, out + tile_out_off[tile], len, tid);
    } else {
        int e[kClvPer];
#pragma unroll
        for (int j = 0; j < kClvPer / 4; ++j) {
            const int4 v = *reinterpret_cast<const int4 *>(&E[base + 4 * j]);
            e[4 * j] = v.x; e[4 * j + 1] = v.y; e[4 * j + 2] = v.z; e[4 * j + 3] = v.w;
        }
        __syncthreads();   // every thread holds its depth/end counts: D and E can be recycled
        double *stage = reinterpret_cast<double *>(DE);
#pragma unroll
        for (int j = 0; j < kClvPer; ++j) {
            const int depth = d[j] + offset;
            // proportions[mask] = ends[mask] / depth[mask] * 100   (frag/_cleavage_profile.py:206-208);
            // 0 / depth * 100 is exactly 0.0, so the fp64 division only runs where an end was counted
            stage[base + j] = (depth != 0 && e[j] != 0) ? (double)e[j] / (double)depth * 100.0 : 0.0;
        }
        __syncthreads();
        double *__restrict__ dst = out + tile_out_off[tile];
        if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {               // coalesced 16-byte streaming stores
            const int pairs = len >> 1;
            for (int p = tid; p < pairs; p += kClvThreads) {
                const double2 v = reinterpret_cast<const double2 *>(stage)[p];
                asm volatile("st.global.L1::no_allocate.v2.f64 [%0], {%1,%2};" :: "l"(dst + 2 * p), "d"(v.x), "d"(v.y) : "memory");
            }
            if ((len & 1) && tid == 0) dst[len - 1] = stage[len - 1];
        } else {
            for (int p = tid; p < len; p += kClvThreads) dst[p] = stage[p];
        }
    }
}

__global__ void __launch_bounds__(kClvThreads)
cleavage_tile_kernel(const int32_t *__restrict__ frag_start, const int32_t *__restrict__ frag_stop,
                     const uint8_t *__restrict__ frag_mapq, const uint8_t *__restrict__ frag_strand,
                     const int32_t *__restrict__ tile_p0, const int32_t *__restrict__ tile_len,
                     const int32_t *__restrict__ tile_ivl_lo, const int32_t *__restrict__ tile_ivl_hi,
                     const int64_t *__restrict__ tile_out_off, const int64_t *__restrict__ ranges,
                     int min_len, int max_len, int min_mapq, double *__restrict__ out) {
    clv_tile_body<ClvMode::kCleavage>(frag_start, frag_stop, frag_mapq, frag_strand, tile_p0, tile_len, tile_ivl_lo,
                                      tile_ivl_hi, tile_out_off, ranges, min_len, max_len, min_mapq, out);
}

template <bool MIDPOINT>
__global__ void __launch_bounds__(kClvThreads)
depth_tile_kernel(const int32_t *__restrict__ frag_start, const int32_t *__restrict__ frag_stop,
                  const uint8_t *__restrict__ frag_mapq,
                  const int32_t *__restrict__ tile_p0, const int32_t *__restrict__ tile_len,
                  const int64_t *__restrict__ tile_out_off, const int64_t *__restrict__ ranges,
                  int min_len, int max_len, int min_mapq, int *__restrict__ out) {
    clv_tile_body<MIDPOINT ? ClvMode::kDepthMid : ClvMode::kDepthSpan>(
        frag_start, frag_stop, frag_mapq, nullptr, tile_p0, tile_len, nullptr, nullptr, tile_out_off, ranges,
        min_len, max_len, min_mapq, out);
}

// ------------------------------------------------------------------------------------------------ GC-weighted depth
// The depth tracks with the GC model applied (DESIGN.md 4.14).  A fragment passes when mapq >= min_mapq and
// min_len <= L <= max_len; when its placement is defined (start >= 0, stop <= contig_len, no N base: the rule of
// gc_observed) it adds its quantised weight Q[(L - min_len) * (max_len + 1) + g] (int64, units of 2^-32) where
// depth_tile_kernel adds 1.  The tile keeps an int64 difference array (40 KB): span mode scans it in int64, midpoint
// mode stores the scattered sums; every position leaves as fp64(sum) * 2^-32.  Integer sums do not depend on the
// order of the atomics, so the track is exact and bit-identical between runs and batchings.  No partial sum can
// exceed (candidates of the tile) * max(Q) in magnitude; a tile where that bound passes INT64_MAX ORs 1 into
// *overflow and writes nothing.
//
// sm_100a has no native 64-bit shared-memory add: red/atom.shared.add.u64 and atomicAdd all lower to a compare-and-
// store spin loop (ATOMS.CAST.SPIN.64).  The 64-bit add is instead two native 32-bit ones on the halves of the
// little-endian word: the low half's add returns the old value, so the thread whose add wraps it carries the 1 into
// the high half itself.  Every wrap is carried exactly once, so the word ends as the exact sum mod 2^64.
__device__ __forceinline__ void shared_add_u64(uint32_t addr, unsigned long long v) {
    const uint32_t lo = (uint32_t)v;
    uint32_t old;
    asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(addr), "r"(lo) : "memory");
    const uint32_t hi = (uint32_t)(v >> 32) + (old > ~lo ? 1u : 0u);   // old + lo wrapped past 2^32
    if (hi != 0) asm volatile("red.shared.add.u32 [%0], %1;" :: "r"(addr + 4u), "r"(hi) : "memory");
}

// Store len int64 sums of the shared tile to dst (8-byte aligned) as fp64(sum) * 2^-32, with coalesced 16-byte
// streaming stores: one leading position reaches a 16-byte boundary, one may trail.
__device__ __forceinline__ void clv_store_q32_f64(const long long *stage, double *__restrict__ dst, int len, int tid) {
    const int head = min((int)((reinterpret_cast<uintptr_t>(dst) >> 3) & 1u), len);
    const int npair = (len - head) >> 1, rest = len - head - 2 * npair;
    for (int p = tid; p < npair; p += kClvThreads) {
        const int i = head + 2 * p;
        const double a = (double)stage[i] * 0x1p-32, b = (double)stage[i + 1] * 0x1p-32;
        asm volatile("st.global.L1::no_allocate.v2.f64 [%0], {%1,%2};" :: "l"(dst + i), "d"(a), "d"(b) : "memory");
    }
    if (tid < head + rest) {
        const int p = tid < head ? tid : len - 1;
        dst[p] = (double)stage[p] * 0x1p-32;
    }
}

template <bool MIDPOINT>
__global__ void __launch_bounds__(kClvThreads)
gc_depth_tile_kernel(const int32_t *__restrict__ frag_start, const int32_t *__restrict__ frag_stop,
                     const uint8_t *__restrict__ frag_mapq, const uint64_t *__restrict__ seq64,
                     const uint32_t *__restrict__ nmask, int64_t contig_len,
                     const int32_t *__restrict__ tile_p0, const int32_t *__restrict__ tile_len,
                     const int64_t *__restrict__ tile_out_off, const int64_t *__restrict__ ranges,
                     const long long *__restrict__ weights, long long max_weight, int min_len, int max_len,
                     int min_mapq, int *__restrict__ overflow, double *__restrict__ out) {
    __shared__ __align__(16) long long D[kClvCap];   // difference array (midpoint: the sums themselves)
    __shared__ long long warp_tot[kClvThreads / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t tile = blockIdx.x;
    const int p0 = tile_p0[tile], len = tile_len[tile];
    const int64_t lo = ranges[2 * tile], hi = ranges[2 * tile + 1];
    if (max_weight > 0 && hi - lo > INT64_MAX / max_weight) {   // the bound on every partial sum
        if (tid == 0) atomicOr(overflow, 1);
        return;
    }
    for (int i = tid; i < kClvCap / 2; i += kClvThreads) reinterpret_cast<longlong2 *>(D)[i] = make_longlong2(0, 0);
    __syncthreads();
    const uint32_t d_addr = smem_addr_once(D);
    const unsigned len_span = (unsigned)(max_len - min_len);
    const int64_t row = (int64_t)max_len + 1;
    auto visit = [&](int fs, int fe, int q, int, int) {
        const int L = fe - fs;                                   // the sentinel (L = -1) fails the length test
        if (!(((unsigned)(L - min_len) <= len_span) & (q >= min_mapq))) return;
        const int s_idx = fs - p0, e_idx = fe - p0;
        const int m_idx = s_idx + (L >> 1);                      // (start + stop) // 2 - p0 without int32 overflow
        if (MIDPOINT ? (m_idx < 0 || m_idx >= len) : (e_idx <= 0 || s_idx >= len)) return;
        if (fs < 0 || (int64_t)fe > contig_len) return;          // placement undefined: weight 0
        const GcWalk gw = gc_walk(seq64, nmask, fs, fe);
        if (gw.has_n) return;
        const long long w = __ldg(weights + (int64_t)(L - min_len) * row + gw.g);
        if (w == 0) return;
        if constexpr (MIDPOINT) {
            shared_add_u64(d_addr + 8u * (unsigned)m_idx, (unsigned long long)w);
        } else {
            shared_add_u64(d_addr + 8u * (unsigned)max(s_idx, 0), (unsigned long long)w);
            if (e_idx < len) shared_add_u64(d_addr + 8u * (unsigned)e_idx, (unsigned long long)-w);
        }
    };
    stream_fragments<kClvThreads, 2>(FragCols{frag_start, frag_stop, frag_mapq, nullptr}, lo, hi, tid, visit);
    __syncthreads();
    if constexpr (!MIDPOINT) {
        // the block prefix scan of clv_tile_body in int64: kClvPer contiguous positions per thread, rewritten in place
        long long d[kClvPer];
        const int base = tid * kClvPer;
#pragma unroll
        for (int j = 0; j < kClvPer / 2; ++j) {
            const longlong2 v = *reinterpret_cast<const longlong2 *>(&D[base + 2 * j]);
            d[2 * j] = v.x; d[2 * j + 1] = v.y;
        }
#pragma unroll
        for (int j = 1; j < kClvPer; ++j) d[j] += d[j - 1];
        long long t = d[kClvPer - 1];
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const long long n = __shfl_up_sync(0xffffffffu, t, off);
            if (lane >= off) t += n;
        }
        if (lane == 31) warp_tot[warp] = t;
        __syncthreads();
        long long offset = t - d[kClvPer - 1];
#pragma unroll
        for (int w = 0; w < kClvThreads / 32; ++w) offset += (w < warp) ? warp_tot[w] : 0;
#pragma unroll
        for (int j = 0; j < kClvPer / 2; ++j)
            *reinterpret_cast<longlong2 *>(&D[base + 2 * j]) = make_longlong2(d[2 * j] + offset, d[2 * j + 1] + offset);
        __syncthreads();
    }
    clv_store_q32_f64(D, out + tile_out_off[tile], len, tid);
}

}  // namespace ftk

using namespace ftk;

// Argument checks of the cleavage and depth entry points, then the tile-range prepass: a fragment covering a tile
// position has stop > p0 (=> start > p0 - max_frag_len) and start < p0 + len; so has a fragment whose midpoint
// lies in the tile.
static int clv_tile_ranges(const int32_t *frag_start, const int32_t *frag_stop, int64_t n_frag, int32_t max_frag_len,
                           const int32_t *tile_p0, const int32_t *tile_len, const int32_t *tile_ivl_lo,
                           const int32_t *tile_ivl_hi, const int64_t *tile_out_off, int64_t n_tiles,
                           int64_t *scratch, const void *out, cudaStream_t stream) {
    if (n_frag < 0 || n_tiles < 0) return FTK_E_INVALID;
    if (!tile_p0 || !tile_len || !tile_ivl_lo || !tile_ivl_hi || !tile_out_off || !scratch || !out) return FTK_E_INVALID;
    if (n_frag > 0 && (!frag_start || !frag_stop)) return FTK_E_INVALID;
    if (n_tiles > INT32_MAX / 2) return FTK_E_RANGE;
    return launch_candidate_ranges(frag_start, n_frag, tile_p0, tile_len, true, n_tiles, max_frag_len < 0 ? 0 : max_frag_len,
                                   0, scratch, stream);
}

extern "C" int ftk_cleavage_tiles_f64(const int32_t *frag_start, const int32_t *frag_stop,
                                      const uint8_t *frag_mapq, const uint8_t *frag_strand,
                                      int64_t n_frag, int32_t max_frag_len,
                                      const int32_t *tile_p0, const int32_t *tile_len,
                                      const int32_t *tile_ivl_lo, const int32_t *tile_ivl_hi,
                                      const int64_t *tile_out_off, int64_t n_tiles,
                                      int32_t min_len, int32_t max_len, int32_t min_mapq,
                                      int64_t *scratch, double *out, ftk_stream_t stream_) {
    if (n_tiles == 0) return FTK_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const int rc = clv_tile_ranges(frag_start, frag_stop, n_frag, max_frag_len, tile_p0, tile_len, tile_ivl_lo,
                                   tile_ivl_hi, tile_out_off, n_tiles, scratch, out, stream);
    if (rc != FTK_OK) return rc;
    cleavage_tile_kernel<<<(unsigned)n_tiles, kClvThreads, 0, stream>>>(
        frag_start, frag_stop, frag_mapq, frag_strand, tile_p0, tile_len, tile_ivl_lo, tile_ivl_hi, tile_out_off,
        scratch, min_len, max_len, min_mapq, out);
    FTK_CHECK_LAUNCH("cleavage_tile_kernel");
    return FTK_OK;
}

extern "C" int ftk_depth_tiles_i32(const int32_t *frag_start, const int32_t *frag_stop, const uint8_t *frag_mapq,
                                   int64_t n_frag, int32_t max_frag_len,
                                   const int32_t *tile_p0, const int32_t *tile_len,
                                   const int32_t *tile_ivl_lo, const int32_t *tile_ivl_hi,
                                   const int64_t *tile_out_off, int64_t n_tiles,
                                   int32_t min_len, int32_t max_len, int32_t min_mapq, int32_t midpoint,
                                   int64_t *scratch, int32_t *out, ftk_stream_t stream_) {
    if (n_tiles == 0) return FTK_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const int rc = clv_tile_ranges(frag_start, frag_stop, n_frag, max_frag_len, tile_p0, tile_len, tile_ivl_lo,
                                   tile_ivl_hi, tile_out_off, n_tiles, scratch, out, stream);
    if (rc != FTK_OK) return rc;
    if (midpoint)
        depth_tile_kernel<true><<<(unsigned)n_tiles, kClvThreads, 0, stream>>>(
            frag_start, frag_stop, frag_mapq, tile_p0, tile_len, tile_out_off, scratch, min_len, max_len, min_mapq, out);
    else
        depth_tile_kernel<false><<<(unsigned)n_tiles, kClvThreads, 0, stream>>>(
            frag_start, frag_stop, frag_mapq, tile_p0, tile_len, tile_out_off, scratch, min_len, max_len, min_mapq, out);
    FTK_CHECK_LAUNCH("depth_tile_kernel");
    return FTK_OK;
}

extern "C" int ftk_gc_depth_tiles_f64(const int32_t *frag_start, const int32_t *frag_stop, const uint8_t *frag_mapq,
                                      int64_t n_frag, int32_t max_frag_len, const uint32_t *seq_words,
                                      const uint32_t *nmask_words, int64_t contig_len,
                                      const int32_t *tile_p0, const int32_t *tile_len,
                                      const int32_t *tile_ivl_lo, const int32_t *tile_ivl_hi,
                                      const int64_t *tile_out_off, int64_t n_tiles,
                                      int32_t min_len, int32_t max_len, int32_t min_mapq, int32_t midpoint,
                                      const int64_t *weights, int64_t max_weight, int64_t *scratch,
                                      int32_t *overflow, double *out, ftk_stream_t stream_) {
    if (n_tiles == 0) return FTK_OK;
    if (!seq_words || !nmask_words || !weights || !overflow || contig_len < 0 || min_len < 1 || max_len < min_len ||
        max_weight < 0)
        return FTK_E_INVALID;
    if ((reinterpret_cast<uintptr_t>(seq_words) & 7) != 0 || (reinterpret_cast<uintptr_t>(out) & 7) != 0)
        return FTK_E_INVALID;   // 64-bit seq words, fp64 stores
    if (max_len > FTK_GC_MAX_LENGTH || contig_len > INT32_MAX || max_weight >= FTK_GC_DEPTH_MAX_WEIGHT)
        return FTK_E_RANGE;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    // a passing fragment is at most max_len long: the candidate search reaches back no further
    const int rc = clv_tile_ranges(frag_start, frag_stop, n_frag, max_frag_len < max_len ? max_frag_len : max_len,
                                   tile_p0, tile_len, tile_ivl_lo, tile_ivl_hi, tile_out_off, n_tiles, scratch, out,
                                   stream);
    if (rc != FTK_OK) return rc;
    const auto *seq64 = reinterpret_cast<const uint64_t *>(seq_words);
    const auto *w = reinterpret_cast<const long long *>(weights);
    if (midpoint)
        gc_depth_tile_kernel<true><<<(unsigned)n_tiles, kClvThreads, 0, stream>>>(
            frag_start, frag_stop, frag_mapq, seq64, nmask_words, contig_len, tile_p0, tile_len, tile_out_off, scratch,
            w, max_weight, min_len, max_len, min_mapq, overflow, out);
    else
        gc_depth_tile_kernel<false><<<(unsigned)n_tiles, kClvThreads, 0, stream>>>(
            frag_start, frag_stop, frag_mapq, seq64, nmask_words, contig_len, tile_p0, tile_len, tile_out_off, scratch,
            w, max_weight, min_len, max_len, min_mapq, overflow, out);
    FTK_CHECK_LAUNCH("gc_depth_tile_kernel");
    return FTK_OK;
}
