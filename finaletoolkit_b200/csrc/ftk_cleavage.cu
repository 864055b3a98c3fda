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
#include "ftk_common.cuh"

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
