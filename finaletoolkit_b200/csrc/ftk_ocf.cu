// Orientation-aware fragment end profiles (OCF, Sun et al. 2019): upstream- and downstream-end offset counts
// around the sites of several site sets, summed over each set's sites.
//
// For every site (centre c, optionally flipped) of set k and every passing fragment [s, e) (mapq >= min_mapq,
// L = e - s >= 1, min_len <= L <= max_len) the upstream end offset is x_U = s - c and the downstream one
// x_D = (e - 1) - c (flipped: x_U = c - (e - 1), x_D = c - s); each end with |x| <= flank adds 1 to its row:
//   out[(k * 2 + 0) * (2 * flank + 1) + x_U + flank] += 1,  out[(k * 2 + 1) * (2 * flank + 1) + x_D + flank] += 1
//
// Work split: one WARP per (site, slice) unit streams the unit's slice of the candidate range with 128-bit loads
// (vplot's layout), but the units are dealt to CTAs by a host table: CTA b takes units [cta_bounds[b],
// cta_bounds[b + 1]), all of one set (the host sorts the sites by set).  Every event of a set lands in the same
// 2 (2 flank + 1) cells, so the CTA counts in shared memory (u32, red.shared.add.u32 = ATOMS.POPC.INC.32; a
// 64-bit shared atomicAdd compiles to a CAS loop) and adds its nonzero cells to `out` with 64-bit global REDs
// at the end.  One candidate fragment adds at most 1 to any cell, so a CTA flushes (and zeroes its counters)
// before the candidates it has taken since its last flush could pass `flush_every` (<= 2^32 - 1).
// Roofline: HBM, 9 B per candidate fragment (start, stop, mapq) - or the shared-memory atomic rate when most
// candidates count (DESIGN.md 4.13).
#include "ftk_common.cuh"

namespace ftk {

constexpr int kOcfThreads = 256;
constexpr int kOcfWarps = kOcfThreads / 32;
constexpr int kOcfUnroll = 4;
constexpr int kOcfMaxSmem = 2 * (2 * FTK_OCF_MAX_FLANK + 1) * 4;

__device__ __forceinline__ void red_global_add_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("red.global.add.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}

// Adds the CTA's nonzero counters to its set's rows of `out` and zeroes them; called by every thread.
__device__ __forceinline__ void ocf_flush(uint32_t *cnt, int cells, unsigned long long *out) {
    __syncthreads();
    for (int i = threadIdx.x; i < cells; i += kOcfThreads) {
        const uint32_t v = cnt[i];
        if (v) {
            red_global_add_u64(out + i, v);
            cnt[i] = 0;
        }
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kOcfThreads)
ocf_kernel(const int32_t *__restrict__ frag_start, const int32_t *__restrict__ frag_stop,
           const uint8_t *__restrict__ frag_mapq, const int32_t *__restrict__ win_lo,
           const uint8_t *__restrict__ site_flip, const int32_t *__restrict__ site_set,
           const int64_t *__restrict__ ranges, const int32_t *__restrict__ cta_bounds, int flank, int len_lo,
           int len_hi, int min_mapq, int splits, int n_units, int n_sets, int64_t flush_every,
           unsigned long long *__restrict__ out) {
    extern __shared__ uint32_t cnt[];                         // [2][2 flank + 1]: the U row, then the D row
    __shared__ int64_t round_cand[2][kOcfWarps];               // candidates per warp, double-buffered by round
    const int u0 = max(__ldg(cta_bounds + blockIdx.x), 0);
    const int u1 = min(__ldg(cta_bounds + blockIdx.x + 1), n_units);
    if (u0 >= u1) return;
    const int set = __ldg(site_set + u0 / splits);
    if (set < 0 || set >= n_sets) return;
    const int row = 2 * flank + 1;
    const int cells = 2 * row;
    for (int i = threadIdx.x; i < cells; i += kOcfThreads) cnt[i] = 0;
    out += (int64_t)set * cells;
    const uint32_t base = smem_addr_once(cnt);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned len_span = (unsigned)(len_hi - len_lo);   // len_lo >= 1: the sentinel (L = -1) fails
    const unsigned width = 2u * (unsigned)flank;              // x + flank in [0, width]

    int64_t since = 0;   // candidates taken since the last flush (the same in every thread)
    int parity = 0;
    __syncthreads();
    for (int b = u0; b < u1; b += kOcfWarps, parity ^= 1) {
        const int unit = b + warp;
        int64_t lo = 0, hi = 0;
        int c = 0;
        bool flip = false;
        if (unit < u1) {
            const int site = unit / splits;
            slice_of(ranges, site, unit % splits, splits, lo, hi);
            c = __ldg(win_lo + site) + flank;                 // the window is [c - flank, c + flank + 1)
            flip = __ldg(site_flip + site) != 0;
        }
        if (lane == 0) round_cand[parity][warp] = hi > lo ? hi - lo : 0;
        __syncthreads();
        int64_t n = 0;
#pragma unroll
        for (int w = 0; w < kOcfWarps; ++w) n += round_cand[parity][w];
        if (since > 0 && since + n > flush_every) {
            ocf_flush(cnt, cells, out);
            since = 0;
        }
        auto visit = [&](int fs, int fe, int q, int, int) {
            const int L = fe - fs;
            const bool ok = ((unsigned)(L - len_lo) <= len_span) & (q >= min_mapq);
            const int64_t xu = flip ? (int64_t)c - (fe - 1) : (int64_t)fs - c;
            const int64_t xd = flip ? (int64_t)c - fs : (int64_t)(fe - 1) - c;
            if (ok & ((uint64_t)(xu + flank) <= width)) red_shared_inc(base + 4u * (uint32_t)(xu + flank));
            if (ok & ((uint64_t)(xd + flank) <= width)) red_shared_inc(base + 4u * (uint32_t)(row + xd + flank));
        };
        const FragCols cols{frag_start, frag_stop, frag_mapq, nullptr};
        if (n <= flush_every) {
            stream_fragments<32, kOcfUnroll>(cols, lo, hi, lane, visit);
            since += n;
        } else {   // a round larger than the threshold: one warp at a time, a flush after each
            for (int w = 0; w < kOcfWarps; ++w) {
                if (w == warp) stream_fragments<32, kOcfUnroll>(cols, lo, hi, lane, visit);
                ocf_flush(cnt, cells, out);
            }
            since = 0;
        }
    }
    ocf_flush(cnt, cells, out);
}

}  // namespace ftk

using namespace ftk;

extern "C" int ftk_ocf_u64(const int32_t *frag_start, const int32_t *frag_stop, const uint8_t *frag_mapq,
                           int64_t n_frag, int32_t max_frag_len, const int32_t *win_lo, const int32_t *win_hi,
                           const uint8_t *site_flip, const int32_t *site_set, int64_t n_sites, int32_t n_sets,
                           int32_t flank, int32_t min_len, int32_t max_len, int32_t min_mapq, int32_t splits,
                           const int32_t *cta_bounds, int32_t n_cta, int64_t flush_every, int64_t *scratch,
                           uint64_t *out, ftk_stream_t stream_) {
    if (n_sites == 0) return FTK_OK;
    if (n_frag < 0 || n_sites < 0 || n_sets < 1 || n_cta < 1 || flank < 0 || splits < 1 || flush_every < 1)
        return FTK_E_INVALID;
    if ((min_len < 0 && min_len != FTK_NONE) || (max_len < 0 && max_len != FTK_NONE) ||
        (min_len != FTK_NONE && max_len != FTK_NONE && max_len < min_len))
        return FTK_E_INVALID;
    if (!win_lo || !win_hi || !site_flip || !site_set || !cta_bounds || !scratch || !out) return FTK_E_INVALID;
    if (n_frag > 0 && (!frag_start || !frag_stop)) return FTK_E_INVALID;
    if (flank > FTK_OCF_MAX_FLANK || flush_every > (int64_t)UINT32_MAX) return FTK_E_RANGE;
    if ((int64_t)n_sets * 2 * (2 * (int64_t)flank + 1) > FTK_OCF_MAX_CELLS) return FTK_E_RANGE;
    if (n_sites > INT32_MAX / 2 || n_sites * (int64_t)splits > INT32_MAX) return FTK_E_RANGE;
    if (n_frag == 0) return FTK_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const int frag_max = max_frag_len < 0 ? 0 : max_frag_len;
    const int len_lo = min_len == FTK_NONE || min_len < 1 ? 1 : min_len;          // L >= 1: a fragment has ends
    const int len_hi = max_len == FTK_NONE || max_len > frag_max ? frag_max : max_len;
    if (len_hi < len_lo) return FTK_OK;                                           // no fragment can pass
    // a right end e - 1 >= c - flank needs s >= c - flank - (L - 1) >= c - flank - len_hi; a left end s <= c + flank
    const int rc = launch_candidate_ranges(frag_start, n_frag, win_lo, win_hi, false, n_sites, len_hi, 0, scratch,
                                           stream);
    if (rc != FTK_OK) return rc;
    int dev = 0;
    const int drc = current_device(&dev);
    if (drc != FTK_OK) return drc;
    // the dynamic shared-memory limit belongs to (kernel, device): raise it on every device this thread launches on
    static thread_local bool smem_opted_in[kMaxDevices] = {};
    if (!smem_opted_in[dev]) {
        FTK_CUDA_TRY(cudaFuncSetAttribute(ocf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kOcfMaxSmem));
        smem_opted_in[dev] = true;
    }
    const size_t smem = (size_t)2 * (2 * flank + 1) * sizeof(uint32_t);
    ocf_kernel<<<(unsigned)n_cta, kOcfThreads, smem, stream>>>(
        frag_start, frag_stop, frag_mapq, win_lo, site_flip, site_set, scratch, cta_bounds, flank, len_lo, len_hi,
        min_mapq, splits, (int)(n_sites * splits), n_sets, flush_every, reinterpret_cast<unsigned long long *>(out));
    FTK_CHECK_LAUNCH("ocf_kernel");
    return FTK_OK;
}
