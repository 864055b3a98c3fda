// Per-interval fragment counts, fragment-length histograms and raw lengths.
//
// Replaces the reference's generator loops over the fragment stream:
//   coverage      frag/_coverage.py:117-130   `for _ in frags: coverage += 1`
//   length dict   frag/_frag_length.py:147-153 `value_counts[len] += 1`
//   raw lengths   frag/_frag_length.py:303     list of stop-start in stream order
// with the stream's predicate folded into the kernels:
//   io/alignment.py:270-302       tabix overlap rows, mapq >= q
//   utils/_frag_generator.py:21-55, 117-123  inclusive length filter + policy
//
// Each (interval, split) pair is one CTA streaming a contiguous slice of the
// start-sorted fragment columns (coalesced loads, several batches in flight),
// counting in registers and binning lengths into a shared-memory-privatised
// histogram that is flushed once with 64-bit global atomics.
// Roofline: HBM, 9 B per candidate fragment (start, stop, mapq).
#include "ftk_common.cuh"

namespace ftk {

constexpr int kHistThreads = 256;
constexpr int kHistSmemBins = 2048;  // lengths below this are privatised in smem
constexpr int kHistUnroll = 4;

struct Pred {
    int policy, min_len, max_len, min_mapq;
};

// Stream membership of one fragment for region [S, E) (FTK_NONE = unbounded), with the
// None handling and the length window folded into per-CTA constants:
//   tabix fetch(contig, S, E): rec.stop > start (None -> 0) and rec.start < stop
//   length filter inclusive; midpoint policy mid in [S, E); "any" = the overlap test itself
// The upper bound is kept inclusive (e_last = E - 1) so that E = None admits a start or midpoint of 2^31 - 1.
struct Stream {
    int len_lo; unsigned len_span; bool len_any;
    int min_mapq; int s_over; int e_last; int s_mid; bool midpoint;
    __device__ __forceinline__ Stream(int S, int E, const Pred &p) {
        len_lo = (p.min_len == FTK_NONE || p.min_len < 0) ? 0 : p.min_len;
        const int hi = (p.max_len == FTK_NONE) ? INT32_MAX : p.max_len;
        len_any = hi >= len_lo;
        len_span = len_any ? (unsigned)(hi - len_lo) : 0u;
        min_mapq = p.min_mapq;
        s_over = (S == FTK_NONE) ? 0 : S;
        s_mid = (S == FTK_NONE) ? INT32_MIN : S;
        e_last = (E == FTK_NONE) ? INT32_MAX : E - 1;   // E > FTK_NONE here: no wrap
        midpoint = p.policy == FTK_POLICY_MIDPOINT;
    }
    // Branch-free: every test is evaluated and AND-ed (predicate logic, no short-circuit branches).
    __device__ __forceinline__ bool operator()(int fs, int fe, int q) const {
        const int L = fe - fs;
        const int mid = fs + (L >> 1);
        const unsigned ok_len = (unsigned)((unsigned)(L - len_lo) <= len_span);
        const unsigned ok_q = (unsigned)(q >= min_mapq);
        const unsigned ok_over = (unsigned)(fe > s_over) & (unsigned)(fs <= e_last);
        const unsigned ok_mid = midpoint ? ((unsigned)(mid >= s_mid) & (unsigned)(mid <= e_last)) : 1u;
        return (ok_len & ok_q & ok_over & ok_mid & (unsigned)len_any) != 0u;
    }
};

__device__ __forceinline__ bool frag_in_stream(int fs, int fe, int q, int S, int E, const Pred &p) {
    return Stream(S, E, p)(fs, fe, q);
}

template <bool HIST>
__global__ void __launch_bounds__(kHistThreads)
interval_hist_kernel(const int32_t *__restrict__ frag_start, const int32_t *__restrict__ frag_stop,
                     const uint8_t *__restrict__ frag_mapq,
                     const int32_t *__restrict__ ivl_start, const int32_t *__restrict__ ivl_stop,
                     const int64_t *__restrict__ ranges, Pred pred, int n_bins, int pooled, int splits,
                     unsigned long long *__restrict__ counts, unsigned long long *__restrict__ hist,
                     int32_t *__restrict__ first_seen) {
    __shared__ int s_cnt[HIST ? kHistSmemBins : 1];
    __shared__ int s_first[HIST ? kHistSmemBins : 1];
    __shared__ unsigned long long s_red[kHistThreads / 32];

    const int tid = threadIdx.x;
    const int64_t ivl = blockIdx.x / splits;
    const int split = blockIdx.x % splits;
    const int64_t row = pooled ? 0 : ivl;
    const int S = ivl_start[ivl], E = ivl_stop[ivl];
    int64_t lo, hi;
    slice_of(ranges, ivl, split, splits, lo, hi);
    const bool want_first = HIST && (first_seen != nullptr);

    if (HIST) {
        for (int b = tid; b < kHistSmemBins; b += kHistThreads) { s_cnt[b] = 0; s_first[b] = INT32_MAX; }
        __syncthreads();
    }

    const Stream in_stream(S, E, pred);
    unsigned my_count32 = 0;  // a CTA slice never holds 2^32 fragments (n_frag <= INT32_MAX)
    const uint32_t cnt_addr = HIST ? smem_addr_once(s_cnt) : 0u, first_addr = HIST ? smem_addr_once(s_first) : 0u;
    auto visit = [&](int fs, int fe, int q, int, int idx) {
        if (!in_stream(fs, fe, q)) return;
        ++my_count32;
        if (HIST) {
            const int L = fe - fs;
            if (L < kHistSmemBins) {
                red_shared_inc(cnt_addr + 4u * (unsigned)L);
                if (want_first) red_shared_min(first_addr + 4u * (unsigned)L, idx);
            } else if (L < n_bins) {
                atomicAdd(&hist[row * n_bins + L], 1ull);
                if (want_first) atomicMin(&first_seen[row * n_bins + L], idx);
            }
        }
    };
    stream_fragments<kHistThreads, kHistUnroll>(FragCols{frag_start, frag_stop, frag_mapq, nullptr}, lo, hi, tid, visit);
    unsigned long long my_count = my_count32;

    // block reduction of the count -> one 64-bit atomic per CTA
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) my_count += __shfl_down_sync(0xffffffffu, my_count, off);
    if ((tid & 31) == 0) s_red[tid >> 5] = my_count;
    __syncthreads();
    if (tid == 0) {
        unsigned long long tot = 0;
#pragma unroll
        for (int w = 0; w < kHistThreads / 32; ++w) tot += s_red[w];
        if (tot) atomicAdd(&counts[row], tot);
    }
    if (HIST) {
        const int nb = min(n_bins, kHistSmemBins);
        for (int b = tid; b < nb; b += kHistThreads) {
            const int c = s_cnt[b];
            if (c) {
                atomicAdd(&hist[row * n_bins + b], (unsigned long long)c);
                if (want_first) atomicMin(&first_seen[row * n_bins + b], s_first[b]);
            }
        }
    }
}

// Counts (coverage): one WARP per (interval, split).  A 5-kb interval at 30x holds ~1600
// candidates - far too few to amortise a CTA's launch, barrier and reduction latency - so eight
// independent warps share a CTA, each streaming its own slice with 128-bit loads (kHistUnroll x 3
// in flight per lane) and finishing with a shuffle reduction + one atomic.  PHIST additionally
// bins the lengths of every counted fragment into ONE pooled histogram (row 0), privatised per
// CTA in shared memory: per-interval coverage and the length distribution of the union of the
// intervals in a single pass over the fragments.
template <bool PHIST>
__global__ void __launch_bounds__(kHistThreads, 4)
interval_count_warp_kernel(const int32_t *__restrict__ frag_start, const int32_t *__restrict__ frag_stop,
                           const uint8_t *__restrict__ frag_mapq,
                           const int32_t *__restrict__ ivl_start, const int32_t *__restrict__ ivl_stop,
                           const int64_t *__restrict__ ranges, Pred pred, int pooled_counts, int splits,
                           int64_t n_units, int n_bins, unsigned long long *__restrict__ counts,
                           unsigned long long *__restrict__ hist, int32_t *__restrict__ first_seen) {
    __shared__ int s_cnt[PHIST ? kHistSmemBins : 1];
    __shared__ int s_first[PHIST ? kHistSmemBins : 1];
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const bool want_first = PHIST && (first_seen != nullptr);
    if (PHIST) {
        for (int b = tid; b < kHistSmemBins; b += kHistThreads) { s_cnt[b] = 0; s_first[b] = INT32_MAX; }
        __syncthreads();
    }
    const int64_t unit = (int64_t)blockIdx.x * (kHistThreads / 32) + (tid >> 5);
    if (unit < n_units) {
        const int64_t ivl = unit / splits;
        const int split = (int)(unit % splits);
        const int S = __ldg(ivl_start + ivl), E = __ldg(ivl_stop + ivl);
        int64_t lo, hi;
        slice_of(ranges, ivl, split, splits, lo, hi);
        const Stream in_stream(S, E, pred);

        // Its own copy of the stream_fragments loop, with the head lanes masked by a flag instead of the
        // sentinel: at the 64-register cap every formulation of the shared loop tried (nvcc 12.9) spilled more.
        const int64_t lo_al = lo & ~(int64_t)3;
        const int skip = (int)(lo - lo_al);
        const int cnt = (hi > lo) ? (int)(hi - lo_al) : 0;
        const int nvec = cnt >> 2;
        const int base_idx = (int)lo_al;
        const int4 *__restrict__ vs = reinterpret_cast<const int4 *>(frag_start + lo_al);
        const int4 *__restrict__ ve = reinterpret_cast<const int4 *>(frag_stop + lo_al);
        const uchar4 *__restrict__ vq = reinterpret_cast<const uchar4 *>(frag_mapq ? frag_mapq + lo_al : nullptr);
        unsigned c = 0;
        const uint32_t cnt_addr = PHIST ? smem_addr_once(s_cnt) : 0u, first_addr = PHIST ? smem_addr_once(s_first) : 0u;
        auto visit = [&](int fs, int fe, int q, int idx, bool masked) {
            if (masked || !in_stream(fs, fe, q)) return;
            ++c;
            if (PHIST) {
                const int L = fe - fs;
                if (L < kHistSmemBins) {
                    red_shared_inc(cnt_addr + 4u * (unsigned)L);
                    if (want_first) red_shared_min(first_addr + 4u * (unsigned)L, idx);
                } else if (L < n_bins) {
                    atomicAdd(&hist[L], 1ull);
                    if (want_first) atomicMin(&first_seen[L], idx);
                }
            }
        };
        for (int v0 = lane; v0 < nvec; v0 += kHistUnroll * 32) {
            int4 s4[kHistUnroll], e4[kHistUnroll];
            uchar4 q4[kHistUnroll];
#pragma unroll
            for (int u = 0; u < kHistUnroll; ++u) {
                const int v = v0 + u * 32;
                if (v < nvec) {
                    s4[u] = __ldcs(vs + v);
                    e4[u] = __ldcs(ve + v);
                    q4[u] = vq ? __ldcs(vq + v) : make_uchar4(255, 255, 255, 255);
                } else {
                    s4[u] = make_int4(0, 0, 0, 0);
                    e4[u] = make_int4(-1, -1, -1, -1);  // L < 0: never in a stream
                    q4[u] = make_uchar4(0, 0, 0, 0);
                }
            }
#pragma unroll
            for (int u = 0; u < kHistUnroll; ++u) {
                const int v = v0 + u * 32;
                const bool head = (v == 0);  // the widened head: mask fragments left of lo
                const int i = base_idx + v * 4;
                visit(s4[u].x, e4[u].x, q4[u].x, i, head && skip > 0);
                visit(s4[u].y, e4[u].y, q4[u].y, i + 1, head && skip > 1);
                visit(s4[u].z, e4[u].z, q4[u].z, i + 2, head && skip > 2);
                visit(s4[u].w, e4[u].w, q4[u].w, i + 3, false);
            }
        }
        {   // tail: at most 3 fragments
            const int i = nvec * 4 + lane;
            if (i < cnt && i >= skip)
                visit(__ldcs(frag_start + lo_al + i), __ldcs(frag_stop + lo_al + i),
                      frag_mapq ? (int)__ldcs(frag_mapq + lo_al + i) : 255, base_idx + i, false);
        }
        c = __reduce_add_sync(0xffffffffu, c);
        if (lane == 0 && c) atomicAdd(&counts[pooled_counts ? 0 : ivl], (unsigned long long)c);
    }
    if (PHIST) {
        __syncthreads();
        const int nb = min(n_bins, kHistSmemBins);
        for (int b = tid; b < nb; b += kHistThreads) {
            const int v = s_cnt[b];
            if (v) {
                atomicAdd(&hist[b], (unsigned long long)v);
                if (want_first) atomicMin(&first_seen[b], s_first[b]);
            }
        }
    }
}

// ---- raw lengths in stream order (frag_length): count / scan / scatter
constexpr int kLenBlock = 1024;  // fragments per CTA

__global__ void one_range_kernel(const int32_t *__restrict__ fs, int64_t n, int S, int E, int halo,
                                 int64_t *__restrict__ r) {
    if (threadIdx.x == 0) r[0] = (S == FTK_NONE) ? 0 : lower_bound(fs, n, (int64_t)S - halo);
    if (threadIdx.x == 1) r[1] = (E == FTK_NONE) ? n : lower_bound(fs, n, (int64_t)E);
}

__global__ void __launch_bounds__(256)
lengths_count_kernel(const int32_t *__restrict__ frag_start, const int32_t *__restrict__ frag_stop,
                     const uint8_t *__restrict__ frag_mapq, const int64_t *__restrict__ range,
                     int S, int E, Pred pred, int32_t *__restrict__ block_counts) {
    __shared__ int s_red[8];
    const int64_t lo = range[0], hi = range[1];
    const int64_t base = lo + (int64_t)blockIdx.x * kLenBlock;
    int c = 0;
#pragma unroll
    for (int u = 0; u < kLenBlock / 256; ++u) {
        const int64_t i = base + u * 256 + threadIdx.x;
        if (i < hi) {
            const int q = frag_mapq ? (int)__ldcs(frag_mapq + i) : 255;
            c += frag_in_stream(__ldcs(frag_start + i), __ldcs(frag_stop + i), q, S, E, pred);
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) c += __shfl_down_sync(0xffffffffu, c, off);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < 8; ++w) t += s_red[w];
        block_counts[blockIdx.x] = t;
    }
}

// single-CTA exclusive scan of block counts (n_blocks <= a few million); writes total to *n_out
__global__ void __launch_bounds__(1024)
lengths_scan_kernel(const int32_t *__restrict__ block_counts, const int64_t *__restrict__ range,
                    int64_t *__restrict__ block_offsets, int64_t *__restrict__ n_out) {
    __shared__ long long s_warp[32];
    __shared__ long long s_carry;
    const int64_t n_blocks = (range[1] - range[0] + kLenBlock - 1) / kLenBlock;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t base = 0; base < n_blocks; base += 1024) {
        const int64_t i = base + threadIdx.x;
        long long v = (i < n_blocks) ? block_counts[i] : 0;
        long long t = v;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            long long n = __shfl_up_sync(0xffffffffu, t, off);
            if (lane >= off) t += n;
        }
        if (lane == 31) s_warp[warp] = t;
        __syncthreads();
        if (warp == 0) {
            long long w = s_warp[lane];
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                long long n = __shfl_up_sync(0xffffffffu, w, off);
                if (lane >= off) w += n;
            }
            s_warp[lane] = w;  // inclusive
        }
        __syncthreads();
        const long long warp_excl = warp ? s_warp[warp - 1] : 0;
        const long long carry = s_carry;
        if (i < n_blocks) block_offsets[i] = carry + warp_excl + t - v;
        __syncthreads();
        if (threadIdx.x == 0) s_carry = carry + s_warp[31];
        __syncthreads();
    }
    if (threadIdx.x == 0) *n_out = s_carry;
}

__global__ void __launch_bounds__(256)
lengths_scatter_kernel(const int32_t *__restrict__ frag_start, const int32_t *__restrict__ frag_stop,
                       const uint8_t *__restrict__ frag_mapq, const int64_t *__restrict__ range,
                       int S, int E, Pred pred, const int64_t *__restrict__ block_offsets,
                       int32_t *__restrict__ out) {
    __shared__ int s_warp[8];
    const int64_t lo = range[0], hi = range[1];
    const int64_t base = lo + (int64_t)blockIdx.x * kLenBlock;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int64_t off = block_offsets[blockIdx.x];
    // stream order = index order: thread t of pass u owns fragment base + u*256 + t
    for (int u = 0; u < kLenBlock / 256; ++u) {
        const int64_t i = base + u * 256 + threadIdx.x;
        int L = 0;
        bool pass = false;
        if (i < hi) {
            const int fs = __ldcs(frag_start + i), fe = __ldcs(frag_stop + i);
            const int q = frag_mapq ? (int)__ldcs(frag_mapq + i) : 255;
            pass = frag_in_stream(fs, fe, q, S, E, pred);
            L = fe - fs;
        }
        const unsigned m = __ballot_sync(0xffffffffu, pass);
        if (lane == 0) s_warp[warp] = __popc(m);
        __syncthreads();
        int before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) { const int c = s_warp[w]; before += (w < warp) ? c : 0; total += c; }
        if (pass) out[off + before + __popc(m & ((1u << lane) - 1))] = L;
        off += total;
        __syncthreads();
    }
}

}  // namespace ftk

using namespace ftk;

static int effective_halo(int policy, int max_frag_len, int max_len) {
    int m = max_frag_len;
    if (max_len != FTK_NONE && max_len < m) m = max_len;
    if (m < 0) m = 0;
    // midpoint: fs + (L>>1) >= S  =>  fs >= S - (maxL>>1);  any: fe > S  =>  fs > S - maxL
    return policy == FTK_POLICY_MIDPOINT ? (m >> 1) : m;
}

extern "C" int ftk_interval_hist_u64(const int32_t *frag_start, const int32_t *frag_stop,
                                     const uint8_t *frag_mapq, int64_t n_frag, int32_t max_frag_len,
                                     const int32_t *ivl_start, const int32_t *ivl_stop, int64_t n_ivl,
                                     int32_t policy, int32_t min_len, int32_t max_len, int32_t min_mapq,
                                     int32_t n_bins, int32_t pooled, int32_t splits,
                                     int64_t *scratch, uint64_t *counts, uint64_t *hist,
                                     int32_t *first_seen, ftk_stream_t stream_) {
    if (n_ivl == 0) return FTK_OK;
    if (n_frag < 0 || n_ivl < 0 || splits < 1 || n_bins < 0 || pooled < 0 || pooled > 2) return FTK_E_INVALID;
    if (policy != FTK_POLICY_MIDPOINT && policy != FTK_POLICY_ANY) return FTK_E_INVALID;
    if (!ivl_start || !ivl_stop || !scratch || !counts) return FTK_E_INVALID;
    if (n_frag > 0 && (!frag_start || !frag_stop)) return FTK_E_INVALID;
    if (n_bins > 0 && !hist) return FTK_E_INVALID;
    if (n_frag > INT32_MAX) return FTK_E_RANGE;  // first-seen indices are int32
    if (n_ivl * (int64_t)splits > INT32_MAX) return FTK_E_RANGE;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const int halo = effective_halo(policy, max_frag_len, max_len);
    const int rc = launch_candidate_ranges(frag_start, n_frag, ivl_start, ivl_stop, false, n_ivl, halo, 0, scratch, stream);
    if (rc != FTK_OK) return rc;
    Pred pred{policy, min_len, max_len, min_mapq};
    const unsigned grid = (unsigned)(n_ivl * splits);
    auto *c = reinterpret_cast<unsigned long long *>(counts);
    auto *h = reinterpret_cast<unsigned long long *>(hist);
    const int64_t n_units = n_ivl * (int64_t)splits;
    const int per_cta = kHistThreads / 32;
    const unsigned wgrid = (unsigned)((n_units + per_cta - 1) / per_cta);
    if (n_bins > 0 && pooled == FTK_POOL_HIST_ONLY)
        // per-interval counts + ONE pooled histogram in a single pass
        interval_count_warp_kernel<true><<<wgrid, kHistThreads, 0, stream>>>(
            frag_start, frag_stop, frag_mapq, ivl_start, ivl_stop, scratch, pred, 0, splits, n_units, n_bins, c, h, first_seen);
    else if (n_bins > 0)
        interval_hist_kernel<true><<<grid, kHistThreads, 0, stream>>>(
            frag_start, frag_stop, frag_mapq, ivl_start, ivl_stop, scratch, pred, n_bins, pooled, splits, c, h, first_seen);
    else
        interval_count_warp_kernel<false><<<wgrid, kHistThreads, 0, stream>>>(
            frag_start, frag_stop, frag_mapq, ivl_start, ivl_stop, scratch, pred, pooled, splits, n_units, 0, c, nullptr, nullptr);
    FTK_CHECK_LAUNCH("interval_hist_kernel");
    return FTK_OK;
}

extern "C" int ftk_frag_lengths_i32(const int32_t *frag_start, const int32_t *frag_stop,
                                    const uint8_t *frag_mapq, int64_t n_frag, int32_t max_frag_len,
                                    int32_t region_start, int32_t region_stop, int32_t policy,
                                    int32_t min_len, int32_t max_len, int32_t min_mapq,
                                    int64_t *scratch, int64_t scratch_len, int32_t *out,
                                    int64_t *n_out, ftk_stream_t stream_) {
    // scratch (int64 slots): [0..1] candidate range, [2 .. 2+nb) block offsets,
    // then nb int32 block counts packed two per slot.
    if (n_frag < 0 || !scratch || !out || !n_out) return FTK_E_INVALID;
    if (policy != FTK_POLICY_MIDPOINT && policy != FTK_POLICY_ANY) return FTK_E_INVALID;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const int64_t nb = (n_frag + kLenBlock - 1) / kLenBlock + 1;
    if (scratch_len < 2 + nb + (nb + 1) / 2) return FTK_E_INVALID;
    if (nb > INT32_MAX) return FTK_E_RANGE;
    if (n_frag == 0) {
        FTK_CUDA_TRY(cudaMemsetAsync(n_out, 0, sizeof(int64_t), stream));
        return FTK_OK;
    }
    if (!frag_start || !frag_stop) return FTK_E_INVALID;
    const int halo = effective_halo(policy, max_frag_len, max_len);
    int64_t *range = scratch;
    int64_t *block_offsets = scratch + 2;
    int32_t *block_counts = reinterpret_cast<int32_t *>(scratch + 2 + nb);
    Pred pred{policy, min_len, max_len, min_mapq};
    one_range_kernel<<<1, 32, 0, stream>>>(frag_start, n_frag, region_start, region_stop, halo, range);
    FTK_CHECK_LAUNCH("one_range_kernel");
    // The candidate range stays on the device (no host sync): the grids cover the
    // whole contig and CTAs beyond the range find nothing to do.
    const unsigned grid = (unsigned)(nb - 1);
    lengths_count_kernel<<<grid, 256, 0, stream>>>(frag_start, frag_stop, frag_mapq, range,
                                                   region_start, region_stop, pred, block_counts);
    FTK_CHECK_LAUNCH("lengths_count_kernel");
    lengths_scan_kernel<<<1, 1024, 0, stream>>>(block_counts, range, block_offsets, n_out);
    FTK_CHECK_LAUNCH("lengths_scan_kernel");
    lengths_scatter_kernel<<<grid, 256, 0, stream>>>(frag_start, frag_stop, frag_mapq, range,
                                                     region_start, region_stop, pred, block_offsets, out);
    FTK_CHECK_LAUNCH("lengths_scatter_kernel");
    return FTK_OK;
}
