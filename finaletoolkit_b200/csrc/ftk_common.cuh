// Shared helpers for the sm_100a kernels of libftk_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "ftk_b200.h"

namespace ftk {

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs

// Record-and-translate a CUDA error; implemented in ftk_api.cu.
int cuda_fail(cudaError_t e, const char *what);

#define FTK_CUDA_TRY(expr)                                      \
    do {                                                        \
        cudaError_t _e = (expr);                                \
        if (_e != cudaSuccess) return ::ftk::cuda_fail(_e, #expr); \
    } while (0)

#define FTK_CHECK_LAUNCH(name)                                   \
    do {                                                         \
        cudaError_t _e = cudaGetLastError();                     \
        if (_e != cudaSuccess) return ::ftk::cuda_fail(_e, name); \
    } while (0)

// Per-device tables (SM counts, shared-memory opt-ins) hold this many devices.
constexpr int kMaxDevices = 64;

// The calling thread's current CUDA device: the one a launch runs on.
inline int current_device(int *dev) {
    FTK_CUDA_TRY(cudaGetDevice(dev));
    return (*dev < 0 || *dev >= kMaxDevices) ? FTK_E_RANGE : FTK_OK;
}

// Streaming (read-once) global loads: keep them out of L1.
__device__ __forceinline__ int ld_stream(const int32_t *p) {
    int v;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ int4 ld_stream4(const int4 *p) {
    int4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ unsigned ld_stream_u8(const uint8_t *p) {
    unsigned v;
    asm volatile("ld.global.nc.L1::no_allocate.u8 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_stream4(int4 *p, const int4 &v) {
    asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// Shared-memory atomics through an explicit 32-bit shared-window address.  For atomicAdd(&smem[i], v) on
// a static __shared__ array nvcc (12.9, sm_100a) re-derives the array's window address next to every
// atomic in an unrolled loop (S2R SR_CgaCtaId + LEA per atomic); computing it once, hiding it behind an
// opaque move and issuing red.shared on it keeps the hot loops free of special-register reads.
__device__ __forceinline__ uint32_t smem_addr_once(const void *p) {
    const uint32_t a = static_cast<uint32_t>(__cvta_generic_to_shared(p));
    uint32_t r;
    asm volatile("mov.b32 %0, %1;" : "=r"(r) : "r"(a));
    return r;
}
__device__ __forceinline__ void red_shared_add(uint32_t addr, int v) {
    asm volatile("red.shared.add.s32 [%0], %1;" :: "r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void red_shared_inc(uint32_t addr) {
    asm volatile("red.shared.add.u32 [%0], 1;" :: "r"(addr) : "memory");
}
__device__ __forceinline__ void red_shared_min(uint32_t addr, int v) {
    asm volatile("red.shared.min.s32 [%0], %1;" :: "r"(addr), "r"(v) : "memory");
}

// first index i in [0, n) with a[i] >= key (a ascending); n if none
__device__ __forceinline__ int64_t lower_bound(const int32_t *__restrict__ a, int64_t n, int64_t key) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        int64_t mid = lo + ((hi - lo) >> 1);
        if ((int64_t)__ldg(a + mid) < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// The reference's fragment predicate (utils/_frag_generator.py:117-123,
// io/alignment.py:291): mapq >= q, min <= L <= max (FTK_NONE = unbounded).
__device__ __forceinline__ bool frag_len_ok(int len, int min_len, int max_len) {
    return (min_len == FTK_NONE || len >= min_len) && (max_len == FTK_NONE || len <= max_len);
}

// Candidate fragment range of every unit k (an interval or a tile) in the start-sorted column, a superset of
// the fragments that can matter to it, written as ranges[2k], ranges[2k+1]:
//   lo:  lo[k] == FTK_NONE ? 0 : lower_bound(frag_start, lo[k] - reach_lo)
//   hi:  hi_or_len[k] == FTK_NONE ? n_frag : lower_bound(frag_start, end + reach_hi),
//        end = hi_is_len ? lo[k] + hi_or_len[k] : hi_or_len[k]   (int64 arithmetic)
// Launches candidate_ranges_kernel, which also zeroes the optional accumulators zero_a / zero_b on the way
// (the fused WPS step thereby stays two launches).  Implemented in ftk_api.cu.
int launch_candidate_ranges(const int32_t *frag_start, int64_t n_frag,
                            const int32_t *lo, const int32_t *hi_or_len, bool hi_is_len, int64_t n,
                            int64_t reach_lo, int64_t reach_hi, int64_t *ranges, cudaStream_t stream,
                            unsigned long long *zero_a = nullptr, int64_t n_zero_a = 0,
                            unsigned long long *zero_b = nullptr, int64_t n_zero_b = 0);

// [lo, hi) of slice `split` of `splits` of a unit's candidate range: contiguous slices of a multiple of 4
// fragments (the last may be shorter; slices past the end of the range are empty, hi <= lo).
__device__ __forceinline__ void slice_of(const int64_t *__restrict__ ranges, int64_t unit, int split, int splits,
                                         int64_t &lo, int64_t &hi) {
    const int64_t lo_all = __ldg(ranges + 2 * unit), hi_all = __ldg(ranges + 2 * unit + 1);
    int64_t chunk = (hi_all - lo_all + splits - 1) / splits;
    chunk = (chunk + 3) & ~(int64_t)3;
    lo = lo_all + (int64_t)split * chunk;
    hi = min(hi_all, lo + chunk);
}

// Fragment columns of one contig; a missing mapq column reads as 255, a missing strand column as 1.
struct FragCols {
    const int32_t *start, *stop;
    const uint8_t *mapq, *strand;
};

// Streams fragments [lo, hi) to visit(start, stop, mapq, strand, index): thread t of a group of STRIDE
// threads takes vectors t, t + STRIDE, ... of 4 fragments, read with 128-bit streaming loads from lo widened
// left to a 16-byte boundary, UNROLL vectors in flight; the (at most 3) fragments past the last vector go
// through a scalar tail.  Lanes outside [lo, hi) - the widened head and the padding of the last batch -
// reach visit as the sentinel fragment (start 0, stop -1, mapq 0, strand 1): visit must reject a fragment of
// negative length.  Indices are int32 (the slice lies below 2^31 fragments).
template <int STRIDE, int UNROLL, class Visit>
__device__ __forceinline__ void stream_fragments(const FragCols &c, int64_t lo, int64_t hi, int t, Visit &&visit) {
    const int64_t lo_al = lo & ~(int64_t)3;
    const int skip = (int)(lo - lo_al);
    const int cnt = (hi > lo) ? (int)(hi - lo_al) : 0;
    const int nvec = cnt >> 2;
    const int base = (int)lo_al;
    const int4 *__restrict__ vs = reinterpret_cast<const int4 *>(c.start + lo_al);
    const int4 *__restrict__ ve = reinterpret_cast<const int4 *>(c.stop + lo_al);
    const uchar4 *__restrict__ vq = reinterpret_cast<const uchar4 *>(c.mapq ? c.mapq + lo_al : nullptr);
    const uchar4 *__restrict__ vd = reinterpret_cast<const uchar4 *>(c.strand ? c.strand + lo_al : nullptr);
    for (int v0 = t; v0 < nvec; v0 += UNROLL * STRIDE) {
        int4 s4[UNROLL], e4[UNROLL];
        uchar4 q4[UNROLL], d4[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const int v = v0 + u * STRIDE;
            if (v < nvec) {
                s4[u] = __ldcs(vs + v); e4[u] = __ldcs(ve + v);
                q4[u] = vq ? __ldcs(vq + v) : make_uchar4(255, 255, 255, 255);
                d4[u] = vd ? __ldcs(vd + v) : make_uchar4(1, 1, 1, 1);
            } else {
                s4[u] = make_int4(0, 0, 0, 0); e4[u] = make_int4(-1, -1, -1, -1);
                q4[u] = make_uchar4(0, 0, 0, 0); d4[u] = make_uchar4(1, 1, 1, 1);
            }
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const int i = base + 4 * (v0 + u * STRIDE);
            const bool head = u == 0 && v0 == 0;   // thread 0's first vector holds the widened head
            const bool mx = head && skip > 0, my = head && skip > 1, mz = head && skip > 2;
            visit(mx ? 0 : s4[u].x, mx ? -1 : e4[u].x, mx ? 0 : (int)q4[u].x, mx ? 1 : (int)d4[u].x, i);
            visit(my ? 0 : s4[u].y, my ? -1 : e4[u].y, my ? 0 : (int)q4[u].y, my ? 1 : (int)d4[u].y, i + 1);
            visit(mz ? 0 : s4[u].z, mz ? -1 : e4[u].z, mz ? 0 : (int)q4[u].z, mz ? 1 : (int)d4[u].z, i + 2);
            visit(s4[u].w, e4[u].w, (int)q4[u].w, (int)d4[u].w, i + 3);
        }
    }
    const int i = nvec * 4 + t;   // the tail (and the head too, when the slice is shorter than a vector)
    if (i < cnt && i >= skip)
        visit(__ldcs(c.start + lo_al + i), __ldcs(c.stop + lo_al + i), c.mapq ? (int)__ldcs(c.mapq + lo_al + i) : 255,
              c.strand ? (int)__ldcs(c.strand + lo_al + i) : 1, base + i);
}

}  // namespace ftk
