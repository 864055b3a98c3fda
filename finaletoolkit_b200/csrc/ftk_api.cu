// ABI bookkeeping (version, error strings, last CUDA error, thread-local) and the candidate-range prepass
// shared by the interval and tile kernels.
#include <stdio.h>

#include "ftk_common.cuh"

namespace ftk {
static thread_local char g_last_cuda_error[512] = "";

int cuda_fail(cudaError_t e, const char *what) {
    snprintf(g_last_cuda_error, sizeof(g_last_cuda_error), "%s: %s (%s)", what,
             cudaGetErrorName(e), cudaGetErrorString(e));
    return FTK_E_CUDA;
}

constexpr int kRangeThreads = 128;

// One thread per bound; the upper levels of the search tree stay in L2, so this costs ~30 us per chr1-scale
// launch.  (A warp-cooperative 32-ary search - 6 dependent rounds instead of 27 - was measured in round 2 and
// lost, 64 us: every round touches 32 sectors per warp.)
__global__ void __launch_bounds__(kRangeThreads)
candidate_ranges_kernel(const int32_t *__restrict__ frag_start, int64_t n_frag,
                        const int32_t *__restrict__ lo, const int32_t *__restrict__ hi_or_len, bool hi_is_len,
                        int64_t n, int64_t reach_lo, int64_t reach_hi, int64_t *__restrict__ ranges,
                        unsigned long long *__restrict__ zero_a, int64_t n_zero_a,
                        unsigned long long *__restrict__ zero_b, int64_t n_zero_b) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t gthreads = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = t; i < n_zero_a; i += gthreads) zero_a[i] = 0ull;
    for (int64_t i = t; i < n_zero_b; i += gthreads) zero_b[i] = 0ull;
    if (t >= 2 * n) return;
    const int64_t k = t >> 1;
    const bool upper = (t & 1) != 0;
    // both bounds of a unit share a warp: pick the key per lane, then ONE search (two in divergent branches
    // would run back to back)
    const int32_t b = upper ? hi_or_len[k] : lo[k];
    const int64_t key = upper ? (hi_is_len ? (int64_t)lo[k] + b : (int64_t)b) + reach_hi : (int64_t)b - reach_lo;
    ranges[t] = (b == FTK_NONE) ? (upper ? n_frag : 0) : lower_bound(frag_start, n_frag, key);
}

int launch_candidate_ranges(const int32_t *frag_start, int64_t n_frag,
                            const int32_t *lo, const int32_t *hi_or_len, bool hi_is_len, int64_t n,
                            int64_t reach_lo, int64_t reach_hi, int64_t *ranges, cudaStream_t stream,
                            unsigned long long *zero_a, int64_t n_zero_a,
                            unsigned long long *zero_b, int64_t n_zero_b) {
    candidate_ranges_kernel<<<(unsigned)((2 * n + kRangeThreads - 1) / kRangeThreads), kRangeThreads, 0, stream>>>(
        frag_start, n_frag, lo, hi_or_len, hi_is_len, n, reach_lo, reach_hi, ranges, zero_a, n_zero_a, zero_b, n_zero_b);
    FTK_CHECK_LAUNCH("candidate_ranges_kernel");
    return FTK_OK;
}
}  // namespace ftk

extern "C" int ftk_abi_version(void) { return FTK_ABI_VERSION; }

extern "C" const char *ftk_last_cuda_error(void) { return ftk::g_last_cuda_error; }

extern "C" const char *ftk_error_string(int code) {
    switch (code) {
        case FTK_OK: return "ok";
        case FTK_E_INVALID: return "invalid argument";
        case FTK_E_CUDA: return "CUDA error (see ftk_last_cuda_error)";
        case FTK_E_RANGE: return "size or coordinate out of the supported range";
        case FTK_E_IO: return "file unreadable or not valid (b)gzip";
        default: return "unknown error";
    }
}
