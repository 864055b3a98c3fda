// Periodicity spectra of back-to-back series (nucleosome repeat strength from WPS).
//
// For segment s (x[offsets[s] .. offsets[s + 1]), N values, mean mu) and every integer period P in
// [min_period, max_period]:
//   X(P) = sum_{n<N} (x[n] - mu) * exp(-2 pi i (n mod P) / P),   I(P) = |X(P)|^2 / N   (fp64)
// computed as X(P) = sum_{r<P} (F_P[r] - mu * c_r) * exp(-2 pi i r / P) from the folds
// F_P[r] = sum_{n = r mod P} x[n] (int64 for int32 input: exact; fp64 for fp64 input) and the residue counts c_r.
// An empty segment gives a row of NaN.
//
// One CTA per (segment, period group): kSpecWarps warps, one period each (group g holds periods g, g + G, ...,
// G = ceil(n_periods / kSpecWarps), so the groups are within one period of each other in size).  The CTA stages
// the segment through shared memory in chunks of kSpecChunk values, so segments of any length work.  Lane l of a
// warp owns residues r = l + 32 j; for each it walks the chunk's blocks of P positions (lanes read 32
// consecutive words: conflict-free) into one register accumulator and adds that to its fold F[r] in shared
// memory once per chunk (only the owning lane touches F[r]: no atomics).  After the last chunk every lane
// turns its residues into (re, im) with fp64 sincospi, the warp reduces them with a fixed xor-shuffle tree and
// lane 0 writes I(P).  The summation order depends only on the segment and P: results are bit-identical
// from run to run and do not depend on the other segments of the launch.
// Roofline: one shared-memory load and one add per (position, period) - the fold additions - bound by the
// shared-memory load rate (DESIGN.md 4.12).
#include <math.h>

#include "ftk_common.cuh"

namespace ftk {

constexpr int kSpecWarps = 16;
constexpr int kSpecThreads = kSpecWarps * 32;
constexpr int kSpecChunk = 8192;   // staged values per chunk: 32 KB (int32) / 64 KB (fp64)

template <class T> struct SpecAcc;
template <> struct SpecAcc<int32_t> { using type = long long; };
template <> struct SpecAcc<double> { using type = double; };

template <class T>
size_t spectrum_smem_bytes(int max_period) {
    return (size_t)kSpecChunk * sizeof(T) + (size_t)kSpecWarps * max_period * sizeof(typename SpecAcc<T>::type);
}

template <class T>
__global__ void __launch_bounds__(kSpecThreads)
spectrum_kernel(const T *__restrict__ x, const int64_t *__restrict__ offsets, int min_period, int n_periods,
                int groups, int max_period, double *__restrict__ out) {
    using Acc = typename SpecAcc<T>::type;
    extern __shared__ __align__(16) unsigned char spec_smem[];
    T *stage = reinterpret_cast<T *>(spec_smem);
    Acc *fold_all = reinterpret_cast<Acc *>(spec_smem + (size_t)kSpecChunk * sizeof(T));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t seg = blockIdx.x / (unsigned)groups;
    const int group = (int)(blockIdx.x % (unsigned)groups);
    const int pi = group + warp * groups;                 // this warp's period index (>= n_periods: idle)
    const bool active = pi < n_periods;
    const int P = min_period + pi;
    const int64_t s0 = __ldg(offsets + seg), N = __ldg(offsets + seg + 1) - s0;
    double *row = out + seg * (int64_t)n_periods;
    if (N <= 0) {
        if (active && lane == 0) row[pi] = __longlong_as_double(0x7ff8000000000000ll);   // quiet NaN
        return;
    }
    Acc *fold = fold_all + warp * max_period;
    if (active)
        for (int r = lane; r < P; r += 32) fold[r] = Acc(0);

    // c0 = k0 * P + cm with 0 <= cm < P, kept incrementally (32-bit divisions only); at the end
    // N = per * P + rem gives the residue counts c_r = per + (r < rem)
    int64_t k0 = 0, per = 0;
    int cm = 0, rem = 0;
    for (int64_t c0 = 0; c0 < N; c0 += kSpecChunk) {
        const int len = (int)min((int64_t)kSpecChunk, N - c0);
        __syncthreads();                                  // the previous chunk is folded
        const T *src = x + s0 + c0;
#pragma unroll 4
        for (int i = threadIdx.x; i < len; i += kSpecThreads) stage[i] = __ldcs(src + i);
        __syncthreads();
        if (!active) continue;
        // chunk position i is segment position c0 + i; block k covers segment positions [kP, kP + P)
        const int first = -cm;                            // chunk index of block k0's residue 0, in (-P, 0]
        const int nblk = (cm + len - 1) / P;              // blocks after k0 that touch the chunk
        for (int r = lane; r - lane < P; r += 32) {
            Acc acc = Acc(0);
            if (r < P) {
                int i = first + r;
                if (i >= 0 && i < len) acc += (Acc)stage[i];
                i += P;
                // interior blocks lie inside the chunk: no bounds test
#pragma unroll 4
                for (int b = 1; b < nblk; ++b, i += P) acc += (Acc)stage[i];
                if (nblk > 0 && i < len) acc += (Acc)stage[i];
                fold[r] += acc;
            }
        }
        per = k0 + (cm + len) / P;
        rem = (cm + len) % P;
        k0 += (cm + kSpecChunk) / P;
        cm = (cm + kSpecChunk) % P;
    }
    if (!active) return;

    // mean from the folds (exact for int64), then the twiddled sum over the residues
    Acc tot = Acc(0);
    for (int r = lane; r < P; r += 32) tot += fold[r];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
    const double mu = (double)tot / (double)N;
    const double two_over_p = 2.0 / (double)P;
    double re = 0.0, im = 0.0;
    for (int r = lane; r < P; r += 32) {
        const double d = (double)fold[r] - mu * (double)(per + (r < rem));
        double sn, cs;
        sincospi((double)r * two_over_p, &sn, &cs);
        re = fma(d, cs, re);
        im = fma(-d, sn, im);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        re += __shfl_xor_sync(0xffffffffu, re, o);
        im += __shfl_xor_sync(0xffffffffu, im, o);
    }
    if (lane == 0) row[pi] = (re * re + im * im) / (double)N;
}

template <class T>
int launch_spectrum(const T *x, const int64_t *offsets, int64_t n_seg, int32_t min_period, int32_t max_period,
                    double *out, ftk_stream_t stream_, const char *name) {
    if (n_seg < 0 || !x || !offsets || !out) return FTK_E_INVALID;
    if (min_period < 2 || max_period < min_period) return FTK_E_INVALID;
    if (max_period > FTK_SPECTRUM_MAX_PERIOD) return FTK_E_RANGE;
    const int n_periods = max_period - min_period + 1;
    const int groups = (n_periods + kSpecWarps - 1) / kSpecWarps;
    if (n_seg > INT32_MAX / groups) return FTK_E_RANGE;
    if (n_seg == 0) return FTK_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const size_t smem = spectrum_smem_bytes<T>(max_period);
    FTK_CUDA_TRY(cudaFuncSetAttribute(spectrum_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    spectrum_kernel<T><<<(unsigned)(n_seg * groups), kSpecThreads, smem, stream>>>(
        x, offsets, min_period, n_periods, groups, max_period, out);
    FTK_CHECK_LAUNCH(name);
    return FTK_OK;
}

}  // namespace ftk

using namespace ftk;

extern "C" int ftk_spectrum_i32_f64(const int32_t *x, const int64_t *offsets, int64_t n_seg, int32_t min_period,
                                    int32_t max_period, double *out, ftk_stream_t stream) {
    return launch_spectrum<int32_t>(x, offsets, n_seg, min_period, max_period, out, stream, "spectrum_kernel<int32>");
}

extern "C" int ftk_spectrum_f64_f64(const double *x, const int64_t *offsets, int64_t n_seg, int32_t min_period,
                                    int32_t max_period, double *out, ftk_stream_t stream) {
    return launch_spectrum<double>(x, offsets, n_seg, min_period, max_period, out, stream, "spectrum_kernel<fp64>");
}
