// adjust_wps on sm_100a: running median / mean subtraction + Savitzky-Golay smoothing.
//
// Replaces _local_filter / _running_stat (frag/_adjust_wps.py:25-45: numpy
// sliding_window_view + np.median / np.mean per window, O(n w log w)) and the
// scipy.signal.savgol_filter call (frag/_adjust_wps.py:135-138, mode='interp') of
// _single_adjust_wps (frag/_adjust_wps.py:63-163).
//
//   adj[j] = s[j + w/2] - stat(s[j : j+w]),  j in [0, n-w),  s = x - shift
//   out    = savgol(adj)  : interior = 21-tap (sg_w) fp64 stencil, first/last sg_w/2
//            outputs = polynomial fit of the first/last sg_w samples (edge matrices)
//
// Raw WPS is integer-valued with a small local range, so the running median is a
// sliding HISTOGRAM median (add one sample, drop one, walk the median bin): O(1) per
// output instead of a sort per window.  Work unit = "run": run_len consecutive outputs
// of one segment, owned by ONE thread that slides its private shared-memory histogram
// (int16 bins, bank-conflict-free layout) along the run, fed from warp-cooperative
// coalesced tile refills.  Runs whose samples are not integers or leave the kAdjBins-wide
// local window are flagged and redone by the generic kernel (sorted-window insertion, any
// float input).  Savitzky-Golay is a separate one-thread-per-output stencil kernel.
// fp64 arithmetic follows numpy's: median of an even window = (lo + hi) / 2 on the
// shifted values; mean = exact integer sum / w.
// Roofline: HBM, 4 B in (float32 sample) + 8 B out (float64) per position.
#include <type_traits>

#include "ftk_common.cuh"

namespace ftk {

constexpr int kAdjThreads = 128;
constexpr int kAdjWarps = kAdjThreads / 32;
constexpr int kAdjBins = 256;       // local value window of the fast path
constexpr int kAdjMaxSg = 127;      // Savitzky-Golay window limit
constexpr int kAdjTile = 16;        // samples staged per lane per refill
constexpr int kAdjTilePitch = 20;   // bytes per tile row: 5-word stride, row reads are bank-conflict-free

struct AdjParams {
    int w;            // median / mean window (even)
    int use_mean;
    int run;          // outputs per run
};

__device__ __forceinline__ long long find_segment(const long long *__restrict__ off, int n_seg, long long v) {
    int lo = 0, hi = n_seg;  // last s with off[s] <= v
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (off[mid] <= v) lo = mid; else hi = mid;
    }
    return lo;
}

// ---------------------------------------------------------------- fast path
// One thread = one run of P.run outputs; it consumes its sample stream g = 0, 1, ... (sample
// index ca + g): every step adds sample g to its private histogram, drops sample g - w, and once
// g >= w - 1 emits adj[c] for c = ca + g - w + 1 (centre sample ca + g - w/2 + 1).
// The three per-lane sequential streams (in, out, centre) would be 32 scattered 4-byte loads per
// warp instruction; instead each warp refills three 32 x 32 byte tiles with COALESCED loads (row
// i = 32 consecutive samples of lane i's stream, 128 B per load, stored as histogram bins
// relative to lane i's base) and every lane then walks its own row from shared memory.
// hist layout: bin-major, slot(tid) = 2*lane + (warp&1) + 64*(warp>>1): the 32 lanes of a warp hit
// 32 distinct banks (two warps share each 32-bit word, 16 bits each).  248 bins x 128 threads x
// int16 + 12.4 KB of tiles = 74.4 KB per CTA -> three CTAs per SM.
// The median state lives in registers (bin m, c_lt = #samples below bin m, hm = H(m)); the
// histogram read-modify-writes are side effects off the critical path and H is only re-read
// when the median bin moves.  Without a shift the adjusted value is an exact half-integer
// ((2*centre - lo - hi) / 2), computed in integers.
template <bool MEAN, bool SHIFT>
__global__ void __launch_bounds__(kAdjThreads, 3)
adjust_hist_kernel(const float *__restrict__ x, const long long *__restrict__ seg_off,
                   const long long *__restrict__ seg_out_off, const long long *__restrict__ seg_run_off,
                   const double *__restrict__ seg_shift, int n_seg, long long n_runs, AdjParams P,
                   double *__restrict__ adj_out, unsigned char *__restrict__ fallback) {
    extern __shared__ short adj_smem[];
    short *hist_smem = adj_smem;                                  // [kAdjBins][kAdjThreads]
    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    unsigned char *tiles = reinterpret_cast<unsigned char *>(adj_smem + kAdjBins * kAdjThreads) +
                           warp * (3 * 32 * kAdjTilePitch);
    unsigned char *t_in = tiles, *t_out = tiles + 32 * kAdjTilePitch, *t_ctr = tiles + 2 * 32 * kAdjTilePitch;
    short *__restrict__ h = hist_smem + (2 * lane + (warp & 1) + 64 * (warp >> 1));
#define H(b) h[(b) * kAdjThreads]
    for (int b = 0; b < kAdjBins; ++b) H(b) = 0;

    const int w = P.w;
    const long long run = (long long)blockIdx.x * kAdjThreads + tid;
    const bool live = run < n_runs;
    int G = 0;                       // steps of this lane's stream
    int limit = 0;                   // samples available from xs_ca on (clamped to int32)
    const float *xs_ca = x;          // &segment[ca]
    double *out_c = adj_out;         // &adj_out[segment output base + ca]
    double shift = 0.0;
    int base = 0;                    // bin = sample - base
    bool bad = false;
    if (live) {
        const long long s = find_segment(seg_run_off, n_seg, run);
        const long long n = seg_off[s + 1] - seg_off[s];
        const long long n_out = n - w;
        const long long ca = (run - seg_run_off[s]) * P.run;
        const long long cb = (ca + P.run < n_out) ? ca + P.run : n_out;
        xs_ca = x + seg_off[s] + ca;
        out_c = adj_out + seg_out_off[s] + ca;
        limit = (int)((n - ca > 0x7fffffff) ? 0x7fffffff : (n - ca));
        G = (int)(cb - ca) + w - 1;
        if (SHIFT) shift = seg_shift[s];
        const float x0 = __ldg(xs_ca);  // centre the bin window on the first sample
        if (x0 != rintf(x0) || fabsf(x0) > 1.0e9f) bad = true;
        base = (int)x0 - kAdjBins / 2;
    }
    const int kl = (w - 1) >> 1, ku = w >> 1;  // 0-based ranks of the two middle order statistics
    int isum = 0;                    // window sum of bins (mean path); |bin| < 256, w <= 32767
    int m = 0, c_lt = 0, hm = 0;
    const int g_max = __reduce_max_sync(0xffffffffu, G);

    // Software-pipelined refill.  A tile holds kAdjTile (16) samples of each of the 32 lanes'
    // three streams.  One load instruction fetches two rows (lanes 0-15 -> row 2i, lanes 16-31 ->
    // row 2i+1: two coalesced 64-byte segments); the loads of tile k+1 are issued into registers
    // BEFORE tile k is processed, so HBM latency hides behind kAdjTile histogram steps.
    float pre[kAdjTile][3];
    const int col = lane & (kAdjTile - 1), sub = lane >> 4;
    auto issue_loads = [&](int g0) {
        const int gi = g0 + col;
        const int i_out = gi - w, i_ctr = gi - (w >> 1) + 1;
#pragma unroll
        for (int i = 0; i < kAdjTile; ++i) {
            const int row = 2 * i + sub;
            const unsigned long long p_i = __shfl_sync(0xffffffffu, (unsigned long long)xs_ca, row);
            const int lim_i = __shfl_sync(0xffffffffu, limit, row);
            const int G_i = __shfl_sync(0xffffffffu, G, row);
            const float fb = (float)__shfl_sync(0xffffffffu, base, row);
            const float *src = reinterpret_cast<const float *>(p_i);
            const bool need = gi < G_i;
            pre[i][0] = (need && gi < lim_i) ? __ldg(src + gi) : fb;
            pre[i][1] = (need && i_out >= 0 && i_out < lim_i) ? __ldg(src + i_out) : fb;
            pre[i][2] = (need && i_ctr >= 0 && i_ctr < lim_i) ? __ldg(src + i_ctr) : fb;
        }
    };
    if (g_max > 0) issue_loads(0);

    for (int g0 = 0; g0 < g_max; g0 += kAdjTile) {
        // ---- registers -> byte tiles (bins relative to the owning lane's base) + validation:
        // a sample must be integer-valued and inside the kAdjBins-wide window around the base
        __syncwarp();   // every lane has finished walking the previous tile
        unsigned inv_bits = 0;
#pragma unroll
        for (int i = 0; i < kAdjTile; ++i) {
            const int row = 2 * i + sub;
            const float fb = (float)__shfl_sync(0xffffffffu, base, row);
            const float d_in = pre[i][0] - fb, d_out = pre[i][1] - fb, d_ctr = pre[i][2] - fb;
            const bool invalid = (d_in != rintf(d_in)) || !(d_in >= 0.0f && d_in < (float)kAdjBins) ||
                                 (d_out != rintf(d_out)) || !(d_out >= 0.0f && d_out < (float)kAdjBins) ||
                                 (d_ctr != rintf(d_ctr)) || !(d_ctr >= 0.0f && d_ctr < (float)kAdjBins);
            inv_bits |= (invalid ? 1u : 0u) << row;
            t_in[row * kAdjTilePitch + col] = (unsigned char)(int)d_in;
            t_out[row * kAdjTilePitch + col] = (unsigned char)(int)d_out;
            t_ctr[row * kAdjTilePitch + col] = (unsigned char)(int)d_ctr;
        }
        if ((__reduce_or_sync(0xffffffffu, inv_bits) >> lane) & 1u) bad = true;
        __syncwarp();
        if (g0 + kAdjTile < g_max) issue_loads(g0 + kAdjTile);   // in flight while this tile is walked
        if (!live || bad) continue;
        // ---- every lane walks its own row
        const int g_end = (G - g0 < kAdjTile) ? (G - g0) : kAdjTile;
        const unsigned char *__restrict__ r_in = t_in + lane * kAdjTilePitch;
        const unsigned char *__restrict__ r_out = t_out + lane * kAdjTilePitch;
        const unsigned char *__restrict__ r_ctr = t_ctr + lane * kAdjTilePitch;
        int t = 0;
        // fill phase: g < w - 1 (histogram only)
        for (; t < g_end && g0 + t < w - 1; ++t) {
            const int bi = r_in[t];
            H(bi) = H(bi) + 1;
            if (MEAN) isum += bi;
        }
        if (t < g_end && g0 + t == w - 1) {  // first complete window: locate the median from scratch
            const int bi = r_in[t];
            H(bi) = H(bi) + 1;
            if (MEAN) isum += bi;
            m = 0; c_lt = 0; hm = H(0);
            while (c_lt + hm <= kl) { c_lt += hm; ++m; hm = H(m); }
        } else if (t < g_end) {
            goto slide;
        } else {
            continue;
        }
        for (;;) {
            {   // emit the output of step g0 + t
                const int bc = r_ctr[t];
                double adj;
                if (MEAN) {
                    const double stat = ((double)isum / (double)w + (double)base) - shift;
                    adj = ((double)(bc + base) - shift) - stat;
                } else {
                    int mu = m;  // upper median: same bin if it still covers rank ku, else next occupied bin
                    if (c_lt + hm <= ku) { do { ++mu; } while (H(mu) == 0); }
                    if (SHIFT) {
                        const double lo = (double)(m + base) - shift, hi = (double)(mu + base) - shift;
                        adj = ((double)(bc + base) - shift) - (lo + hi) / 2.0;
                    } else {
                        adj = (double)(2 * bc - m - mu) * 0.5;
                    }
                }
                out_c[g0 + t - (w - 1)] = adj;
            }
            if (++t >= g_end) break;
        slide:
            {   // slide phase: g >= w
                const int bi = r_in[t], bo = r_out[t];
                H(bi) = H(bi) + 1;
                H(bo) = H(bo) - 1;
                if (MEAN) isum += bi - bo;
                c_lt += (bi < m) - (bo < m);
                hm += (bi == m) - (bo == m);
                while (c_lt > kl) { --m; hm = H(m); c_lt -= hm; }
                while (c_lt + hm <= kl) { c_lt += hm; ++m; hm = H(m); }
            }
        }
    }
    if (live && bad) fallback[run] = 1;
#undef H
}

// ------------------------------------------------------------ generic path
// Any float input: the window is kept sorted in a per-thread scratch array (binary
// search + shift on every step, O(w) per output).  Only flagged runs come here.
// NaN has no place in a sorted order: the window keeps its non-NaN samples sorted
// (len of them) and counts the NaNs; a window holding a NaN has median NaN, as numpy's.
__global__ void __launch_bounds__(64)
adjust_generic_kernel(const float *__restrict__ x, const long long *__restrict__ seg_off,
                      const long long *__restrict__ seg_out_off, const long long *__restrict__ seg_run_off,
                      const double *__restrict__ seg_shift, int n_seg,
                      const long long *__restrict__ run_list, long long n_list, AdjParams P,
                      double *__restrict__ adj_out, float *__restrict__ scratch /* [n_list][w] */) {
    const long long li = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (li >= n_list) return;
    const long long run = run_list[li];
    float *__restrict__ win = scratch + li * (long long)P.w;
    const long long s = find_segment(seg_run_off, n_seg, run);
    const long long n = seg_off[s + 1] - seg_off[s];
    const long long n_out = n - P.w;
    const float *__restrict__ xs = x + seg_off[s];
    double *__restrict__ out = adj_out + seg_out_off[s];
    const double shift = seg_shift ? seg_shift[s] : 0.0;
    const long long ca = (run - seg_run_off[s]) * P.run;
    const long long cb = (ca + P.run < n_out) ? ca + P.run : n_out;
    const int w = P.w;
    int len = 0, n_nan = 0;        // sorted non-NaN samples in win[0, len), NaNs in the window
    auto insert = [&](float v) {
        if (v != v) { ++n_nan; return; }
        int k = len++;
        while (k > 0 && win[k - 1] > v) { win[k] = win[k - 1]; --k; }
        win[k] = v;
    };
    auto find = [&](float v) {     // position of one copy of v
        int lo = 0, hi = len;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (win[mid] < v) lo = mid + 1; else hi = mid; }
        return lo;
    };
    if (!P.use_mean)
        for (int t = 0; t < w; ++t) insert(xs[ca + t]);   // insertion sort of the first window
    for (long long c = ca; c < cb; ++c) {
        double stat;
        if (P.use_mean) {
            double sum = 0.0;  // fp64 left-to-right sum of the shifted window (numpy: pairwise; <= 1e-13 rel apart)
            for (int t = 0; t < w; ++t) sum += (double)xs[c + t] - shift;
            stat = sum / (double)w;
        } else if (n_nan) {
            stat = nan("");
        } else {
            const double lo = (double)win[(w - 1) >> 1] - shift, hi = (double)win[w >> 1] - shift;
            stat = (lo + hi) / 2.0;
        }
        out[c] = ((double)xs[c + (w >> 1)] - shift) - stat;
        if (c + 1 < cb && !P.use_mean) {
            const float vo = xs[c], vi = xs[c + w];
            if (vo != vo || vi != vi) {   // a NaN enters or leaves: drop vo, then insert vi
                if (vo != vo) --n_nan;
                else {
                    for (int k = find(vo); k + 1 < len; ++k) win[k] = win[k + 1];
                    --len;
                }
                insert(vi);
            } else {                      // replace vo by vi in one pass
                int k = find(vo);
                if (vi >= vo) { while (k + 1 < len && win[k + 1] < vi) { win[k] = win[k + 1]; ++k; } }
                else { while (k > 0 && win[k - 1] > vi) { win[k] = win[k - 1]; --k; } }
                win[k] = vi;
            }
        }
    }
}

// ---------------------------------------------------------- Savitzky-Golay
// scipy.signal.savgol_filter(adj, sg_w, deg) with mode='interp': interior = sg_w-tap stencil,
// the first / last sg_w/2 outputs of every segment = polynomial fit of its first / last sg_w
// samples evaluated at those positions (the two edge matrices).
// A CTA stages adj[o0 - half, o0 + kSgTile + half) in shared memory; every thread owns FOUR
// consecutive outputs and slides a 4-register window over the taps, so a tap costs one tile read
// and one (broadcast) coefficient read for four fused multiply-adds - the one-output-per-thread
// version re-read both operands for every FMA and sat on the shared-memory pipe.  Element e lives
// at slot e + (e >> 4): with that padding the 32 lanes' 8-byte reads (stride 4 elements) hit every
// bank pair exactly twice, i.e. they are conflict-free.  Results go back through shared memory so
// the global stores are coalesced.  Taps are accumulated in tap order like the reference stencil.
constexpr int kSgThreads = 256;
constexpr int kSgPerThread = 4;
constexpr int kSgTile = kSgThreads * kSgPerThread;   // outputs per CTA
__device__ __forceinline__ int sg_slot(int e) { return e + (e >> 4); }

// SGW > 0: window known at compile time (the reference default, 21): the thread's SGW + 3 inputs are
// loaded into registers once and the taps are fully unrolled; SGW == 0: any odd window <= 127.
template <int SGW>
__global__ void __launch_bounds__(kSgThreads)
adjust_savgol_kernel(const double *__restrict__ adj, const long long *__restrict__ seg_out_off, int n_seg,
                     long long n_total, int sg_w, const double *__restrict__ coef,
                     const double *__restrict__ edge_first, const double *__restrict__ edge_last,
                     double *__restrict__ out) {
    constexpr int kIn = kSgTile + kAdjMaxSg + 3;
    __shared__ double s_coef[kAdjMaxSg + 1];
    __shared__ double s_tile[kIn + (kIn >> 4) + 1];
    __shared__ double s_out[kSgTile + (kSgTile >> 4) + 1];
    __shared__ long long s_seg0;
    const int half = sg_w >> 1;
    for (int i = threadIdx.x; i < sg_w; i += kSgThreads) s_coef[i] = coef[i];
    const long long o0 = (long long)blockIdx.x * kSgTile;
    if (threadIdx.x == 0) s_seg0 = find_segment(seg_out_off, n_seg, o0);
    for (int i = threadIdx.x; i < kSgTile + 2 * half + 3; i += kSgThreads) {   // coalesced tile load
        const long long g = o0 - half + i;
        s_tile[sg_slot(i)] = (g >= 0 && g < n_total) ? adj[g] : 0.0;
    }
    __syncthreads();

    const int l0 = threadIdx.x * kSgPerThread;        // first of this thread's 4 consecutive outputs
    // interior stencil for all four (edge outputs are overwritten below)
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    if (SGW > 0) {
        double r[SGW + 3];
#pragma unroll
        for (int i = 0; i < SGW + 3; ++i) r[i] = s_tile[sg_slot(l0 + i)];
#pragma unroll
        for (int i = 0; i < SGW; ++i) {
            const double c = s_coef[i];
            a0 += c * r[i]; a1 += c * r[i + 1]; a2 += c * r[i + 2]; a3 += c * r[i + 3];
        }
    } else {
        double r0 = s_tile[sg_slot(l0)], r1 = s_tile[sg_slot(l0 + 1)], r2 = s_tile[sg_slot(l0 + 2)];
        for (int i = 0; i < sg_w; ++i) {
            const double r3 = s_tile[sg_slot(l0 + i + 3)];
            const double c = s_coef[i];
            a0 += c * r0; a1 += c * r1; a2 += c * r2; a3 += c * r3;
            r0 = r1; r1 = r2; r2 = r3;
        }
    }
    // first / last `half` outputs of a segment: polynomial edge fit instead of the stencil.  The
    // segment of the thread's first output is located once; the other three only test its end.
    long long s = s_seg0;
    const long long o_first = o0 + l0;
    while (s + 1 < n_seg && seg_out_off[s + 1] <= o_first) ++s;
    long long seg_b = seg_out_off[s], seg_e = seg_out_off[s + 1];
    auto finish = [&](int k, double interior) {
        const long long o = o_first + k;
        double v = interior;
        if (o < n_total) {
            while (o >= seg_e && s + 1 < n_seg) { ++s; seg_b = seg_e; seg_e = seg_out_off[s + 1]; }
            const long long j = o - seg_b, n_out = seg_e - seg_b;
            if (j < half) {
                const double *__restrict__ p = adj + seg_b;
                v = 0.0;
                for (int i = 0; i < sg_w; ++i) v += edge_first[j * sg_w + i] * p[i];
            } else if (j >= n_out - half) {
                const double *__restrict__ p = adj + seg_e - sg_w;
                v = 0.0;
                for (int i = 0; i < sg_w; ++i) v += edge_last[(j - (n_out - half)) * sg_w + i] * p[i];
            }
        }
        s_out[sg_slot(l0 + k)] = v;
    };
    finish(0, a0); finish(1, a1); finish(2, a2); finish(3, a3);
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kSgPerThread; ++k) {
        const int local = k * kSgThreads + threadIdx.x;
        const long long o = o0 + local;
        if (o < n_total) out[o] = s_out[sg_slot(local)];
    }
}

// ------------------------------------------------- rank-bitmap median + fused Savitzky-Golay
// The sliding-histogram kernel above is one long serial chain per thread (w-1 fill steps before the
// first output, then a histogram read-modify-write per step): latency- and occupancy-bound at 8 % of
// the HBM roofline.  This kernel removes the fill and the private histograms:
//
//   * one CTA per tile = up to ~4000 consecutive outputs of ONE segment; its A + w samples are
//     staged in shared memory once (coalesced, int16);
//   * for a band of 32 consecutive value levels the CTA builds level bitmaps (every lane turns its
//     sample into a 32-level mask, a 5-step shuffle transpose turns 32 masks into 32 bitmap words:
//     bit i of B[r] = sample i <= level r) plus per-word prefix popcounts, so the rank
//     F(r, j) = #{samples of window j <= level r} is TWO popcount lookups for ANY window j - O(1)
//     random access instead of a w-step fill;
//   * every thread owns a short run of R (~11) consecutive outputs: binary search over the band for
//     its first lower median (7 rank queries), then slides (+1 / -1 sample, two compares) and
//     consults the bitmaps only when the median changes level; the upper median (even window) is
//     the same level or the next occupied one;
//   * the band is centred on a sampled median of the tile; an order statistic that falls outside is
//     picked up by further passes with the band moved down / up (each of the two middle order
//     statistics of an output resolves independently, in whichever band holds it), a tile that
//     cannot be resolved (non-integer samples, |x| > 32000, > kRankMaxPasses bands) is flagged and
//     redone by the histogram / generic path;
//   * the adjusted series never leaves the SM: Savitzky-Golay (interior stencil + per-segment edge
//     fits) runs on the shared-memory copy (+-sg_w/2 halo outputs are recomputed per tile) and only
//     the final float64 result is written, warp-staged for coalesced stores.
// HBM traffic = the algorithmic 4 B in + 8 B out per position (the split design moved 28 B).
#ifndef FTK_RANK_THREADS
#define FTK_RANK_THREADS 384
#endif
constexpr int kRankThreads = FTK_RANK_THREADS;
constexpr int kRankWarps = kRankThreads / 32;
constexpr int kRankLevels = 32;        // band rows: one bitmap row per lane
constexpr int kRankMaxPasses = 12;
constexpr int kRankMaxAbs = 32000;     // samples are staged as int16

struct RankGeom {                       // shared-memory carve-up, identical on host and device
    int a_slots;                        // adj elements incl. padding
    int nwp;                            // words per bitmap row (odd, >= ceil(S/32) + 1)
    int s_pad;                          // staged samples (multiple of 32)
};
__host__ __device__ inline RankGeom rank_geom(int a_cap, int s_cap) {
    RankGeom g;
    g.a_slots = a_cap + (a_cap >> 4) + 2;
    const int nword = (s_cap + 31) / 32;
    g.nwp = (nword + 1) | 1;
    if (g.nwp < 69) g.nwp = 69;     // the bitmap area doubles as the 12 x 136-double store staging
    g.s_pad = nword * 32;
    return g;
}
__host__ __device__ inline size_t rank_smem_bytes(int a_cap, int s_cap, bool shifted) {
    const RankGeom g = rank_geom(a_cap, s_cap);
    size_t b = (size_t)g.a_slots * (shifted ? sizeof(double) : sizeof(int));
    b = (b + 15) & ~(size_t)15;
    b += (size_t)kRankLevels * g.nwp * 8;       // (bitmap word, prefix popcount) pairs: one 64-bit read per rank query
    b = (b + 15) & ~(size_t)15;
    b += (size_t)(g.s_pad + 32) * 2;            // samples
    return b;
}

__device__ __forceinline__ bool rank_stage(float v, int &iv) {
    iv = (int)v;
    return (v == (float)iv) && (fabsf(v) <= (float)kRankMaxAbs);
}
__device__ __forceinline__ bool rank_stage(int v, int &iv) {
    iv = v;
    return (v >= -kRankMaxAbs) && (v <= kRankMaxAbs);
}

// 32 x 32 bit-matrix transpose across a warp: lane i holds row i, afterwards lane r holds column r.
// Stage s swaps the off-diagonal s x s blocks between lanes l and l ^ s: the lower lane takes the
// partner's word shifted up by s into its high sub-blocks, the upper lane takes it shifted down into
// its low sub-blocks - one rotate (the unwanted half of the rotation is masked away) and one
// select-by-mask per stage.
__device__ __forceinline__ unsigned warp_transpose32(unsigned x, int lane) {
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const unsigned msk = (s == 16) ? 0x0000ffffu : (s == 8) ? 0x00ff00ffu : (s == 4) ? 0x0f0f0f0fu
                           : (s == 2) ? 0x33333333u : 0x55555555u;
        const bool upper = (lane & s) != 0;
        const unsigned take = upper ? msk : ~msk;            // bits this lane receives from its partner
        const unsigned y = __shfl_xor_sync(0xffffffffu, x, s);
        const unsigned rot = __funnelshift_l(y, y, upper ? 32 - s : s);
        x = (x & ~take) | (rot & take);
    }
    return x;
}

// SHIFT = subtract_edges (per-segment fp64 shift): the adjusted value is then a general double;
// without it 2 * adj is an integer and the tile keeps THAT as int32 (half the shared memory: three
// CTAs per SM instead of two), the factor 1/2 folded into the Savitzky-Golay coefficients
// (fma(c/2, 2a, acc) == fma(c, a, acc) bit for bit).
// MOM: exact sliding-moment smoothing (no SHIFT, rational coefficients given): the adjusted values then sit
// unpadded in shared memory (the 1-in-16 padding only serves the fp64 stencil's 8-byte reads)
template <typename InT, bool SHIFT, int SGW, bool MOM>   // SGW: 21 = unrolled default, 0 = runtime window, -1 = no smoothing
__global__ void __launch_bounds__(kRankThreads, 3)
adjust_rank_kernel(const InT *__restrict__ x, const long long *__restrict__ seg_off,
                   const long long *__restrict__ seg_out_off, const double *__restrict__ seg_shift,
                   const int *__restrict__ tile_seg, const int *__restrict__ tile_t0,
                   const int *__restrict__ tile_n, int w, int sg_w, const double *__restrict__ coef,
                   const double *__restrict__ edge_first, const double *__restrict__ edge_last,
                   long long sg_a, long long sg_b, double sg_scale, int sg_fit32,
                   int a_cap, int s_cap, double *__restrict__ out, unsigned char *__restrict__ tile_flag) {
    extern __shared__ __align__(16) unsigned char rank_smem[];
    __shared__ int s_ctl[4];            // 0: need lower band, 1: need higher band, 2: unused, 3: centre
    __shared__ int s_tot[kRankWarps][kRankLevels];   // per-warp-chunk row totals of the bitmap build
    __shared__ double s_coef[kAdjMaxSg + 1];
    using AdjT = typename std::conditional<SHIFT, double, int>::type;
    const RankGeom G = rank_geom(a_cap, s_cap);
    // adj slot j first holds the two middle order statistics of window j as an int16 pair, then the
    // adjusted value (double, or the integer 2 * adj)
    AdjT *__restrict__ adj = reinterpret_cast<AdjT *>(rank_smem);
    const size_t o_b = ((size_t)G.a_slots * sizeof(AdjT) + 15) & ~(size_t)15;
    uint2 *__restrict__ B = reinterpret_cast<uint2 *>(rank_smem + o_b);      // .x bitmap word, .y samples before it <= level
    const size_t o_x = (o_b + (size_t)kRankLevels * G.nwp * 8 + 15) & ~(size_t)15;
    short *__restrict__ xs = reinterpret_cast<short *>(rank_smem + o_x);
    const int nwp = G.nwp;

    auto aslot = [](int e) { return MOM ? e : sg_slot(e); };
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tile = blockIdx.x;
    const int sg = tile_seg[tile];
    const int t0 = tile_t0[tile], n_t = tile_n[tile];
    const long long seg0 = seg_off[sg];
    const int n = (int)(seg_off[sg + 1] - seg0);
    const int n_out = n - w;
    const int half = (SGW < 0) ? 0 : (sg_w >> 1);
    // adjusted values this tile needs: its outputs +- half, plus the first / last sg_w of the
    // segment when it holds edge outputs
    int a0 = max(t0 - half, 0), a1 = min(t0 + n_t + half, n_out);
    if (SGW >= 0) {
        if (t0 < half) a1 = max(a1, min(sg_w, n_out));
        if (t0 + n_t > n_out - half) a0 = min(a0, max(n_out - sg_w, 0));
    }
    const int A = a1 - a0, S = A + w;
    if (tid < 3) s_ctl[tid] = 0;
    if (SGW >= 0) for (int i = tid; i < sg_w; i += kRankThreads) s_coef[i] = SHIFT ? coef[i] : coef[i] * 0.5;
    bool bad = (A > a_cap) || (S > s_cap) || (A <= 0);
    // ---- stage the samples (coalesced), validate: integer-valued and small
    if (!bad) {
        const InT *__restrict__ src = x + seg0 + a0;
        // eight loads per thread are in flight before the first one is looked at: the tile's samples cost
        // two DRAM round trips instead of one per 384 samples
        constexpr int kStageU = 8;
        for (int i0 = tid; i0 < G.s_pad + 32; i0 += kStageU * kRankThreads) {
            InT v[kStageU];
#pragma unroll
            for (int u = 0; u < kStageU; ++u) {
                const int i = i0 + u * kRankThreads;
                v[u] = (i < S) ? __ldg(src + i) : InT(0);
            }
#pragma unroll
            for (int u = 0; u < kStageU; ++u) {
                const int i = i0 + u * kRankThreads;
                int iv = 32767;                   // sentinel beyond every level: never counted
                if (i < S) {
                    if (!rank_stage(v[u], iv)) { bad = true; iv = 0; }
                }
                if (i < G.s_pad + 32) xs[i] = (short)iv;
            }
        }
    }
    if (__syncthreads_or(bad ? 1 : 0)) {
        if (tid == 0) tile_flag[tile] = 1;
        return;
    }
    // ---- band centre: median of 32 samples spread over the tile (rank by 32 shuffles)
    if (warp == 0) {
        const int mine = xs[(int)(((long long)lane * S) >> 5) + (S >> 6)];
        int rank = 0;
#pragma unroll
        for (int l = 0; l < 32; ++l) {
            const int o = __shfl_sync(0xffffffffu, mine, l);
            rank += (o < mine) || (o == mine && l < lane);
        }
        if (rank == 16) s_ctl[3] = mine;
    }
    __syncthreads();

    const int kl = (w - 1) >> 1, ku = w >> 1;   // 0-based ranks of the two middle order statistics
    const int R = (A + kRankThreads - 1) / kRankThreads;   // outputs per thread (<= 32)
    const int j0 = tid * R;
    const int mine_n = max(min(A - j0, R), 0);
    const unsigned full_mask = (mine_n >= 32) ? 0xffffffffu : ((1u << mine_n) - 1u);
    auto cnt = [&](int r, int i) -> int {       // #{samples [0, i) <= level r}
        const int wd = i >> 5;
        const uint2 e = B[r * nwp + wd];
        return (int)e.y + __popc(e.x & ((1u << (i & 31)) - 1u));
    };
    auto F = [&](int r, int j) -> int { return cnt(r, j + w) - cnt(r, j); };
    // smallest row whose rank count reaches `need`: -1 below the band (row 0 already does), 32 above
    auto locate = [&](int j, int need, int &flo, int &fhi) -> int {
        flo = F(0, j);
        if (flo >= need) return -1;
        fhi = F(kRankLevels - 1, j);
        if (fhi < need) return kRankLevels;
        int lo = 0, hi = kRankLevels - 1;
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            const int f = F(mid, j);
            if (f >= need) { hi = mid; fhi = f; } else { lo = mid; flo = f; }
        }
        return hi;
    };
    // words each warp turns into bitmaps: one contiguous chunk per warp (running row counts in registers)
    const int n_words = min(((S + 31) >> 5) + 1, nwp);
    const int wpw = (n_words + kRankWarps - 1) / kRankWarps;
    const int wd_lo = min(warp * wpw, n_words), wd_hi = min(wd_lo + wpw, n_words);

    unsigned done_m = 0, done_u = 0;             // per-output bits: lower / upper median known
    int n_fast = 0;                              // outputs the first pass' fast walk finished (adj already final)
    int L0 = s_ctl[3] - (kRankLevels / 2 - 1);   // row r <-> level L0 - 1 + r; rows 1..31 resolve
    int lo_band = L0, hi_band = L0;
    bool is_lowest = true, is_highest = true, pend_lo = false, pend_hi = false;
    for (int pass = 0;; ++pass) {
        // ---- level bitmaps + chunk-local per-word prefix popcounts (lane r owns row r)
        {
            int run = 0;
            for (int wd = wd_lo; wd < wd_hi; ++wd) {
                const int d = (int)xs[wd * 32 + lane] - (L0 - 1);     // sample <= level r  <=>  r >= d
                // ~0 << d with d clamped to [0, 32]: one max + one clamping funnel shift
                const unsigned mask = __funnelshift_lc(0u, 0xffffffffu, (unsigned)max(d, 0));
                const unsigned bits = warp_transpose32(mask, lane);
                B[lane * nwp + wd] = make_uint2(bits, (unsigned)run);
                run += __popc(bits);
            }
            s_tot[warp][lane] = run;
        }
        __syncthreads();
        {   // add the totals of the chunks to the left (every warp fixes up its own chunk)
            int off = 0;
            for (int c = 0; c < warp; ++c) off += s_tot[c][lane];
            if (off)
                for (int wd = wd_lo; wd < wd_hi; ++wd) B[lane * nwp + wd].y += (unsigned)off;
        }
        __syncthreads();
        // ---- every thread walks its run
        int i_first = 0;
        if (pass == 0 && mine_n > 0) {
            // fast path of the first pass: both middle order statistics of every output are still
            // unknown and almost always inside the band - locate the first lower median, then slide;
            // the general loop below takes over at the first output that does not resolve here
            int flo, fhi;
            int m = locate(j0, kl + 1, flo, fhi);
            if (m >= 0 && m < kRankLevels) {
                int c_lt = flo, hm = fhi - flo;
                int slot_i = aslot(j0);
                for (;;) {
                    const int j = j0 + i_first;
                    int ru = m;                              // upper median: same level unless rank ku is past it
                    if (c_lt + hm <= ku) {
                        const int below = c_lt + hm;
                        ru = -1;
                        for (int r = m + 1; r <= kRankLevels - 1; ++r)
                            if (F(r, j) > below) { ru = r; break; }
                        if (ru < 0) break;                   // next occupied level above the band: general loop
                    }
                    const int lvl = L0 - 1;
                    if (SHIFT)
                        *reinterpret_cast<unsigned *>(adj + slot_i) = ((unsigned)(lvl + ru) << 16) | ((unsigned)(lvl + m) & 0xffffu);
                    else        // both medians known: store 2 * adj right away (exact integer)
                        adj[slot_i] = (AdjT)(2 * (int)xs[j + (w >> 1)] - 2 * lvl - m - ru);
                    if (++i_first >= mine_n) break;
                    // slide to window j + 1
                    const int lv = lvl + m;
                    const int xo = xs[j], xi = xs[j + w];
                    c_lt += (xi < lv) - (xo < lv);
                    hm += (xi == lv) - (xo == lv);
                    slot_i += MOM ? 1 : 1 + (((j + 1) & 15) == 0);
                    bool ok = true;
                    while (c_lt > kl) {                      // median moved down
                        if (--m < 1) { ok = false; break; }
                        const int q = F(m - 1, j + 1);
                        hm = c_lt - q; c_lt = q;
                    }
                    while (ok && c_lt + hm <= kl) {          // median moved up
                        c_lt += hm;
                        if (++m > kRankLevels - 1) { ok = false; break; }
                        hm = F(m, j + 1) - c_lt;
                    }
                    if (!ok) break;
                }
            }
            const unsigned got = (i_first >= 32) ? 0xffffffffu : ((1u << i_first) - 1u);
            done_m = got; done_u = got;
            n_fast = i_first;
        }
        {
            bool valid = false;                  // (m, c_lt, hm) describe window j - 1's lower median
            int m = 0, c_lt = 0, hm = 0;
            for (int i = i_first; i < mine_n; ++i) {
                const int j = j0 + i;
                const bool need_m = !((done_m >> i) & 1u), need_u = !((done_u >> i) & 1u);
                short *__restrict__ slot = reinterpret_cast<short *>(adj + aslot(j));
                if (!need_m) { valid = false; }
                else if (valid) {
                    const int lv = L0 - 1 + m;
                    const int xo = xs[j - 1], xi = xs[j - 1 + w];
                    c_lt += (xi < lv) - (xo < lv);
                    hm += (xi == lv) - (xo == lv);
                    while (c_lt > kl) {                 // median moved down
                        if (--m < 1) { valid = false; s_ctl[0] = 1; break; }
                        const int q = F(m - 1, j);
                        hm = c_lt - q; c_lt = q;
                    }
                    while (valid && c_lt + hm <= kl) {  // median moved up
                        c_lt += hm;
                        if (++m > kRankLevels - 1) { valid = false; s_ctl[1] = 1; break; }
                        hm = F(m, j) - c_lt;
                    }
                } else {
                    int flo, fhi;
                    const int r = locate(j, kl + 1, flo, fhi);
                    if (r < 0) s_ctl[0] = 1;
                    else if (r >= kRankLevels) s_ctl[1] = 1;
                    else { m = r; c_lt = flo; hm = fhi - flo; valid = true; }
                }
                if (need_m && valid) { slot[0] = (short)(L0 - 1 + m); done_m |= 1u << i; }
                if (need_u) {
                    int ru = -2;                         // row of the upper median, -2 = not in this band
                    if (need_m && valid) {               // next to the lower median just found
                        if (c_lt + hm > ku) ru = m;
                        else {
                            const int below = c_lt + hm;
                            for (int r = m + 1; r <= kRankLevels - 1; ++r)
                                if (F(r, j) > below) { ru = r; break; }
                            if (ru < 0) s_ctl[1] = 1;    // next occupied level lies above the band
                        }
                    } else {                             // on its own (its lower partner lives in another band)
                        int flo, fhi;
                        const int r = locate(j, ku + 1, flo, fhi);
                        if (r < 0) s_ctl[0] = 1;
                        else if (r >= kRankLevels) s_ctl[1] = 1;
                        else ru = r;
                    }
                    if (ru >= 0) { slot[1] = (short)(L0 - 1 + ru); done_u |= 1u << i; }
                }
            }
        }
        const bool done = (done_m == full_mask) && (done_u == full_mask);
        const int all_done = __syncthreads_and(done ? 1 : 0);
        const int need_lo = s_ctl[0], need_hi = s_ctl[1];
        __syncthreads();
        if (all_done) break;
        if (tid == 0) { s_ctl[0] = 0; s_ctl[1] = 0; }
        if (is_lowest) pend_lo = need_lo != 0;
        if (is_highest) pend_hi = need_hi != 0;
        if (pass + 1 >= kRankMaxPasses || (!pend_lo && !pend_hi)) {
            if (tid == 0) tile_flag[tile] = 1;
            return;
        }
        if (pend_lo) { L0 = lo_band - (kRankLevels - 1); lo_band = L0; is_lowest = true; is_highest = false; }
        else { L0 = hi_band + (kRankLevels - 1); hi_band = L0; is_highest = true; is_lowest = false; }
        __syncthreads();    // s_ctl reset visible before the next walk; bitmaps free to rebuild
    }

    // ---- (lower, upper) median -> adjusted value, in place (numpy: median of an even window = mean of the two)
    {
        if (SHIFT) {
            const double shift = seg_shift[sg];
            for (int j = tid; j < A; j += kRankThreads) {
                const short *slot = reinterpret_cast<const short *>(adj + aslot(j));
                const int vm = slot[0], vu = slot[1];
                const int bc = xs[j + (w >> 1)];
                const double lo_s = (double)vm - shift, hi_s = (double)vu - shift;
                adj[aslot(j)] = (AdjT)(((double)bc - shift) - (lo_s + hi_s) / 2.0);
            }
        } else {
            for (int i = n_fast; i < mine_n; ++i) {                  // usually none
                const int j = j0 + i;
                const short *slot = reinterpret_cast<const short *>(adj + aslot(j));
                const int vm = slot[0], vu = slot[1];
                adj[aslot(j)] = (AdjT)(2 * (int)xs[j + (w >> 1)] - vm - vu);   // 2 * adj, exact
            }
        }
    }
    __syncthreads();

    // ---- Savitzky-Golay on the shared-memory series + coalesced store
    double *__restrict__ dst = out + seg_out_off[sg] + t0;
    auto val = [&](int k) -> double {            // adjusted value at tile-relative index k (edge fits, no smoothing)
        return SHIFT ? (double)adj[aslot(k)] : (double)adj[aslot(k)] * 0.5;
    };
    if (SGW < 0) {
        for (int k = tid; k < n_t; k += kRankThreads) dst[k] = val(t0 - a0 + k);
        return;
    }
    if (MOM) {
        // Exact sliding-moment smoothing.  For polynomial degree <= 3 the interior coefficients are
        // c_i = (sg_a + sg_b * i^2) / den, so with x = 2 * adj (integers)
        //     y_j = (sg_a * S0_j + sg_b * M2_j) / (2 den),  S0 = sum x, M1 = sum i x, M2 = sum i^2 x over the window,
        // and the three moments slide in O(1): every thread owns a run of consecutive outputs, pays the
        // sg_w-tap sum once and then two shared-memory reads + a handful of integer operations per output
        // (the stencil above costs sg_w fp64 FMAs + sg_w / 4 + 1 loads and conversions per output).  The
        // result is the correctly rounded exact rational times one rounded constant (<= 1 ulp off the
        // true value; the fp64 stencil is ~1e-16 x sum |c_i x_i| off it).  Edge outputs keep the
        // per-segment polynomial fit.  The bitmaps / samples are dead by now: their space stages the
        // results so the global stores are coalesced.
        double *__restrict__ ystage = reinterpret_cast<double *>(rank_smem + o_b);
        const int Ro = ((n_t + kRankThreads - 1) / kRankThreads) | 1;      // odd run length: conflict-free 8-byte staging
        const int k_lo = min(tid * Ro, n_t), k_hi = min(k_lo + Ro, n_t);
        const int h = half, h1 = half + 1;
        const int hh = h * h, h1h1 = h1 * h1;
        int S0 = 0, M1 = 0, M2 = 0;
        // interior outputs of this thread's run (the segment's first / last `half` outputs are edge fits, below)
        const int ki_lo = max(k_lo, h - t0), ki_hi = min(k_hi, n_out - h - t0);
        for (int k = ki_lo; k < ki_hi; ++k) {
            const int c = t0 + k - a0;           // index of the output's adjusted value in the tile
            if (k == ki_lo) {
                for (int i = -h; i <= h; ++i) {
                    const int xv = adj[aslot(c + i)];
                    S0 += xv; M1 += i * xv; M2 += i * i * xv;
                }
            } else {                              // window centre c - 1 -> c
                const int xo = adj[aslot(c - h1)], xi = adj[aslot(c + h)];
                M2 += S0 - 2 * M1 - h1h1 * xo + hh * xi;
                M1 += h1 * xo + h * xi - S0;
                S0 += xi - xo;
            }
            // (the launcher passes |sg_a|, |sg_b| < 2^31; sg_fit32: the combination itself fits int32)
            ystage[k] = sg_fit32 ? (double)((int)sg_a * S0 + (int)sg_b * M2) * sg_scale
                                 : (double)(sg_a * (long long)S0 + sg_b * (long long)M2) * sg_scale;
        }
        // the 2 * half edge outputs of the segment (polynomial fit of its first / last sg_w adjusted
        // values), one thread each so the table loads of different outputs overlap
        for (int e = tid; e < 2 * h; e += kRankThreads) {
            const bool head = e < h;
            const int j = head ? e : n_out - 2 * h + e;
            if (j < t0 || j >= t0 + n_t) continue;
            const double *__restrict__ tab = head ? edge_first + (size_t)e * sg_w : edge_last + (size_t)(e - h) * sg_w;
            const int first = head ? -a0 : n_out - sg_w - a0;
            double acc = 0.0;
            for (int i = 0; i < sg_w; ++i) acc += tab[i] * val(first + i);
            ystage[j - t0] = acc;
        }
        __syncthreads();
        if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {       // 16-byte stores (ystage is 16-byte aligned)
            const int n2 = n_t >> 1;
            for (int k = tid; k < n2; k += kRankThreads)
                reinterpret_cast<double2 *>(dst)[k] = reinterpret_cast<const double2 *>(ystage)[k];
            if ((n_t & 1) && tid == 0) dst[n_t - 1] = ystage[n_t - 1];
        } else {
            for (int k = tid; k < n_t; k += kRankThreads) dst[k] = ystage[k];
        }
        return;
    }
    double *__restrict__ stage = reinterpret_cast<double *>(B) + warp * (128 + 8);   // per-warp 128 outputs, padded
    const int groups = (n_t + 127) / 128;        // a warp-iteration covers 128 consecutive outputs
    const int taps = (SGW > 0) ? SGW : sg_w;
    for (int gi = warp; gi < groups; gi += kRankWarps) {
        const int k0 = gi * 128 + 4 * lane;      // first of this lane's 4 consecutive outputs (tile-relative output index)
        const int c0 = t0 - a0 + k0 - half;      // adj index of the first tap of output k0
        double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0, acc3 = 0.0;
        // s_coef holds c (SHIFT) or c / 2 (the tile then stores 2 * adj): the products are the same
        if (c0 >= 0 && c0 + taps + 3 <= A) {     // every tap in range: unguarded loads
            const AdjT *__restrict__ p = adj;
            double r0 = (double)p[aslot(c0)], r1 = (double)p[aslot(c0 + 1)], r2 = (double)p[aslot(c0 + 2)];
            if (SGW > 0) {
#pragma unroll
                for (int i = 0; i < (SGW > 0 ? SGW : 1); ++i) {
                    const double r3 = (double)p[aslot(c0 + i + 3)];
                    const double c = s_coef[i];
                    acc0 += c * r0; acc1 += c * r1; acc2 += c * r2; acc3 += c * r3;
                    r0 = r1; r1 = r2; r2 = r3;
                }
            } else {
                for (int i = 0; i < sg_w; ++i) {
                    const double r3 = (double)p[aslot(c0 + i + 3)];
                    const double c = s_coef[i];
                    acc0 += c * r0; acc1 += c * r1; acc2 += c * r2; acc3 += c * r3;
                    r0 = r1; r1 = r2; r2 = r3;
                }
            }
        } else {
            auto ld = [&](int k) -> double { return (k >= 0 && k < A) ? (double)adj[aslot(k)] : 0.0; };
            double r0 = ld(c0), r1 = ld(c0 + 1), r2 = ld(c0 + 2);
            for (int i = 0; i < taps; ++i) {
                const double r3 = ld(c0 + i + 3);
                const double c = s_coef[i];
                acc0 += c * r0; acc1 += c * r1; acc2 += c * r2; acc3 += c * r3;
                r0 = r1; r1 = r2; r2 = r3;
            }
        }
        double v[4] = {acc0, acc1, acc2, acc3};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int j = t0 + k0 + k;           // segment-relative output index
            if (k0 + k < n_t) {
                if (j < half) {                  // polynomial fit of the first sg_w adjusted values
                    double e = 0.0;
                    for (int i = 0; i < sg_w; ++i) e += edge_first[j * sg_w + i] * val(i - a0);
                    v[k] = e;
                } else if (j >= n_out - half) {
                    double e = 0.0;
                    const int jj = j - (n_out - half);
                    for (int i = 0; i < sg_w; ++i) e += edge_last[jj * sg_w + i] * val(n_out - sg_w + i - a0);
                    v[k] = e;
                }
            }
            const int e_ = 4 * lane + k;
            stage[e_ + (e_ >> 4)] = v[k];
        }
        __syncwarp();
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int e_ = k * 32 + lane;
            const int o = gi * 128 + e_;
            if (o < n_t) dst[o] = stage[e_ + (e_ >> 4)];
        }
        __syncwarp();
    }
}

// subtract_edges (frag/_adjust_wps.py:119-123): shift[s] = mean(mean(x[:e]), mean(x[-e:])) with Python's slice
// bounds: e >= n takes all of x twice, e == 0 an empty head (x[-0:] is all of x), e < 0 drops |e| samples from the
// other end.  The mean of an empty slice is 0 / 0 = NaN, and so is the shift then.
__global__ void adjust_edge_shift_kernel(const float *__restrict__ x, const long long *__restrict__ seg_off,
                                         int n_seg, int edge, double *__restrict__ shift) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seg) return;
    const long long n = seg_off[s + 1] - seg_off[s];
    const float *xs = x + seg_off[s];
    const long long e = edge;
    const long long a_end = e >= 0 ? (e < n ? e : n) : (n + e > 0 ? n + e : 0);                 // x[:e]
    const long long b_beg = e > 0 ? (n - e > 0 ? n - e : 0) : e == 0 ? 0 : (-e < n ? -e : n);  // x[-e:]
    double a = 0.0, b = 0.0;  // exact for integer-valued samples (|sum| < 2^53)
    for (long long t = 0; t < a_end; ++t) a += (double)xs[t];
    for (long long t = b_beg; t < n; ++t) b += (double)xs[t];
    shift[s] = ((a / (double)a_end) + (b / (double)(n - b_beg))) / 2.0;
}

}  // namespace ftk

using namespace ftk;

extern "C" int ftk_adjust_edge_shift_f64(const float *x, const int64_t *seg_off, int32_t n_seg,
                                         int32_t edge_size, double *shift, ftk_stream_t stream_) {
    if (n_seg == 0) return FTK_OK;
    if (!x || !seg_off || !shift || n_seg < 0) return FTK_E_INVALID;
    adjust_edge_shift_kernel<<<(n_seg + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream_)>>>(
        x, reinterpret_cast<const long long *>(seg_off), n_seg, edge_size, shift);
    FTK_CHECK_LAUNCH("adjust_edge_shift_kernel");
    return FTK_OK;
}

static int adjust_check(const float *x, const int64_t *seg_off, const int64_t *seg_out_off,
                        const int64_t *seg_run_off, int32_t n_seg, int64_t n_runs, int32_t w,
                        int32_t run_len, double *out) {
    if (!x || !seg_off || !seg_out_off || !seg_run_off || !out || n_seg < 0 || n_runs < 0) return FTK_E_INVALID;
    if (w < 2 || (w & 1) || w > 32767 || run_len < 1) return FTK_E_INVALID;
    return FTK_OK;
}

extern "C" int ftk_adjust_wps_f64(const float *x, const int64_t *seg_off, const int64_t *seg_out_off,
                                  const int64_t *seg_run_off, const double *seg_shift, int32_t n_seg,
                                  int64_t n_runs, int32_t w, int32_t use_mean, int32_t run_len,
                                  double *adj_out, uint8_t *fallback, ftk_stream_t stream_) {
    if (n_runs == 0 || n_seg == 0) return FTK_OK;
    int rc = adjust_check(x, seg_off, seg_out_off, seg_run_off, n_seg, n_runs, w, run_len, adj_out);
    if (rc != FTK_OK) return rc;
    if (!fallback) return FTK_E_INVALID;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    AdjParams P{w, use_mean, run_len};
    const int smem = kAdjBins * kAdjThreads * (int)sizeof(short) + kAdjWarps * 3 * 32 * kAdjTilePitch;
    FTK_CUDA_TRY(cudaMemsetAsync(fallback, 0, (size_t)n_runs, stream));
    const unsigned grid = (unsigned)((n_runs + kAdjThreads - 1) / kAdjThreads);
    const long long *so = reinterpret_cast<const long long *>(seg_off);
    const long long *oo = reinterpret_cast<const long long *>(seg_out_off);
    const long long *ro = reinterpret_cast<const long long *>(seg_run_off);
    int dev = 0;
    rc = ftk::current_device(&dev);
    if (rc != FTK_OK) return rc;
    // the dynamic shared-memory limit belongs to (kernel, device): raise it on every device this thread launches on
#define FTK_ADJ_LAUNCH(M, S)                                                                                   \
    do {                                                                                                       \
        static thread_local bool smem_opted_in[ftk::kMaxDevices] = {};                                         \
        if (!smem_opted_in[dev]) {                                                                             \
            FTK_CUDA_TRY(cudaFuncSetAttribute(adjust_hist_kernel<M, S>,                                         \
                                              cudaFuncAttributeMaxDynamicSharedMemorySize, smem));             \
            smem_opted_in[dev] = true;                                                                         \
        }                                                                                                      \
        adjust_hist_kernel<M, S><<<grid, kAdjThreads, smem, stream>>>(x, so, oo, ro, seg_shift, n_seg, n_runs, \
                                                                      P, adj_out, fallback);                   \
    } while (0)
    if (use_mean) { if (seg_shift) FTK_ADJ_LAUNCH(true, true); else FTK_ADJ_LAUNCH(true, false); }
    else          { if (seg_shift) FTK_ADJ_LAUNCH(false, true); else FTK_ADJ_LAUNCH(false, false); }
#undef FTK_ADJ_LAUNCH
    FTK_CHECK_LAUNCH("adjust_hist_kernel");
    return FTK_OK;
}

extern "C" int ftk_adjust_wps_generic_f64(const float *x, const int64_t *seg_off, const int64_t *seg_out_off,
                                          const int64_t *seg_run_off, const double *seg_shift, int32_t n_seg,
                                          const int64_t *run_list, int64_t n_list, int32_t w,
                                          int32_t use_mean, int32_t run_len, double *adj_out,
                                          float *scratch, ftk_stream_t stream_) {
    if (n_list == 0 || n_seg == 0) return FTK_OK;
    int rc = adjust_check(x, seg_off, seg_out_off, seg_run_off, n_seg, n_list, w, run_len, adj_out);
    if (rc != FTK_OK) return rc;
    if (!run_list || !scratch) return FTK_E_INVALID;
    AdjParams P{w, use_mean, run_len};
    adjust_generic_kernel<<<(unsigned)((n_list + 63) / 64), 64, 0, static_cast<cudaStream_t>(stream_)>>>(
        x, reinterpret_cast<const long long *>(seg_off), reinterpret_cast<const long long *>(seg_out_off),
        reinterpret_cast<const long long *>(seg_run_off), seg_shift, n_seg,
        reinterpret_cast<const long long *>(run_list), n_list, P, adj_out, scratch);
    FTK_CHECK_LAUNCH("adjust_generic_kernel");
    return FTK_OK;
}

extern "C" int ftk_savgol_f64(const double *adj, const int64_t *seg_out_off, int32_t n_seg, int64_t n_total,
                              int32_t sg_w, const double *coef, const double *edge_first,
                              const double *edge_last, double *out, ftk_stream_t stream_) {
    if (n_total == 0 || n_seg == 0) return FTK_OK;
    if (!adj || !seg_out_off || !coef || !edge_first || !edge_last || !out || n_seg < 0 || n_total < 0)
        return FTK_E_INVALID;
    if (sg_w < 1 || !(sg_w & 1) || sg_w > kAdjMaxSg || adj == out) return FTK_E_INVALID;
    const unsigned grid = (unsigned)((n_total + kSgTile - 1) / kSgTile);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const long long *oo = reinterpret_cast<const long long *>(seg_out_off);
    if (sg_w == 21)
        adjust_savgol_kernel<21><<<grid, kSgThreads, 0, stream>>>(adj, oo, n_seg, n_total, sg_w, coef, edge_first,
                                                                  edge_last, out);
    else
        adjust_savgol_kernel<0><<<grid, kSgThreads, 0, stream>>>(adj, oo, n_seg, n_total, sg_w, coef, edge_first,
                                                                 edge_last, out);
    FTK_CHECK_LAUNCH("adjust_savgol_kernel");
    return FTK_OK;
}

// One CTA per tile (tile_seg / tile_t0 / tile_n: segment, first output and output count, planned
// by the caller so that every tile needs at most a_cap adjusted values and s_cap samples).
template <typename InT>
static int launch_rank(const InT *x, const long long *so, const long long *oo, const double *seg_shift,
                       const int *tile_seg, const int *tile_t0, const int *tile_n, int64_t n_tiles, int w,
                       int sg_w, const double *coef, const double *ef, const double *el, long long sg_a,
                       long long sg_b, double sg_scale, int sg_fit32, int a_cap, int s_cap,
                       double *out, unsigned char *flag, cudaStream_t stream) {
    const unsigned grid = (unsigned)n_tiles;
#define FTK_RANK(SHIFT, SGW, MOM)                                                                                      \
    do {                                                                                                          \
        const int smem = (int)rank_smem_bytes(a_cap, s_cap, SHIFT);                                               \
        if (smem > 227 * 1024) return FTK_E_RANGE;                                                                \
        FTK_CUDA_TRY(cudaFuncSetAttribute(adjust_rank_kernel<InT, SHIFT, SGW, MOM>,                                \
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, smem));                    \
        adjust_rank_kernel<InT, SHIFT, SGW, MOM><<<grid, kRankThreads, smem, stream>>>(                            \
            x, so, oo, seg_shift, tile_seg, tile_t0, tile_n, w, sg_w, coef, ef, el, sg_a, sg_b, sg_scale, sg_fit32,\
            a_cap, s_cap, out, flag);                                                                                    \
    } while (0)
    if (seg_shift) {
        if (sg_w == 0) FTK_RANK(true, -1, false); else if (sg_w == 21) FTK_RANK(true, 21, false); else FTK_RANK(true, 0, false);
    } else if (sg_w != 0 && sg_scale != 0.0) {       // exact sliding-moment smoothing
        if (sg_w == 21) FTK_RANK(false, 21, true); else FTK_RANK(false, 0, true);
    } else {
        if (sg_w == 0) FTK_RANK(false, -1, false); else if (sg_w == 21) FTK_RANK(false, 21, false); else FTK_RANK(false, 0, false);
    }
#undef FTK_RANK
    FTK_CHECK_LAUNCH("adjust_rank_kernel");
    return FTK_OK;
}

extern "C" int ftk_adjust_rank_f64(const void *x, int32_t x_kind, const int64_t *seg_off, const int64_t *seg_out_off,
                                   const double *seg_shift, int32_t n_seg, const int32_t *tile_seg,
                                   const int32_t *tile_t0, const int32_t *tile_n, int64_t n_tiles, int32_t w,
                                   int32_t sg_w, const double *coef, const double *edge_first,
                                   const double *edge_last, int64_t sg_num_a, int64_t sg_num_b, int64_t sg_den,
                                   int32_t a_cap, int32_t s_cap, double *out,
                                   uint8_t *tile_flag, ftk_stream_t stream_) {
    if (n_tiles == 0 || n_seg == 0) return FTK_OK;
    if (!x || !seg_off || !seg_out_off || !tile_seg || !tile_t0 || !tile_n || !out || !tile_flag) return FTK_E_INVALID;
    if (n_seg < 0 || n_tiles < 0 || n_tiles > INT32_MAX || (x_kind != 0 && x_kind != 1)) return FTK_E_INVALID;
    if (w < 2 || (w & 1) || w > 32767) return FTK_E_INVALID;
    if (sg_w != 0 && (sg_w < 1 || !(sg_w & 1) || sg_w > kAdjMaxSg || !coef || !edge_first || !edge_last)) return FTK_E_INVALID;
    if (a_cap < 1 || a_cap > 32 * kRankThreads || s_cap < a_cap + w || s_cap > 65535 - 64) return FTK_E_RANGE;
    // exact sliding-moment smoothing: only when every intermediate provably fits (|2 adj| < 2^17)
    double sg_scale = 0.0;
    int sg_fit32 = 0;                    // the final combination a * S0 + b * M2 itself fits int32
    if (sg_w > 0 && sg_den != 0) {
        if (sg_den < 0) return FTK_E_INVALID;
        const long long h = sg_w >> 1;
        const long long s2 = h * (h + 1) * (2 * h + 1) / 3;                 // sum of i^2 over the window
        const long long bound = 1ll << 17;
        const long long aa = sg_num_a < 0 ? -sg_num_a : sg_num_a, bb = sg_num_b < 0 ? -sg_num_b : sg_num_b;
        // every term of the moment updates summed in absolute value stays inside int32, the final
        // combination inside 2^53 (exactly representable)
        if ((s2 + 2 * h * (h + 1) + sg_w + 2 * (h + 1) * (h + 1)) * bound < (1ll << 31) && aa < (1ll << 31) &&
            bb < (1ll << 31) && (aa * sg_w + bb * s2) < (1ll << 36))
        {
            sg_scale = 0.5 / (double)sg_den;
            sg_fit32 = (aa * sg_w + bb * s2) * bound < (1ll << 31);
        }
    }
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    FTK_CUDA_TRY(cudaMemsetAsync(tile_flag, 0, (size_t)n_tiles, stream));
    const long long *so = reinterpret_cast<const long long *>(seg_off);
    const long long *oo = reinterpret_cast<const long long *>(seg_out_off);
    if (x_kind == 0)
        return launch_rank<float>(static_cast<const float *>(x), so, oo, seg_shift, tile_seg, tile_t0, tile_n, n_tiles,
                                  w, sg_w, coef, edge_first, edge_last, sg_num_a, sg_num_b, sg_scale, sg_fit32, a_cap, s_cap, out,
                                  tile_flag, stream);
    return launch_rank<int>(static_cast<const int *>(x), so, oo, seg_shift, tile_seg, tile_t0, tile_n, n_tiles,
                            w, sg_w, coef, edge_first, edge_last, sg_num_a, sg_num_b, sg_scale, sg_fit32, a_cap, s_cap, out,
                            tile_flag, stream);
}
