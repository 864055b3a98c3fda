// Windowed Protection Score on sm_100a.
//
// Replaces the reference's O(len x n_frag) per-position loop
// (frag/_wps.py:176-188 -> _single_nt_wps, frag/_wps.py:25-53) with a
// fragment-event scatter into a shared-memory difference array followed by a
// block prefix scan.  For window [c-a, c+b] (even W: a=W/2, b=W/2-1; odd W:
// a=b=(W-1)/2 around c' = c - ((c-a)&1), which is what np.rint's
// round-half-even does at frag/_wps.py:177-178) a fragment (fs, fe), L=fe-fs:
//   L <= W : contributes -1 on [fs-b, fe+a]               (either end inside)
//   L >  W : -1 on [fs-b, fs+a], +1 on [fs+a+1, fe-b-1], -1 on [fe-b, fe+a]
// i.e. D[fs-b]-=1, D[fe+a+1]+=1 and, iff L>W, D[fs+a+1]+=2, D[fe-b]-=2;
// WPS = inclusive prefix sum of D.  Events left of the tile are clamped onto
// its first slot (they belong to the prefix), events right of it are dropped,
// so tiles are independent: no inter-CTA carry, no collective.
//
// Roofline: HBM.  Algorithmic bytes = 9 B per fragment (start, stop int32 +
// mapq uint8) + 4 B per output position (DESIGN.md §4).
#include "ftk_common.cuh"

namespace ftk {

constexpr int kWpsCap = 5120;                    // smem slots per tile
static_assert(FTK_WPS_TILE < kWpsCap, "one guard slot for odd windows");

// ---------------------------------------------------------------------------
// Tile parameters, the fragment scatter and the score stores
// ---------------------------------------------------------------------------
struct WpsParams {
    int window, a, b;       // window [c-a, c+b]
    int len_lo;             // fragment-length window as an unsigned range test
    unsigned len_span;
    int min_mapq;
    int max_len;
};

struct TileCtx {
    int p0, len, mid_lo, g0, glen;
    int zl_excl;            // fused coverage: a zero-length fragment sitting exactly here is not in the stream
    int eb;                 // b + g0: first event slot of a fragment = fs - eb
    unsigned mid_span;
    bool need_mid;          // tile-uniform: the midpoint test can exclude a contributing fragment
};

template <bool ODD>
__device__ __forceinline__ TileCtx make_tile_ctx(const WpsParams &P, int p0, int len, int mid_lo, int mid_hi) {
    TileCtx t;
    t.p0 = p0; t.len = len; t.mid_lo = mid_lo;
    t.zl_excl = INT32_MIN;
    t.mid_span = (mid_hi > mid_lo) ? (unsigned)(mid_hi - mid_lo) : 0u;
    // grid of the symmetric-window score G: one extra slot on the left for odd W
    t.g0 = ODD ? p0 - 1 : p0;
    t.glen = ODD ? len + 1 : len;
    t.eb = P.b + t.g0;
    // The interval's padded fetch window [S-max_len, E+max_len) (frag/_wps.py:156-157) contains
    // the midpoint of every fragment that can touch the interval whenever W + 2 <= max_len, so
    // the test is only needed for wide windows or where the window was clamped to the contig.
    t.need_mid = (P.window + 2 > P.max_len) || ((long long)mid_hi < (long long)p0 + len + P.max_len) ||
                 ((long long)mid_lo > (long long)p0 - P.max_len);
    return t;
}

// One fragment's events -> shared atomics (2, or 4 when L > W).  The predicate is the
// reference's (utils/_frag_generator.py:117-123; mapq io/alignment.py:291) as unsigned range
// tests: min_len <= L <= max_len and mid_lo <= (fs+fe)//2 < mid_hi (L < 0 never passes).
// Event slots relative to the tile: e0 = fs-b-g0 (-1), e0+W (+2), e0+L (-2), e0+L+W (+1).
__device__ __forceinline__ void wps_scatter(int *__restrict__ D, const WpsParams &P, const TileCtx &T,
                                            int fs, int fe, int q) {
    const int L = fe - fs;
    bool pass = (q >= P.min_mapq) && ((unsigned)(L - P.len_lo) <= P.len_span);
    if (T.need_mid) pass = pass && ((unsigned)(fs + (L >> 1) - T.mid_lo) < T.mid_span);
    if (!pass) return;
    const int e0 = fs - T.eb;
    const int e3 = e0 + L + P.window;
    if (e0 >= 0 && e3 < T.glen) {  // interior fragment (97 % at 30x): no clamping
        int *__restrict__ p = D + e0;
        atomicAdd(p, -1);
        atomicAdd(p + (L + P.window), 1);
        if (L > P.window) {
            atomicAdd(p + P.window, 2);
            atomicAdd(p + L, -2);
        }
        return;
    }
    if (e3 <= 0 || e0 >= T.glen) return;  // cancels on slot 0 / entirely right of the tile
    atomicAdd(&D[max(e0, 0)], -1);
    if (e3 < T.glen) atomicAdd(&D[e3], 1);
    if (L > P.window) {
        const int e1 = e0 + P.window, e2 = e0 + L;
        if (e1 < T.glen) atomicAdd(&D[max(e1, 0)], 2);
        if (e2 < T.glen) atomicAdd(&D[max(e2, 0)], -2);
    }
}

// Store four consecutive scores.  int32: one 128-bit streaming store.  int16 (halves the
// device->host bytes of the end-to-end path): one 64-bit store + a range check that raises
// *overflow so the caller can redo the launch in int32 (|WPS| <= local depth, so this needs a
// > 32767-fold pile-up).
__device__ __forceinline__ void store4(int32_t *p, const int4 &r, int *) {
    st_stream4(reinterpret_cast<int4 *>(p), r);
}
__device__ __forceinline__ void store4(int16_t *p, const int4 &r, int *overflow) {
    const unsigned bad = ((unsigned)(r.x + 32768) | (unsigned)(r.y + 32768) | (unsigned)(r.z + 32768) |
                          (unsigned)(r.w + 32768)) >> 16;
    if (bad) atomicOr(overflow, 1);
    int2 v;
    v.x = (r.x & 0xffff) | (r.y << 16);
    v.y = (r.z & 0xffff) | (r.w << 16);
    asm volatile("st.global.L1::no_allocate.v2.s32 [%0], {%1,%2};" :: "l"(p), "r"(v.x), "r"(v.y) : "memory");
}
// int8 (a quarter of the int32 bytes on the wire; fits whenever the local depth stays below 128):
// one 32-bit store + the same overflow protocol.
__device__ __forceinline__ void store4(int8_t *p, const int4 &r, int *overflow) {
    const unsigned bad = ((unsigned)(r.x + 128) | (unsigned)(r.y + 128) | (unsigned)(r.z + 128) |
                          (unsigned)(r.w + 128)) >> 8;
    if (bad) atomicOr(overflow, 1);
    const int v = (r.x & 0xff) | ((r.y & 0xff) << 8) | ((r.z & 0xff) << 16) | (r.w << 24);
    asm volatile("st.global.L1::no_allocate.s32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void store1(int8_t *p, int v, int *overflow) {
    if ((unsigned)(v + 128) >> 8) atomicOr(overflow, 1);
    *p = (int8_t)v;
}
__device__ __forceinline__ void store1(int32_t *p, int v, int *) { *p = v; }
__device__ __forceinline__ void store1(int16_t *p, int v, int *overflow) {
    if ((unsigned)(v + 32768) >> 16) atomicOr(overflow, 1);
    *p = (int16_t)v;
}

// ---------------------------------------------------------------------------
// The WPS kernel: persistent, warp-specialised, TMA-fed.
//
// A producer lane runs ahead of the consumer warps: it reads the next tile's descriptor and
// fragment range and issues 1-D bulk async copies (cp.async.bulk ... mbarrier::complete_tx::bytes,
// SASS UBLKCP) of the start / stop / mapq slices into a shared-memory staging buffer.  The
// consumers wait on the buffer's "full" mbarrier, turn the staged fragments into shared atomics,
// release the buffer through its "empty" mbarrier, then scan and store the tile - while the next
// tile's bytes are already in flight.  HBM latency is therefore never exposed to the compute warps.
//
// The consumer warps form groups of four, each with its own difference array, its own staging
// buffer and its own named barrier; producer warp p feeds groups 2p and 2p+1 alternately.  While
// one group scans and stores its tile the other one is scattering the next, so the barrier / phase
// latency of a tile is overlapped inside the CTA instead of across CTAs.  Both shapes keep six
// tiles in flight per SM:
//   * plain WPS: two groups and one producer warp per CTA, three CTAs per SM;
//   * fused pass (FUSE): six groups and three producer warps, ONE CTA per SM.  The SM's shared
//     memory is then one allocation: the 2 KB the two extra CTAs lose to the per-CTA reservation
//     plus the slack at the end leave room for a CTA-wide 1024-bin length histogram, which is what
//     lets the step make ONE pass over the fragments:
//       - per-interval coverage (frag/_coverage.py:117-130, midpoint policy): a fragment's midpoint
//         lies in exactly one tile of an interval, so the count of an interval is the sum of its
//         tiles' counts - a register count per lane, one shuffle reduction and one 64-bit atomic
//         per warp and tile;
//       - pooled length histogram of the counted fragments (frag/_frag_length.py:147-153): shared
//         atomics on the CTA's histogram, flushed once with 64-bit global atomics when the CTA
//         ends (a CTA sees < 2^31 fragments: n_frag <= INT32_MAX).
//     The coverage predicate has its own length window and mapq cut; the staged range is widened
//     on the left so that every fragment whose midpoint can fall into the tile is staged.
// ---------------------------------------------------------------------------
constexpr int kStreamFrags = 1920;                   // fragments per staging buffer (multiple of 16)
constexpr int kGroupWarps = 4;
constexpr int kGroupThreads = kGroupWarps * 32;
constexpr int kScanHalf = kWpsCap / 2;               // slots scanned per pass
constexpr int kWpsSpan = kScanHalf / kGroupWarps;    // positions per warp and pass
constexpr int kWpsIters = kWpsSpan / 128;            // int4 groups per lane and pass
static_assert(2 * kWpsIters * kGroupThreads * 4 == kWpsCap, "tile must split evenly");
constexpr int kPlainGroups = 2;
constexpr int kFusedGroups = 6;
constexpr int kFuseBins = 1024;                      // lengths below this are privatised in shared memory

template <int GROUPS> constexpr int kStreamThreads = GROUPS * kGroupThreads + 32 * (GROUPS / 2);
template <int GROUPS> constexpr int kStreamCtasPerSm = 6 / GROUPS;

struct __align__(16) StreamDesc {
    int tile;        // -1: no more work
    int p0, len, mid_lo, mid_hi;
    int n;           // staged fragments (multiple of 16, may be 0)
    int first, last; // first / last chunk of its tile
    int ivl;         // interval the tile belongs to (fused coverage counts); bit 31 = its first tile
    long long out_off;
    long long tail_lo, tail_hi;  // ragged end of the contig, read straight from global (rare)
};

template <int GROUPS, bool FUSE>
struct __align__(128) StreamSmem {
    int D[GROUPS][kWpsCap];
    int start[GROUPS][kStreamFrags];
    int stop[GROUPS][kStreamFrags];
    unsigned char mapq[GROUPS][kStreamFrags];
    StreamDesc desc[GROUPS];
    unsigned long long full_bar[GROUPS];
    unsigned long long empty_bar[GROUPS];
    int warp_tot[GROUPS][kGroupWarps];
    int hist[FUSE ? kFuseBins : 1];
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(void *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(void *bar, unsigned parity) {
    const uint32_t addr = smem_u32(bar);
    unsigned ok;
    do {
        // the suspend-time hint lets the hardware park the warp until the phase flips instead of
        // returning every few hundred cycles: 12 % of the kernel's issued instructions were this loop
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(addr), "r"(parity), "r"(1000000u) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void mbar_arrive(void *bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}"
                 :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(void *bar, unsigned bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}"
                 :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// 1-D TMA: global -> shared, completion counted in bytes on an mbarrier
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, void *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void group_sync(int g) {
    asm volatile("bar.sync %0, %1;" :: "r"(1 + g), "n"(kGroupThreads) : "memory");
}

// Block prefix scan of D and the store of the tile by one 4-warp group, in two passes of kScanHalf
// slots.  Lane owns int4 groups, warp owns a contiguous span, one barrier for the warp totals of a
// pass; the stores stay coalesced and the register footprint stays at 5 int4.
template <bool ODD, typename OutT>
__device__ __forceinline__ void wps_scan_store_group(int *__restrict__ D, int *__restrict__ warp_tot,
                                                     const WpsParams &P, const TileCtx &T,
                                                     OutT *__restrict__ dst, int *overflow, int gt, int g) {
    const int lane = gt & 31, warp = gt >> 5;
    const bool aligned = ((reinterpret_cast<uintptr_t>(dst) & (4 * sizeof(OutT) - 1)) == 0);
    int base_carry = 0;
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
        int4 v[kWpsIters];
        int carry = 0;
        const int span0 = half * kScanHalf + warp * kWpsSpan;
#pragma unroll
        for (int j = 0; j < kWpsIters; ++j) {
            const int base = span0 + j * 128 + lane * 4;
            int4 d = *reinterpret_cast<const int4 *>(&D[base]);
            d.y += d.x; d.z += d.y; d.w += d.z;
            int t = d.w;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                int n = __shfl_up_sync(0xffffffffu, t, off);
                if (lane >= off) t += n;
            }
            const int excl = t - d.w + carry;
            v[j] = make_int4(d.x + excl, d.y + excl, d.z + excl, d.w + excl);
            carry += __shfl_sync(0xffffffffu, t, 31);
        }
        if (lane == 0) warp_tot[warp] = carry;
        group_sync(g);
        int offset = base_carry, total = 0;
#pragma unroll
        for (int w = 0; w < kGroupWarps; ++w) {
            const int wt = warp_tot[w];
            offset += (w < warp) ? wt : 0;
            total += wt;
        }
        base_carry += total;
#pragma unroll
        for (int j = 0; j < kWpsIters; ++j) {
            const int base = span0 + j * 128 + lane * 4;
            const int4 r = make_int4(v[j].x + offset, v[j].y + offset, v[j].z + offset, v[j].w + offset);
            if (ODD) {
                *reinterpret_cast<int4 *>(&D[base]) = r;      // stage G; gathered below
            } else if (aligned && base + 3 < T.len) {
                store4(dst + base, r, overflow);
            } else {
                if (base + 0 < T.len) store1(dst + base + 0, r.x, overflow);
                if (base + 1 < T.len) store1(dst + base + 1, r.y, overflow);
                if (base + 2 < T.len) store1(dst + base + 2, r.z, overflow);
                if (base + 3 < T.len) store1(dst + base + 3, r.w, overflow);
            }
        }
        group_sync(g);   // warp_tot is rewritten by the next pass / D by the next tile
    }
    if (ODD) {
        // odd W: out[c] = G[c - ((c - a) & 1)]
        for (int k = gt; k < T.len; k += kGroupThreads) {
            const int c = T.p0 + k;
            store1(dst + k, D[c - ((c - P.a) & 1) - T.g0], overflow);
        }
        group_sync(g);
    }
}

struct CovParams {
    int len_lo;
    unsigned len_span;
    int min_mapq;
    int n_bins;             // 0: no histogram
};

// Coverage / histogram side of one staged fragment: the stream of region [p0, p0+len) under the
// midpoint policy (io/alignment.py:270-302 overlap rows: stop > S; utils/_frag_generator.py:117-123).
__device__ __forceinline__ void cov_visit(int *__restrict__ hist_s, unsigned long long *__restrict__ ghist,
                                          const CovParams &C, const TileCtx &T, int fs, int fe, int q, int &cnt) {
    const int L = fe - fs;
    // tabix overlap "stop > S": only a zero-length row sitting on the interval's own start fails it
    // once its midpoint is inside (zl_excl = S on the interval's first tile, INT32_MIN elsewhere)
    const bool pass = (q >= C.min_mapq) & ((unsigned)(L - C.len_lo) <= C.len_span) &
                      ((unsigned)(fs + (L >> 1) - T.p0) < (unsigned)T.len) & ((L > 0) | (fs != T.zl_excl));
    if (pass) {
        ++cnt;
        if (L < C.n_bins) {
            if (L < kFuseBins) atomicAdd(&hist_s[L], 1);
            else atomicAdd(&ghist[L], 1ull);
        }
    }
}

struct TileRec {
    int64_t lo, hi;
    long long ooff;
    int tile, p0, len, mlo, mhi, ivl;
};

template <bool ODD, typename OutT, int GROUPS, bool FUSE>
__global__ void __launch_bounds__(kStreamThreads<GROUPS>, kStreamCtasPerSm<GROUPS>)
wps_stream_kernel(const int32_t *__restrict__ frag_start, const int32_t *__restrict__ frag_stop,
                  const uint8_t *__restrict__ frag_mapq, int64_t n_frag,
                  const int32_t *__restrict__ tile_p0, const int32_t *__restrict__ tile_len,
                  const int32_t *__restrict__ tile_mid_lo, const int32_t *__restrict__ tile_mid_hi,
                  const int64_t *__restrict__ tile_out_off, const int32_t *__restrict__ tile_ivl,
                  const int64_t *__restrict__ ranges, int n_tiles, WpsParams P, CovParams C,
                  OutT *__restrict__ out, int *__restrict__ overflow,
                  unsigned long long *__restrict__ counts, unsigned long long *__restrict__ ghist) {
    constexpr int kConsumerThreads = GROUPS * kGroupThreads;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    StreamSmem<GROUPS, FUSE> &S = *reinterpret_cast<StreamSmem<GROUPS, FUSE> *>(smem_raw);
    const int tid = threadIdx.x;

    if (tid == 0) {
#pragma unroll
        for (int g = 0; g < GROUPS; ++g) {
            mbar_init(&S.full_bar[g], 1);
            mbar_init(&S.empty_bar[g], 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (FUSE) {
        for (int b = tid; b < kFuseBins; b += kStreamThreads<GROUPS>) S.hist[b] = 0;
    }
    __syncthreads();

    if (tid < kConsumerThreads) {
        // ========================= consumer groups =========================
        const int g = tid / kGroupThreads;
        const int gt = tid - g * kGroupThreads;
        int *__restrict__ D = S.D[g];
        unsigned phase = 0;
        int cnt = 0;
        TileCtx T = make_tile_ctx<ODD>(P, 0, 0, 0, 0);
        for (;;) {
            mbar_wait(&S.full_bar[g], phase);
            const StreamDesc d = S.desc[g];
            if (d.tile < 0) break;
            if (d.first) {
                T = make_tile_ctx<ODD>(P, d.p0, d.len, d.mid_lo, d.mid_hi);
                if (FUSE && d.ivl < 0) T.zl_excl = d.p0;
                cnt = 0;
#pragma unroll
                for (int j = 0; j < kWpsCap / (4 * kGroupThreads); ++j)
                    reinterpret_cast<int4 *>(D)[j * kGroupThreads + gt] = make_int4(0, 0, 0, 0);
                group_sync(g);
            }
            const int nvec = d.n >> 2;
            const int4 *__restrict__ vs = reinterpret_cast<const int4 *>(S.start[g]);
            const int4 *__restrict__ ve = reinterpret_cast<const int4 *>(S.stop[g]);
            const uchar4 *__restrict__ vq = reinterpret_cast<const uchar4 *>(S.mapq[g]);
            for (int v = gt; v < nvec; v += kGroupThreads) {
                const int4 s = vs[v], e = ve[v];
                const uchar4 q = frag_mapq ? vq[v] : make_uchar4(255, 255, 255, 255);
                wps_scatter(D, P, T, s.x, e.x, q.x);
                wps_scatter(D, P, T, s.y, e.y, q.y);
                wps_scatter(D, P, T, s.z, e.z, q.z);
                wps_scatter(D, P, T, s.w, e.w, q.w);
                if (FUSE) {
                    cov_visit(S.hist, ghist, C, T, s.x, e.x, q.x, cnt);
                    cov_visit(S.hist, ghist, C, T, s.y, e.y, q.y, cnt);
                    cov_visit(S.hist, ghist, C, T, s.z, e.z, q.z, cnt);
                    cov_visit(S.hist, ghist, C, T, s.w, e.w, q.w, cnt);
                }
            }
            if (d.tail_hi > d.tail_lo) {
                const int64_t i = d.tail_lo + gt;
                if (i < d.tail_hi) {
                    const int fs = __ldcs(frag_start + i), fe = __ldcs(frag_stop + i);
                    const int q = frag_mapq ? (int)__ldcs(frag_mapq + i) : 255;
                    wps_scatter(D, P, T, fs, fe, q);
                    if (FUSE) cov_visit(S.hist, ghist, C, T, fs, fe, q, cnt);
                }
            }
            group_sync(g);                                   // scatter done; the staging buffer is free
            if (gt == 0) mbar_arrive(&S.empty_bar[g]);
            if (d.last) {
                if (FUSE) {
                    const int c = __reduce_add_sync(0xffffffffu, cnt);
                    if ((gt & 31) == 0 && c) atomicAdd(&counts[d.ivl & 0x7fffffff], (unsigned long long)c);
                }
                wps_scan_store_group<ODD>(D, S.warp_tot[g], P, T, out + d.out_off, overflow, gt, g);
            }
            phase ^= 1u;
        }
        if (FUSE && C.n_bins > 0) {
            // all consumer groups are done: flush the CTA's histogram (the producers have exited)
            asm volatile("bar.sync %0, %1;" :: "n"(GROUPS + 1), "n"(kConsumerThreads) : "memory");
            const int nb = min(C.n_bins, kFuseBins);
            for (int b = tid; b < nb; b += kConsumerThreads) {
                const int v = S.hist[b];
                if (v) atomicAdd(&ghist[b], (unsigned long long)v);
            }
        }
        return;
    }

    // ============ producer warps (one elected lane each, two groups per producer) ============
    const int pt = tid - kConsumerThreads;
    if ((pt & 31) == 0) {
        const int p = pt >> 5;
        // bit sub: phase of group 2p + sub (a runtime-indexed array would live in local memory)
        unsigned ph = 0u;
        const int64_t n16 = n_frag & ~(int64_t)15;
        // the CTA's k-th tile is blockIdx.x + k * gridDim.x and goes to group k % GROUPS; this
        // producer's j-th tile is k = GROUPS * (j / 2) + 2p + (j & 1)
        auto fetch = [&](int j, TileRec &r) -> bool {
            const int64_t k = GROUPS * (int64_t)(j >> 1) + 2 * p + (j & 1);
            const int64_t tile = blockIdx.x + k * (int64_t)gridDim.x;
            if (tile >= n_tiles) return false;
            r.tile = (int)tile;
            r.lo = ranges[2 * tile]; r.hi = ranges[2 * tile + 1];
            r.p0 = tile_p0[tile]; r.len = tile_len[tile];
            r.mlo = tile_mid_lo[tile]; r.mhi = tile_mid_hi[tile];
            r.ooff = tile_out_off[tile];
            r.ivl = FUSE ? tile_ivl[tile] : 0;
            return true;
        };
        TileRec r, rn;
        bool have = fetch(0, r);
        for (int j = 0; have; ++j) {
            // the next tile's descriptor loads are in flight while this tile waits for its buffer
            const bool have_next = fetch(j + 1, rn);
            const int sub = j & 1;
            const int g = 2 * p + sub;
            const int64_t lo16 = r.lo & ~(int64_t)15;
            int64_t hi16 = (r.hi + 15) & ~(int64_t)15;
            if (hi16 > n16) hi16 = n16;
            if (hi16 < lo16) hi16 = lo16;
            const int64_t t_lo = (hi16 > lo16) ? hi16 : lo16;
            const bool has_tail = r.hi > t_lo;
            const int64_t span = hi16 - lo16;
            const int n_chunks = span > 0 ? (int)((span + kStreamFrags - 1) / kStreamFrags) : 1;
            for (int c = 0; c < n_chunks; ++c) {
                mbar_wait(&S.empty_bar[g], ((ph >> sub) & 1u) ^ 1u);
                const int64_t c0 = lo16 + (int64_t)c * kStreamFrags;
                const int n = (int)min((int64_t)kStreamFrags, hi16 - c0);
                StreamDesc &d = S.desc[g];
                d.tile = r.tile; d.p0 = r.p0; d.len = r.len; d.mid_lo = r.mlo; d.mid_hi = r.mhi;
                d.n = n > 0 ? n : 0;
                d.first = (c == 0); d.last = (c == n_chunks - 1);
                d.ivl = r.ivl;
                d.out_off = r.ooff;
                d.tail_lo = (d.last && has_tail) ? t_lo : 0;
                d.tail_hi = (d.last && has_tail) ? r.hi : 0;
                if (n > 0) {
                    const unsigned bytes = (unsigned)n * (frag_mapq ? 9u : 8u);
                    mbar_arrive_expect_tx(&S.full_bar[g], bytes);
                    bulk_g2s(S.start[g], frag_start + c0, (unsigned)n * 4u, &S.full_bar[g]);
                    bulk_g2s(S.stop[g], frag_stop + c0, (unsigned)n * 4u, &S.full_bar[g]);
                    if (frag_mapq) bulk_g2s(S.mapq[g], frag_mapq + c0, (unsigned)n, &S.full_bar[g]);
                } else {
                    mbar_arrive(&S.full_bar[g]);
                }
                ph ^= 1u << sub;
            }
            r = rn;
            have = have_next;
        }
#pragma unroll 1
        for (int sub = 0; sub < 2; ++sub) {
            const int g = 2 * p + sub;
            mbar_wait(&S.empty_bar[g], ((ph >> sub) & 1u) ^ 1u);
            S.desc[g].tile = -1;
            mbar_arrive(&S.full_bar[g]);
        }
    }
}

}  // namespace ftk

extern "C" int64_t ftk_wps_plan_tiles(const int64_t *ivl_start, const int64_t *ivl_stop,
                                      const int64_t *ivl_out_off, int64_t n_ivl,
                                      int64_t chrom_size, int32_t max_len,
                                      int32_t *tile_p0, int32_t *tile_len,
                                      int32_t *tile_mid_lo, int32_t *tile_mid_hi,
                                      int64_t *tile_out_off) {
    if (n_ivl < 0 || (n_ivl > 0 && (!ivl_start || !ivl_stop || !ivl_out_off))) return FTK_E_INVALID;
    if (chrom_size < 0 || chrom_size > INT32_MAX || max_len < 0) return FTK_E_RANGE;
    constexpr int64_t cap4 = FTK_WPS_TILE & ~3;  // keep int4-aligned pieces
    int64_t n_tiles = 0;
    for (int64_t k = 0; k < n_ivl; ++k) {
        const int64_t S = ivl_start[k], E = ivl_stop[k];
        if (E <= S) continue;  // degenerate interval: no output (frag/_wps.py:145-152)
        if (S < INT32_MIN / 2 || E > INT32_MAX) return FTK_E_RANGE;
        // frag/_wps.py:156-157 : padded fetch window = midpoint predicate of this interval
        int64_t mlo = S - max_len; if (mlo < 0) mlo = 0;
        int64_t mhi = E + max_len; if (mhi > chrom_size) mhi = chrom_size;
        const int64_t len = E - S;
        const int64_t pieces = (len + cap4 - 1) / cap4;
        int64_t piece = (len + pieces - 1) / pieces;
        piece = (piece + 3) & ~(int64_t)3;
        for (int64_t s = 0; s < len; s += piece) {
            if (tile_p0) {
                tile_p0[n_tiles] = (int32_t)(S + s);
                tile_len[n_tiles] = (int32_t)((len - s < piece) ? (len - s) : piece);
                tile_mid_lo[n_tiles] = (int32_t)mlo;
                tile_mid_hi[n_tiles] = (int32_t)mhi;
                tile_out_off[n_tiles] = ivl_out_off[k] + s;
            }
            ++n_tiles;
        }
    }
    return n_tiles;
}

static int wps_check_args(const int32_t *frag_start, const int32_t *frag_stop, int64_t n_frag,
                          const int32_t *tile_p0, const int32_t *tile_len, int64_t n_tiles,
                          int32_t window_size, int32_t max_len, const int64_t *scratch) {
    if (n_frag < 0 || n_tiles < 0 || window_size < 1) return FTK_E_INVALID;
    if (!tile_p0 || !tile_len || !scratch) return FTK_E_INVALID;
    if (n_frag > 0 && (!frag_start || !frag_stop)) return FTK_E_INVALID;
    // the reference requires an integer max_length (frag/_wps.py:156 round(start - max_length))
    if (max_len == FTK_NONE || max_len < 0) return FTK_E_INVALID;
    if (n_tiles > INT32_MAX / 2) return FTK_E_RANGE;
    return FTK_OK;
}

// Per-tile fragment index range [lo, hi): a superset of the fragments with any event inside the tile.
// left_reach: how far left of p0 - 1 a fragment may start and still matter to the tile; a fragment's first
// event sits at fs - b and must be < p0 + len.
static int launch_tile_ranges(const int32_t *frag_start, int64_t n_frag, const int32_t *tile_p0,
                              const int32_t *tile_len, int64_t n_tiles, int32_t window_size,
                              int64_t left_reach, int64_t *scratch, cudaStream_t stream,
                              unsigned long long *zero_a = nullptr, int64_t n_zero_a = 0,
                              unsigned long long *zero_b = nullptr, int64_t n_zero_b = 0) {
    const bool odd = (window_size & 1) != 0;
    const int a = odd ? (window_size - 1) / 2 : window_size / 2;
    const int b = odd ? a : a - 1;
    if (left_reach > INT32_MAX / 2) left_reach = INT32_MAX / 2;
    return ftk::launch_candidate_ranges(frag_start, n_frag, tile_p0, tile_len, true, n_tiles, 1 + left_reach, b,
                                        scratch, stream, zero_a, n_zero_a, zero_b, n_zero_b);
}

static int64_t wps_left_reach(int32_t window_size, int32_t max_len) {
    // last event of a fragment sits at fe+a+1 <= fs+max_len+a+1; it must be > g0 >= p0-1
    const int a = (window_size & 1) ? (window_size - 1) / 2 : window_size / 2;
    return (int64_t)a + (int64_t)max_len;
}

extern "C" int ftk_wps_tile_ranges(const int32_t *frag_start, int64_t n_frag,
                                   const int32_t *tile_p0, const int32_t *tile_len, int64_t n_tiles,
                                   int32_t window_size, int32_t max_len, int64_t *scratch,
                                   ftk_stream_t stream_) {
    if (n_tiles == 0) return FTK_OK;
    int rc = wps_check_args(frag_start, frag_start, n_frag, tile_p0, tile_len, n_tiles, window_size, max_len, scratch);
    if (rc != FTK_OK) return rc;
    return launch_tile_ranges(frag_start, n_frag, tile_p0, tile_len, n_tiles, window_size,
                              wps_left_reach(window_size, max_len), scratch, static_cast<cudaStream_t>(stream_));
}

// SM count of the current device, which is returned in *dev
static int device_sm_count(int *sm, int *dev) {
    static thread_local int sm_count[ftk::kMaxDevices] = {0};
    int rc = ftk::current_device(dev);
    if (rc != FTK_OK) return rc;
    if (!sm_count[*dev])
        FTK_CUDA_TRY(cudaDeviceGetAttribute(&sm_count[*dev], cudaDevAttrMultiProcessorCount, *dev));
    *sm = sm_count[*dev];
    return FTK_OK;
}

struct WpsLaunch {
    const int32_t *frag_start, *frag_stop; const uint8_t *frag_mapq; int64_t n_frag;
    const int32_t *tile_p0, *tile_len, *tile_mid_lo, *tile_mid_hi; const int64_t *tile_out_off;
    const int32_t *tile_ivl; int64_t n_tiles; const int64_t *ranges;
    ftk::WpsParams P; ftk::CovParams C;
    int *overflow; unsigned long long *counts, *hist;
    cudaStream_t stream;
};

template <bool ODD, typename OutT, int GROUPS, bool FUSE>
static int launch_stream(const WpsLaunch &a, OutT *out) {
    using namespace ftk;
    using Smem = StreamSmem<GROUPS, FUSE>;
    constexpr int ctas_per_sm = kStreamCtasPerSm<GROUPS>;
    static_assert(sizeof(Smem) <= 227 * 1024, "a CTA may own at most 227 KB of shared memory on sm_100a");
    static_assert(ctas_per_sm * (sizeof(Smem) + 1024) <= 228 * 1024,
                  "the resident CTAs, with the 1 KB reserved for each, must fit the SM's 228 KB");
    int sm = 0, dev = 0;
    int rc = device_sm_count(&sm, &dev);
    if (rc != FTK_OK) return rc;
    // the dynamic shared-memory limit belongs to (kernel, device): raise it on every device this thread launches on
    static thread_local bool smem_opted_in[kMaxDevices] = {};
    const int smem = (int)sizeof(Smem);
    if (!smem_opted_in[dev]) {
        FTK_CUDA_TRY(cudaFuncSetAttribute(wps_stream_kernel<ODD, OutT, GROUPS, FUSE>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        smem_opted_in[dev] = true;
    }
    // persistent CTAs; a plain-WPS CTA is launched only when there are two tiles for its two groups
    int64_t grid = (int64_t)sm * ctas_per_sm;
    const int64_t max_grid = GROUPS == kPlainGroups ? (a.n_tiles + 1) / 2 : a.n_tiles;
    if (grid > max_grid) grid = max_grid;
    wps_stream_kernel<ODD, OutT, GROUPS, FUSE><<<(unsigned)grid, kStreamThreads<GROUPS>, smem, a.stream>>>(
        a.frag_start, a.frag_stop, a.frag_mapq, a.n_frag, a.tile_p0, a.tile_len, a.tile_mid_lo, a.tile_mid_hi,
        a.tile_out_off, a.tile_ivl, a.ranges, (int)a.n_tiles, a.P, a.C, out, a.overflow, a.counts, a.hist);
    FTK_CHECK_LAUNCH("wps_stream_kernel");
    return FTK_OK;
}

static void wps_fill_params(ftk::WpsParams &P, int32_t window_size, int32_t min_len, int32_t max_len,
                            int32_t min_mapq) {
    const bool odd = (window_size & 1) != 0;
    P.window = window_size;
    P.a = odd ? (window_size - 1) / 2 : window_size / 2;
    P.b = odd ? P.a : P.a - 1;
    P.len_lo = (min_len == FTK_NONE || min_len < 0) ? 0 : min_len;
    P.max_len = max_len;
    if (max_len < P.len_lo) {  // empty length window: every position scores 0
        // (still run the kernel so `out` is fully written; nothing passes the range test)
        P.len_lo = 1; P.len_span = 0; P.min_mapq = 256;
    } else {
        P.len_span = (unsigned)(max_len - P.len_lo);
        P.min_mapq = min_mapq;
    }
}

template <typename OutT>
static int wps_tiles_impl(const int32_t *frag_start, const int32_t *frag_stop,
                          const uint8_t *frag_mapq, int64_t n_frag,
                          const int32_t *tile_p0, const int32_t *tile_len,
                          const int32_t *tile_mid_lo, const int32_t *tile_mid_hi,
                          const int64_t *tile_out_off, int64_t n_tiles,
                          int32_t window_size, int32_t min_len, int32_t max_len, int32_t min_mapq,
                          int32_t ranges_ready, int64_t *scratch, OutT *out, int *overflow,
                          ftk_stream_t stream_) {
    using namespace ftk;
    if (n_tiles == 0) return FTK_OK;
    int rc = wps_check_args(frag_start, frag_stop, n_frag, tile_p0, tile_len, n_tiles, window_size, max_len, scratch);
    if (rc != FTK_OK) return rc;
    if (!tile_mid_lo || !tile_mid_hi || !tile_out_off || !out) return FTK_E_INVALID;
    if (!ranges_ready) {
        rc = ftk_wps_tile_ranges(frag_start, n_frag, tile_p0, tile_len, n_tiles, window_size, max_len, scratch, stream_);
        if (rc != FTK_OK) return rc;
    }
    WpsLaunch a{};
    a.frag_start = frag_start; a.frag_stop = frag_stop; a.frag_mapq = frag_mapq; a.n_frag = n_frag;
    a.tile_p0 = tile_p0; a.tile_len = tile_len; a.tile_mid_lo = tile_mid_lo; a.tile_mid_hi = tile_mid_hi;
    a.tile_out_off = tile_out_off; a.tile_ivl = nullptr; a.n_tiles = n_tiles; a.ranges = scratch;
    a.overflow = overflow; a.counts = nullptr; a.hist = nullptr;
    a.stream = static_cast<cudaStream_t>(stream_);
    wps_fill_params(a.P, window_size, min_len, max_len, min_mapq);
    a.C = CovParams{0, 0u, 0, 0};
    return (window_size & 1) ? launch_stream<true, OutT, kPlainGroups, false>(a, out)
                             : launch_stream<false, OutT, kPlainGroups, false>(a, out);
}

extern "C" int ftk_wps_tiles_i32(const int32_t *frag_start, const int32_t *frag_stop,
                                 const uint8_t *frag_mapq, int64_t n_frag,
                                 const int32_t *tile_p0, const int32_t *tile_len,
                                 const int32_t *tile_mid_lo, const int32_t *tile_mid_hi,
                                 const int64_t *tile_out_off, int64_t n_tiles,
                                 int32_t window_size, int32_t min_len, int32_t max_len, int32_t min_mapq,
                                 int32_t ranges_ready, int64_t *scratch, int32_t *out,
                                 ftk_stream_t stream_) {
    return wps_tiles_impl<int32_t>(frag_start, frag_stop, frag_mapq, n_frag, tile_p0, tile_len, tile_mid_lo,
                                   tile_mid_hi, tile_out_off, n_tiles, window_size, min_len, max_len, min_mapq,
                                   ranges_ready, scratch, out, nullptr, stream_);
}

extern "C" int ftk_wps_tiles_i16(const int32_t *frag_start, const int32_t *frag_stop,
                                 const uint8_t *frag_mapq, int64_t n_frag,
                                 const int32_t *tile_p0, const int32_t *tile_len,
                                 const int32_t *tile_mid_lo, const int32_t *tile_mid_hi,
                                 const int64_t *tile_out_off, int64_t n_tiles,
                                 int32_t window_size, int32_t min_len, int32_t max_len, int32_t min_mapq,
                                 int32_t ranges_ready, int64_t *scratch, int16_t *out,
                                 int32_t *overflow_flag, ftk_stream_t stream_) {
    if (n_tiles > 0 && !overflow_flag) return FTK_E_INVALID;
    return wps_tiles_impl<int16_t>(frag_start, frag_stop, frag_mapq, n_frag, tile_p0, tile_len, tile_mid_lo,
                                   tile_mid_hi, tile_out_off, n_tiles, window_size, min_len, max_len, min_mapq,
                                   ranges_ready, scratch, out, overflow_flag, stream_);
}

extern "C" int ftk_wps_tiles_i8(const int32_t *frag_start, const int32_t *frag_stop,
                                const uint8_t *frag_mapq, int64_t n_frag,
                                const int32_t *tile_p0, const int32_t *tile_len,
                                const int32_t *tile_mid_lo, const int32_t *tile_mid_hi,
                                const int64_t *tile_out_off, int64_t n_tiles,
                                int32_t window_size, int32_t min_len, int32_t max_len, int32_t min_mapq,
                                int32_t ranges_ready, int64_t *scratch, int8_t *out,
                                int32_t *overflow_flag, ftk_stream_t stream_) {
    if (n_tiles > 0 && !overflow_flag) return FTK_E_INVALID;
    return wps_tiles_impl<int8_t>(frag_start, frag_stop, frag_mapq, n_frag, tile_p0, tile_len, tile_mid_lo,
                                  tile_mid_hi, tile_out_off, n_tiles, window_size, min_len, max_len, min_mapq,
                                  ranges_ready, scratch, out, overflow_flag, stream_);
}

// ---- fused pass: WPS + per-interval coverage + pooled length histogram (wps_stream_kernel<.., FUSE>)
// a fragment whose midpoint fs + (L >> 1) is >= p0 starts at fs >= p0 - (Lmax >> 1)
static int64_t fused_left_reach(int32_t window_size, int32_t max_len, int32_t cov_max_len, int32_t max_frag_len) {
    const int64_t cov_hi = (cov_max_len == FTK_NONE) ? INT32_MAX : cov_max_len;
    const int64_t lmax = cov_hi < max_frag_len ? cov_hi : max_frag_len;
    int64_t reach = wps_left_reach(window_size, max_len);
    if ((lmax >> 1) + 1 > reach) reach = (lmax >> 1) + 1;
    return reach;
}

extern "C" int ftk_wps_cov_tile_ranges(const int32_t *frag_start, int64_t n_frag,
                                       const int32_t *tile_p0, const int32_t *tile_len, int64_t n_tiles,
                                       int32_t window_size, int32_t max_len, int32_t cov_max_len,
                                       int32_t max_frag_len, int64_t *scratch,
                                       uint64_t *zero_counts, int64_t n_counts, uint64_t *zero_hist, int64_t n_hist,
                                       ftk_stream_t stream_) {
    if (n_tiles == 0) return FTK_OK;
    int rc = wps_check_args(frag_start, frag_start, n_frag, tile_p0, tile_len, n_tiles, window_size, max_len, scratch);
    if (rc != FTK_OK) return rc;
    if (max_frag_len < 0 || n_counts < 0 || n_hist < 0) return FTK_E_INVALID;
    if ((n_counts > 0 && !zero_counts) || (n_hist > 0 && !zero_hist)) return FTK_E_INVALID;
    return launch_tile_ranges(frag_start, n_frag, tile_p0, tile_len, n_tiles, window_size,
                              fused_left_reach(window_size, max_len, cov_max_len, max_frag_len), scratch,
                              static_cast<cudaStream_t>(stream_),
                              reinterpret_cast<unsigned long long *>(zero_counts), n_counts,
                              reinterpret_cast<unsigned long long *>(zero_hist), n_hist);
}

extern "C" int ftk_wps_cov_tiles(const int32_t *frag_start, const int32_t *frag_stop,
                                 const uint8_t *frag_mapq, int64_t n_frag, int32_t max_frag_len,
                                 const int32_t *tile_p0, const int32_t *tile_len,
                                 const int32_t *tile_mid_lo, const int32_t *tile_mid_hi,
                                 const int64_t *tile_out_off, const int32_t *tile_ivl, int64_t n_tiles,
                                 int32_t window_size, int32_t min_len, int32_t max_len, int32_t min_mapq,
                                 int32_t cov_min_len, int32_t cov_max_len, int32_t cov_min_mapq, int32_t n_bins,
                                 int32_t ranges_ready, int64_t *scratch, int32_t out_kind, void *out,
                                 int32_t *overflow_flag, uint64_t *counts, uint64_t *hist, ftk_stream_t stream_) {
    using namespace ftk;
    if (n_tiles == 0) return FTK_OK;
    int rc = wps_check_args(frag_start, frag_stop, n_frag, tile_p0, tile_len, n_tiles, window_size, max_len, scratch);
    if (rc != FTK_OK) return rc;
    if (!tile_mid_lo || !tile_mid_hi || !tile_out_off || !tile_ivl || !out || !counts) return FTK_E_INVALID;
    if (out_kind < 0 || out_kind > 2 || n_bins < 0 || max_frag_len < 0) return FTK_E_INVALID;
    if (out_kind != 0 && !overflow_flag) return FTK_E_INVALID;
    if (n_bins > 0 && !hist) return FTK_E_INVALID;
    if (n_frag > INT32_MAX) return FTK_E_RANGE;   // a CTA's shared histogram counts in int32
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    WpsLaunch a{};
    wps_fill_params(a.P, window_size, min_len, max_len, min_mapq);
    // coverage stream predicate (FTK_NONE = unbounded), as Stream in ftk_hist.cu
    a.C.len_lo = (cov_min_len == FTK_NONE || cov_min_len < 0) ? 0 : cov_min_len;
    const int cov_hi = (cov_max_len == FTK_NONE) ? INT32_MAX : cov_max_len;
    if (cov_hi < a.C.len_lo) { a.C.len_lo = 1; a.C.len_span = 0; a.C.min_mapq = 256; }
    else { a.C.len_span = (unsigned)(cov_hi - a.C.len_lo); a.C.min_mapq = cov_min_mapq; }
    a.C.n_bins = n_bins;
    if (!ranges_ready) {
        rc = ftk_wps_cov_tile_ranges(frag_start, n_frag, tile_p0, tile_len, n_tiles, window_size, max_len,
                                     cov_max_len, max_frag_len, scratch, nullptr, 0, nullptr, 0, stream_);
        if (rc != FTK_OK) return rc;
    }
    a.frag_start = frag_start; a.frag_stop = frag_stop; a.frag_mapq = frag_mapq; a.n_frag = n_frag;
    a.tile_p0 = tile_p0; a.tile_len = tile_len; a.tile_mid_lo = tile_mid_lo; a.tile_mid_hi = tile_mid_hi;
    a.tile_out_off = tile_out_off; a.tile_ivl = tile_ivl; a.n_tiles = n_tiles; a.ranges = scratch;
    a.overflow = overflow_flag;
    a.counts = reinterpret_cast<unsigned long long *>(counts);
    a.hist = reinterpret_cast<unsigned long long *>(hist);
    a.stream = stream;
    const bool odd = (window_size & 1) != 0;
#define FTK_FUSED(T)                                                            \
    (odd ? launch_stream<true, T, kFusedGroups, true>(a, static_cast<T *>(out)) \
         : launch_stream<false, T, kFusedGroups, true>(a, static_cast<T *>(out)))
    if (out_kind == 0) return FTK_FUSED(int32_t);
    if (out_kind == 1) return FTK_FUSED(int16_t);
    return FTK_FUSED(int8_t);
#undef FTK_FUSED
}
