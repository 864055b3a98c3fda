// G/C content of a fragment on the 2-bit packed contig, shared by the GC kernels (ftk_gc.cu) and the GC-weighted
// depth tiles (ftk_cleavage.cu).
//
// Packed layout (synth.pack_twobit): base i in bits 2(i%16) of seq word i/16 (A0 C1 G2 T3), its N flag in bit
// i%32 of nmask word i/32.  A 64-bit seq word k and nmask word k cover the same 32 bases, so every read here is
// one aligned 64-bit seq load + one 32-bit nmask load per 32 bases; G/C <=> bit0 ^ bit1 of a base's code.
#pragma once
#include <stdint.h>

namespace ftk {

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

}  // namespace ftk
