// Per-word arithmetic of the strand-doubled batch (ingest.cu, k_both_strands), shared with the host-compiled test
// (tests/test_strands_host.py).
//
// A read of L bases sits in words src[0 .. 4 * chunks) of the packed layout (16 bases per word, MSB-first, pad bits zero).
// Word w of its copy is src[w]; word w of its reverse complement holds bases 16w .. 16w+15 of RC, base k of RC being
// 3 - base[L-1-k].  Those come from the 16-base source window [L-16-16w, L-16w): aligned by a funnel shift, its 16
// fields reversed (bit reversal, then the two bits of each field swapped back) and complemented (~x is x ^ 3 per field).
// Bases at or past L come out as zero in both words, so the output equals gsm_pack_reads of the two strings.
#pragma once
#include <stdint.h>

#include "fm_core.cuh"

namespace gsm {

// bases of word w that lie inside a read of L bases, as a mask of their bit fields (top 2 * valid bits)
GSM_HD uint32_t strand_word_mask(uint32_t L, uint32_t w) {
    const uint32_t t0 = w * 16u;
    if (t0 >= L) return 0u;
    const uint32_t valid = L - t0;
    return valid >= 16u ? 0xFFFFFFFFu : ~(0xFFFFFFFFu >> (2u * valid));
}

GSM_HD uint32_t strand_brev(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return __brev(x);
#else
    x = ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
    x = ((x >> 2) & 0x33333333u) | ((x & 0x33333333u) << 2);
    x = ((x >> 4) & 0x0F0F0F0Fu) | ((x & 0x0F0F0F0Fu) << 4);
    x = ((x >> 8) & 0x00FF00FFu) | ((x & 0x00FF00FFu) << 8);
    return (x >> 16) | (x << 16);
#endif
}

// the top 32 bits of (hi:lo) << sh, sh in [0, 32)
GSM_HD uint32_t strand_funnel(uint32_t lo, uint32_t hi, uint32_t sh) {
#if defined(__CUDA_ARCH__)
    return __funnelshift_l(lo, hi, sh);
#else
    return sh ? (hi << sh) | (lo >> (32u - sh)) : hi;
#endif
}

// the 16 2-bit fields of x in reverse order
GSM_HD uint32_t strand_reverse_fields(uint32_t x) {
    const uint32_t b = strand_brev(x);
    return ((b >> 1) & 0x55555555u) | ((b & 0x55555555u) << 1);
}

// Source words of RC word w: the window starts at base s = L - 16 - 16w, i.e. in word q = floor(s / 16) at field
// s mod 16.  q may be -1 (the window starts before the read: those fields are zero) and word q + 1 is needed only when
// the window is not word-aligned.  Returns false for a word past the read (it is zero).
struct StrandSrc {
    int32_t q;      // first source word, -1 .. L/16
    uint32_t sh;    // left shift in bits, 2 * (s mod 16)
};

GSM_HD bool strand_rc_src(uint32_t L, uint32_t w, StrandSrc* s) {
    if (w * 16u >= L) return false;
    const int32_t start = (int32_t)L - 16 - 16 * (int32_t)w;      // >= -15
    const int32_t q = start >= 0 ? start / 16 : -1;
    s->q = q;
    s->sh = 2u * (uint32_t)(start - 16 * q);
    return true;
}

// RC word w from its two source words (hi = src[q] or 0 when q < 0, lo = src[q + 1], unused when sh == 0)
GSM_HD uint32_t strand_rc_word(uint32_t hi, uint32_t lo, uint32_t sh, uint32_t L, uint32_t w) {
    return ~strand_reverse_fields(strand_funnel(lo, hi, sh)) & strand_word_mask(L, w);
}

}  // namespace gsm
