// kmer_bits.cuh -- the bit-level pieces of the sketch kernel, written host+device so the
// exact same code is exercised on the CPU by tests/host/tile_views_test.cpp.
//
// What they replace in the reference (all relative to /root/reference):
//   fold_and_classify8 : the whole-sequence uppercase copy (src/lib.rs:253-256) and the
//                        per-window validity scan _checkdna (src/lib.rs:795-804) -- done ONCE
//                        per base instead of k times
//   revcomp views      : revcomp (src/lib.rs:677-689), which heap-allocates per k-mer -- here
//                        the reverse-complement STRAND of a whole tile is materialised once
//   canonical_is_fw    : the byte-wise `kmer < rc` (src/lib.rs:263-267) as one integer compare
//
// Tile views (B = staged bases, a multiple of 16):
//   fA[j]      upper-cased ASCII of base j                                   (B bytes)
//   rA[B-1-j]  ASCII complement of base j, so rc(window i) = rA[B-K-i .. B-i) (B bytes)
//   f2         2-bit codes A0 C1 G2 T3, base j at bits 2(j%16) of word j/16   (B/16 words)
//   r2         same layout for the reverse-complement strand                 (B/16 words)
//   bad        bit j set = base j is not one of ACGTacgt                      (B/32 words)
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define KB_HD __host__ __device__ __forceinline__
#else
#define KB_HD inline
#endif

namespace smb200 {

// ---- portable spellings of the three integer intrinsics used below ----------------------
KB_HD uint32_t kb_byte_perm(uint32_t a, uint32_t b, uint32_t sel) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(a, b, sel);
#else
    const uint64_t pool = ((uint64_t)b << 32) | a;
    uint32_t r = 0;
    for (int i = 0; i < 4; i++) {
        const uint32_t s = (sel >> (4 * i)) & 0x7u;  // (msb replicate mode is never used here)
        r |= (uint32_t)((pool >> (8 * s)) & 0xFFu) << (8 * i);
    }
    return r;
#endif
}
KB_HD uint32_t kb_brev(uint32_t x) {
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
// low 32 bits of ((hi:lo) >> (s & 31))
KB_HD uint32_t kb_funnel_r(uint32_t lo, uint32_t hi, uint32_t s) {
#if defined(__CUDA_ARCH__)
    return __funnelshift_r(lo, hi, s);
#else
    s &= 31u;
    return s ? ((lo >> s) | (hi << (32 - s))) : lo;
#endif
}

// ---- 4 raw ASCII bytes -> folded bytes, codes, validity ----------------------------------
struct Quad {
    uint32_t upper;   // the 4 bytes with bit 5 cleared (== to_ascii_uppercase for every valid base)
    uint32_t comp;    // ASCII complement of each byte (garbage where invalid)
    uint32_t codes8;  // 4 x 2-bit codes, base t at bits 2t
    uint32_t bad4;    // bit t set = byte t is not ACGTacgt
};
KB_HD Quad classify4(uint32_t raw) {
    Quad q;
    const uint32_t u = raw & 0xDFDFDFDFu;
    const uint32_t c = ((u >> 1) ^ (u >> 2)) & 0x03030303u;  // A0 C1 G2 T3 in each byte
    // nibble selector for PRMT: code of byte t in nibble t
    const uint32_t sel = (c & 0x3u) | ((c >> 4) & 0x30u) | ((c >> 8) & 0x300u) | ((c >> 12) & 0x3000u);
    const uint32_t expect = kb_byte_perm(0x54474341u /* 'A','C','G','T' */, 0u, sel);
    const uint32_t x = expect ^ u;  // non-zero byte <=> not a DNA base
    const uint32_t nz = (x | ((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu)) & 0x80808080u;
    q.upper = u;
    q.comp = kb_byte_perm(0x41434754u /* 'T','G','C','A' */, 0u, sel);
    q.codes8 = (c * 0x01041040u) >> 24;
    q.bad4 = ((nz >> 7) * 0x01020408u) >> 24;
    return q;
}

// reverse the order of the eight 2-bit fields of a 16-bit value
KB_HD uint32_t pair_reverse16(uint32_t x) {
    x = kb_brev(x) >> 16;
    return ((x >> 1) & 0x5555u) | ((x & 0x5555u) << 1);
}

// ---- 8 bases (two raw words) -> everything the tile views need ----------------------------
struct Oct {
    uint32_t fA0, fA1;  // forward ASCII words (bases 0-3, 4-7)
    uint32_t rA0, rA1;  // reverse-complement ASCII words, in increasing rA address order
    uint32_t f2;        // 16 bits of forward codes
    uint32_t r2;        // 16 bits of reverse-complement codes
    uint32_t bad8;      // 8 invalid bits
};
KB_HD Oct classify8(uint32_t raw0, uint32_t raw1) {
    const Quad a = classify4(raw0), b = classify4(raw1);
    Oct o;
    o.fA0 = a.upper;
    o.fA1 = b.upper;
    o.rA0 = kb_byte_perm(b.comp, 0u, 0x0123u);  // bases 7,6,5,4 complemented
    o.rA1 = kb_byte_perm(a.comp, 0u, 0x0123u);  // bases 3,2,1,0 complemented
    o.f2 = a.codes8 | (b.codes8 << 8);
    o.r2 = (~pair_reverse16(o.f2)) & 0xFFFFu;
    o.bad8 = a.bad4 | (b.bad4 << 4);
    return o;
}

// ---- per-window extraction ------------------------------------------------------------------
template <int K>
struct KmerGeom {
    static constexpr int NE = (2 * K + 31) / 32;  // 32-bit words of a 2-bit packed k-mer
    static constexpr int NW = (K + 3) / 4;        // 32-bit words of an ASCII k-mer
    static constexpr uint32_t TOP2 = (2 * K) % 32 ? ((1u << ((2 * K) % 32)) - 1u) : 0xFFFFFFFFu;
    static constexpr uint32_t TOPA = (K % 4) ? ((1u << ((K % 4) * 8)) - 1u) : 0xFFFFFFFFu;
};

// 2K bits starting at base `start` of a 2-bit stream (words must be readable up to
// (start/16) + NE inclusive)
template <int K>
KB_HD void extract2(const uint32_t *stream, int start, uint32_t (&e)[KmerGeom<K>::NE]) {
    const int w = start >> 4;
    const uint32_t s = (uint32_t)(start & 15) * 2u;
    uint32_t prev = stream[w];
#pragma unroll
    for (int j = 0; j < KmerGeom<K>::NE; j++) {
        const uint32_t next = stream[w + j + 1];
        e[j] = kb_funnel_r(prev, next, s);
        prev = next;
    }
    e[KmerGeom<K>::NE - 1] &= KmerGeom<K>::TOP2;
}

// same as extract2 with the word pointer and the bit shift already split (the kernel keeps both
// loop-invariant per thread); only the low 5 bits of `s` are used (funnel shift wraps)
template <int K>
KB_HD void extract2w(const uint32_t *w, uint32_t s, uint32_t (&e)[KmerGeom<K>::NE]) {
    uint32_t prev = w[0];
#pragma unroll
    for (int j = 0; j < KmerGeom<K>::NE; j++) {
        const uint32_t next = w[j + 1];
        e[j] = kb_funnel_r(prev, next, s);
        prev = next;
    }
    e[KmerGeom<K>::NE - 1] &= KmerGeom<K>::TOP2;
}

// NE words whose TOP bits are the k-mer's last base: `w`/`s` address bit 2 * (start + K) - 32 * NE of
// the stream, so the 32 * NE - 2K low bits are whatever precedes the k-mer.  For ODD K that is
// harmless to canonical_is_fw: a k-mer of odd length never equals its reverse complement, so the
// comparison is decided inside the K real bases, which sit above the extra low bits on both sides.
// Saves the two top-word masks of extract2.
template <int K>
KB_HD void extract2_end(const uint32_t *w, uint32_t s, uint32_t (&e)[KmerGeom<K>::NE]) {
    static_assert(K % 2 == 1, "end-aligned strand comparison needs an odd k");
    uint32_t prev = w[0];
#pragma unroll
    for (int j = 0; j < KmerGeom<K>::NE; j++) {
        const uint32_t next = w[j + 1];
        e[j] = kb_funnel_r(prev, next, s);
        prev = next;
    }
}

// lexicographic `fw < rc` (src/lib.rs:263) from the little-endian 2-bit integers of the two
// strands: with comp(c) = ~c, BE(fw) = ~E(rc) and BE(rc) = ~E(fw), so fw <lex rc <=> E(fw) < E(rc).
template <int K>
KB_HD bool canonical_is_fw(const uint32_t (&ef)[KmerGeom<K>::NE], const uint32_t (&er)[KmerGeom<K>::NE]) {
    // multi-word unsigned compare: up to two words as one 64-bit compare (ISETP + ISETP.EX), more as a borrow
    // chain on the device; ties -> rc, as the reference's `else` arm (identical bytes anyway)
    constexpr int NE = KmerGeom<K>::NE;
    if (NE == 1) return ef[0] < er[0];
    if (NE == 2) return (((uint64_t)ef[1] << 32) | ef[0]) < (((uint64_t)er[1] << 32) | er[0]);
#if defined(__CUDA_ARCH__)
    // one borrow chain ef - er over all words (missing top words are 0 - 0, which pass the borrow on): fw < rc
    // exactly when it borrows out of the top word.  Replaces a compare / compare / select per word.
    static_assert(NE <= 4, "borrow chain spelled for up to four words");
    uint32_t f[4] = {0, 0, 0, 0}, r[4] = {0, 0, 0, 0}, borrow;
#pragma unroll
    for (int j = 0; j < NE; j++) { f[j] = ef[j]; r[j] = er[j]; }
    asm("{\n\t.reg .u32 t;\n\t"
        "sub.cc.u32 t, %1, %5;\n\t"
        "subc.cc.u32 t, %2, %6;\n\t"
        "subc.cc.u32 t, %3, %7;\n\t"
        "subc.cc.u32 t, %4, %8;\n\t"
        "subc.u32 %0, 0, 0;\n\t}"
        : "=r"(borrow)
        : "r"(f[0]), "r"(f[1]), "r"(f[2]), "r"(f[3]), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]));
    return borrow != 0;
#else
    bool lt = false;
#pragma unroll
    for (int j = 0; j < NE; j++) {  // least significant word first; later words override
        if (ef[j] != er[j]) lt = ef[j] < er[j];
    }
    return lt;
#endif
}

// K ASCII bytes starting at byte `start` of a byte stream viewed as words (readable up to
// (start/4) + NW inclusive); bytes past K in the last word are zeroed.
template <int K>
KB_HD void extractA(const uint32_t *words, int start, uint32_t (&kw)[KmerGeom<K>::NW]) {
    const int w = start >> 2;
    const uint32_t s = (uint32_t)(start & 3) * 8u;
    uint32_t prev = words[w];
#pragma unroll
    for (int j = 0; j < KmerGeom<K>::NW; j++) {
        const uint32_t next = words[w + j + 1];
        kw[j] = kb_funnel_r(prev, next, s);
        prev = next;
    }
    kw[KmerGeom<K>::NW - 1] &= KmerGeom<K>::TOPA;
}

// same with the word pointer and the bit shift (low 5 bits used) already split
template <int K>
KB_HD void extractAw(const uint32_t *w, uint32_t s, uint32_t (&kw)[KmerGeom<K>::NW]) {
    uint32_t prev = w[0];
#pragma unroll
    for (int j = 0; j < KmerGeom<K>::NW; j++) {
        const uint32_t next = w[j + 1];
        kw[j] = kb_funnel_r(prev, next, s);
        prev = next;
    }
    kw[KmerGeom<K>::NW - 1] &= KmerGeom<K>::TOPA;
}

// window-start bitmap: bit p of the result word covers start q = 32*w + p and is set when any
// of `span` stream bits q .. q+span-1 is set.  in[0..2] are stream words w, w+1, w+2 (span <= 64).
// Doubling on the 96-bit window V: D_1 = V, D_2s = D_s | (D_s >> s), and for the largest power of two
// a <= span, D_span = D_a | (D_a >> (span - a)) -- about 30 operations for k = 31 instead of 2 per base
// of the span.
KB_HD void kb_shr96(uint32_t &x0, uint32_t &x1, uint32_t &x2, int s) {  // (x2:x1:x0) >>= s, 0 < s < 64
    if (s < 32) {
        x0 = kb_funnel_r(x0, x1, (uint32_t)s);
        x1 = kb_funnel_r(x1, x2, (uint32_t)s);
        x2 >>= s;
    } else {
        x0 = kb_funnel_r(x1, x2, (uint32_t)(s - 32));  // s == 32: funnel by 0 returns x1
        x1 = (s == 32) ? x2 : (x2 >> (s - 32));
        x2 = 0;
    }
}
KB_HD uint32_t dilate_word(uint32_t in0, uint32_t in1, uint32_t in2, int span) {
    if (span <= 0) return 0;
    uint32_t d0 = in0, d1 = in1, d2 = in2;
    int a = 1;
    while (2 * a <= span) {
        uint32_t y0 = d0, y1 = d1, y2 = d2;
        kb_shr96(y0, y1, y2, a);
        d0 |= y0; d1 |= y1; d2 |= y2;
        a *= 2;
    }
    if (span > a) {
        uint32_t y0 = d0, y1 = d1, y2 = d2;
        kb_shr96(y0, y1, y2, span - a);
        d0 |= y0;
    }
    return d0;
}

}  // namespace smb200
