// MurmurHash3 x64_128 (seed as u64, h1 = h2 = seed) -- host + device.
//
// Replaces the third-party crate call `murmurhash3_x64_128(kmer, seed).0`
// (reference src/lib.rs:29,33-35; crate murmurhash3 ~0.0.5, Cargo.toml:49).
// Written from the published algorithm; pinned by tests/test.rs:5 and the
// SMHasher verification value (see oracle/oracle.c).
//
// Two entry points:
//   murmur3_h1_bytes(ptr, len, seed)   any byte string (host add_word / hash_murmur,
//                                      generic-k device kernel)
//   murmur3_h1_words<K>(w, seed)       K bytes already held as little-endian
//                                      32-bit words in registers (templated kernel);
//                                      bytes past K in the last word must be zero.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define SM_HD __host__ __device__ __forceinline__
#else
#define SM_HD inline
#endif

namespace smb200 {

constexpr uint64_t MM_C1 = 0x87c37b91114253d5ULL;
constexpr uint64_t MM_C2 = 0x4cf5ad432745937fULL;

// ---- 64-bit primitives -------------------------------------------------------------------
// On the device the 64-bit multiplies and rotates are spelled on 32-bit halves: ptxas expands a
// plain `x * C` into IMAD + IMAD + IMAD.WIDE + IADD (4 issue slots, shorter dependency chain) and
// a plain rotate into 3-4 shifts/ors; the sketch kernel is issue-bound, so the three-instruction
// multiply (IMAD.WIDE, IMAD, IMAD: each accumulating into the high word) and the two-funnel-shift
// rotate are forced here.  Same values, 86 instead of 117 SASS instructions per k=31 hash.
template <uint64_t C>
SM_HD uint64_t mm_mulc(uint64_t x) {
#if defined(__CUDA_ARCH__)
    uint64_t r;
    asm("{\n\t.reg .u32 lo, hi, rl, rh;\n\t.reg .u64 t;\n\t"
        "mov.b64 {lo, hi}, %1;\n\t"
        "mul.wide.u32 t, lo, %2;\n\t"
        "mov.b64 {rl, rh}, t;\n\t"
        "mad.lo.u32 rh, lo, %3, rh;\n\t"
        "mad.lo.u32 rh, hi, %2, rh;\n\t"
        "mov.b64 %0, {rl, rh};\n\t}"
        : "=l"(r)
        : "l"(x), "n"((uint32_t)C), "n"((uint32_t)(C >> 32)));
    return r;
#else
    return x * C;
#endif
}
// x * 5 + ADD.  On the device this compiles to IMAD.WIDE.U32 with the constant as a 64-bit addend + IMAD +
// IMAD.IADD: the fewest issue slots of the forms tried, which is what the sketch kernels are bound by.  A
// `mul.wide.u32` + `mad.lo` + `add.cc/addc` form and an ALU shift-add form take fewer FMA-heavy cycles by the
// static model but no fewer instructions, and measured no faster (DESIGN 4.1).
template <uint32_t ADD>
SM_HD uint64_t mm_mul5add(uint64_t x) {
    return x * 5 + ADD;
}
template <int R>
SM_HD uint64_t mm_rotl64(uint64_t x) {
#if defined(__CUDA_ARCH__)
    const uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
    constexpr uint32_t S = (uint32_t)(R & 31);
    uint32_t nlo, nhi;
    if (R < 32) { nhi = __funnelshift_l(lo, hi, S); nlo = __funnelshift_l(hi, lo, S); }
    else        { nhi = __funnelshift_l(hi, lo, S); nlo = __funnelshift_l(lo, hi, S); }
    return ((uint64_t)nhi << 32) | nlo;
#else
    return (x << R) | (x >> (64 - R));
#endif
}

// k ^ (k >> 33): only the low word changes, by hi >> 1.  (MM_XS_IMADHI spells the shift as the high
// half of hi * 2^31 to move it from the ALU to the FMA pipe; IMAD.HI occupies that pipe for 4 cycles
// on sm_100a -- tests/manual/intpeak.py -- and measured slower, so it is off.)
SM_HD uint64_t mm_xorshift33(uint64_t k) {
#if defined(__CUDA_ARCH__) && defined(MM_XS_IMADHI)
    uint32_t lo = (uint32_t)k, hi = (uint32_t)(k >> 32), t;
    asm("mul.hi.u32 %0, %1, 0x80000000;" : "=r"(t) : "r"(hi));
    lo ^= t;
    return ((uint64_t)hi << 32) | lo;
#else
    return k ^ (k >> 33);
#endif
}
// fmix64 without its last xorshift33, which leaves the high word as it is: the sketch kernels test the high words
// first and finish the hash only for the rare windows that may pass (murmur3_h1_words_parts)
SM_HD uint64_t mm_fmix64_pre(uint64_t k) {
    k = mm_xorshift33(k);
    k = mm_mulc<0xff51afd7ed558ccdULL>(k);
    k = mm_xorshift33(k);
    k = mm_mulc<0xc4ceb9fe1a85ec53ULL>(k);
    return k;
}
SM_HD uint64_t mm_fmix64(uint64_t k) { return mm_xorshift33(mm_fmix64_pre(k)); }

SM_HD uint64_t mm_mix_k1(uint64_t k1) {
    k1 = mm_mulc<MM_C1>(k1); k1 = mm_rotl64<31>(k1); k1 = mm_mulc<MM_C2>(k1);
    return k1;
}
SM_HD uint64_t mm_mix_k2(uint64_t k2) {
    k2 = mm_mulc<MM_C2>(k2); k2 = mm_rotl64<33>(k2); k2 = mm_mulc<MM_C1>(k2);
    return k2;
}
SM_HD void mm_body(uint64_t &h1, uint64_t &h2, uint64_t k1, uint64_t k2) {
    h1 ^= mm_mix_k1(k1);
    h1 = mm_rotl64<27>(h1); h1 += h2; h1 = mm_mul5add<0x52dce729u>(h1);
    h2 ^= mm_mix_k2(k2);
    h2 = mm_rotl64<31>(h2); h2 += h1; h2 = mm_mul5add<0x38495ab5u>(h2);
}
SM_HD uint64_t mm_final_h1(uint64_t h1, uint64_t h2, uint64_t len) {
    h1 ^= len; h2 ^= len;
    h1 += h2; h2 += h1;
    h1 = mm_fmix64(h1); h2 = mm_fmix64(h2);
    h1 += h2;
    return h1;  // .0 of the (h1, h2) pair
}

// Generic byte-string version (unaligned safe: assembles words bytewise).
SM_HD uint64_t murmur3_h1_bytes(const uint8_t *data, uint64_t len, uint64_t seed) {
    uint64_t h1 = seed, h2 = seed;
    const uint64_t nblocks = len / 16;
    for (uint64_t b = 0; b < nblocks; b++) {
        uint64_t k1 = 0, k2 = 0;
        for (int j = 7; j >= 0; j--) {
            k1 = (k1 << 8) | data[16 * b + j];
            k2 = (k2 << 8) | data[16 * b + 8 + j];
        }
        mm_body(h1, h2, k1, k2);
    }
    const uint8_t *tail = data + nblocks * 16;
    const int rem = (int)(len & 15);
    uint64_t k1 = 0, k2 = 0;
    for (int j = rem - 1; j >= 8; j--) k2 = (k2 << 8) | tail[j];
    for (int j = (rem < 8 ? rem : 8) - 1; j >= 0; j--) k1 = (k1 << 8) | tail[j];
    if (rem > 8) h2 ^= mm_mix_k2(k2);
    if (rem > 0) h1 ^= mm_mix_k1(k1);
    return mm_final_h1(h1, h2, len);
}

// K bytes held in ceil(K/4) little-endian 32-bit words; fully unrolled.  Returns the hash in two parts,
// h1 = mm_xorshift33(a) + mm_xorshift33(b) (mod 2^64), where the high words of a and b are those of the two addends.
template <int K>
SM_HD void murmur3_h1_words_parts(const uint32_t *w, uint64_t seed, uint64_t &a, uint64_t &b) {
    constexpr int NB = K / 16;
    constexpr int REM = K % 16;
    uint64_t h1 = seed, h2 = seed;
#pragma unroll
    for (int b = 0; b < NB; b++) {
        const uint64_t k1 = ((uint64_t)w[4 * b + 1] << 32) | w[4 * b + 0];
        const uint64_t k2 = ((uint64_t)w[4 * b + 3] << 32) | w[4 * b + 2];
        mm_body(h1, h2, k1, k2);
    }
    if (REM > 8) {
        const uint32_t hi = (REM > 12) ? w[4 * NB + 3] : 0u;
        const uint64_t k2 = ((uint64_t)hi << 32) | w[4 * NB + 2];
        h2 ^= mm_mix_k2(k2);
    }
    if (REM > 0) {
        const uint32_t hi = (REM > 4) ? w[4 * NB + 1] : 0u;
        const uint64_t k1 = ((uint64_t)hi << 32) | w[4 * NB + 0];
        h1 ^= mm_mix_k1(k1);
    }
    h1 ^= (uint64_t)K; h2 ^= (uint64_t)K;
    h1 += h2; h2 += h1;
    a = mm_fmix64_pre(h1); b = mm_fmix64_pre(h2);
}
template <int K>
SM_HD uint64_t murmur3_h1_words(const uint32_t *w, uint64_t seed) {
    uint64_t a, b;
    murmur3_h1_words_parts<K>(w, seed, a, b);
    return mm_xorshift33(a) + mm_xorshift33(b);
}

}  // namespace smb200
