// sketch.cu -- the hot kernel: ASCII DNA in HBM -> canonical k-mers -> MurmurHash3 x64_128
// -> threshold filter -> survivor list.  One launch covers a whole batch of sequences.
//
// Replaces the per-k-mer body of KmerMinHash::add_sequence (reference src/lib.rs:252-274):
// the uppercase copy (lib.rs:253-256), _checkdna (lib.rs:795-804), the allocating revcomp
// (lib.rs:677-689), the lexicographic min (lib.rs:263-267), _hash_murmur (lib.rs:33-35) and the
// acceptance gate of add_hash (lib.rs:198-209).  The sorted insert of add_hash is done for all
// survivors at once by the sort / reduce / merge kernels of sortops.cu.
//
// Shape of the kernel (sm_100a):
//   * persistent CTAs, grid = SM count x resident CTAs; tiles of TILE window starts are handed out
//     dynamically (first tile = block index, then an atomic counter fetched one tile ahead);
//   * the tile's TILE + halo ASCII bytes are brought HBM -> shared memory by ONE TMA bulk copy
//     (cp.async.bulk, completion on an mbarrier); the copy of the NEXT tile is issued as soon as
//     the current raw bytes have been consumed, so it overlaps the whole hashing phase;
//   * the CTA turns the raw bytes into five shared-memory views (kmer_bits.cuh): upper-cased
//     forward ASCII, reverse-complement ASCII, both strands 2-bit packed, and an invalid-base
//     bitmap; a second short phase dilates the invalid/sequence-end bitmaps into a
//     "window start is unusable" bitmap per k-size;
//   * one launch serves up to three sketches (k-sizes) of the same batch: the staging above is
//     done once per tile, then one k-mer loop per k-size walks it;
//   * one thread per k-mer: one bit test for validity, two unaligned end-aligned 2-bit extractions
//     + one integer compare for the canonical strand, one unaligned ASCII extraction of the
//     chosen strand, MurmurHash3 x64_128 fully unrolled for the compile-time K (murmur3.cuh),
//     `<= threshold`; survivors leave through a predicated branch.
// Bound: the ALU and FMA-heavy integer pipes (160 executed instructions per k-mer at k=31 for
// 1 byte of HBM traffic; 59-70 % of a kernel that does nothing but the hash), see DESIGN.md 4.1.
#include "device.hpp"
#include "kernels.cuh"
#include "kmer_bits.cuh"
#include "murmur3.cuh"

namespace smb200 {

#ifndef SK_UNROLL
#define SK_UNROLL 4   // windows per trip of the k-mer loop (SK_TILE / SK_THREADS must be a multiple)
#endif
#ifndef SK_SHIFTED
#define SK_SHIFTED 1  // four byte-shifted copies of each ASCII strand: the k-mer loop reads aligned words (0: funnel shifts)
#endif
#ifndef SK_UNROLL_FUSED
#define SK_UNROLL_FUSED 2
#endif
#ifndef SK_MIN_CTAS
#define SK_MIN_CTAS SK_CTAS_PER_SM
#endif

// ---------------------------------------------------------------------------------------
// mbarrier / TMA bulk-copy primitives (PTX; SASS: SYNCS.*, UBLKCP)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// 1-D bulk copy global -> shared; dst/src 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void tma_load_1d(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// ---------------------------------------------------------------------------------------
// shared-memory tile
// ---------------------------------------------------------------------------------------
struct TileViews {
    uint8_t *raw;     // B bytes, 128-byte aligned (TMA destination)
    uint32_t *fA;     // B/4 + 2 words
    uint32_t *rA;     // B/4 + 2 words
    uint32_t *f2;     // SK_PAD2 + B/16 + 2 words (f2 points past the pad: end-aligned extraction reads before base 0)
    uint32_t *r2;     // SK_PAD2 + B/16 + 2 words
    uint32_t *bad;    // B/32 + 3 words   invalid-base bitmap
    uint32_t *end;    // B/32 + 3 words   "last base of a sequence" bitmap
    uint32_t *sbad;   // nk * TILE/32 words   window start unusable, one bitmap per k-size of the launch
};
constexpr int SK_PAD2 = 4;  // words in front of each 2-bit stream (extract2_end reaches up to 64 bases back)
__host__ __device__ constexpr int tile_bases(int K) { return SK_TILE + ((K - 1 + 15) / 16) * 16; }
// words between the byte-shifted copies of an ASCII strand: at least the (B + 8) bytes of one copy, and
// = 8 (mod 32) so that the 4 copies x 8 consecutive words a warp touches fall into 32 different banks
__host__ __device__ constexpr int copy_stride_words(int B) {
    int w = (B + 8) / 4 + 4;  // (+ 4: the copy builder reads one quad past the slack words)
    while (w % 32 != 8) w++;
    return w;
}
__host__ __device__ constexpr size_t tile_smem_bytes(int B, int nk = 1) {
    return (size_t)B                      // raw
           + (SK_SHIFTED ? 8 * (size_t)copy_stride_words(B) * 4 : 2 * ((size_t)B + 16))   // fA, rA (+ their byte-shifted copies)
           + 2 * ((size_t)B / 4 + 8 + 4 * SK_PAD2)  // f2, r2
           + 2 * ((size_t)(B + 31) / 32 * 4 + 12)  // bad, end
           + (size_t)nk * (SK_TILE / 8)   // sbad
           + 128;                         // alignment slack
}
__device__ __forceinline__ TileViews carve_tile(uint8_t *base, int B) {
    TileViews v;
    uint8_t *p = base;
    v.raw = p; p += B;                                   // B is a multiple of 16
    // with SK_SHIFTED, copy c (bytes shifted down by c) of a strand sits c * copy_stride_words(B) words after copy 0
    v.fA = reinterpret_cast<uint32_t *>(p); p += SK_SHIFTED ? 16 * copy_stride_words(B) : (B + 16);  // 16-byte aligned strands
    v.rA = reinterpret_cast<uint32_t *>(p); p += SK_SHIFTED ? 16 * copy_stride_words(B) : (B + 16);
    v.f2 = reinterpret_cast<uint32_t *>(p) + SK_PAD2; p += B / 4 + 8 + 4 * SK_PAD2;
    v.r2 = reinterpret_cast<uint32_t *>(p) + SK_PAD2; p += B / 4 + 8 + 4 * SK_PAD2;
    const int wm = (B + 31) / 32 + 3;
    v.bad = reinterpret_cast<uint32_t *>(p); p += wm * 4;
    v.end = reinterpret_cast<uint32_t *>(p); p += wm * 4;
    v.sbad = reinterpret_cast<uint32_t *>(p);
    return v;
}

// bytes the TMA copy of tile `tile` moves (0 when the tile starts at or after the buffer end)
__device__ __forceinline__ uint32_t tile_copy_bytes(uint64_t t0, uint64_t n, int B) {
    if (t0 >= n) return 0;
    const uint64_t left = ((n - t0) + 15) & ~15ull;
    return (uint32_t)(left < (uint64_t)B ? left : (uint64_t)B);
}

// raw -> fA, rA, f2, r2, bad, end   (all threads; ends with the views complete after a barrier
// by the caller)
__device__ __forceinline__ void build_views(const TileViews &v, int B, uint64_t t0, const SketchBatch &sb) {
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int wm = (B + 31) / 32 + 3;
    for (int w = tid; w < wm; w += nthr) v.end[w] = 0;
    for (int w = (B + 31) / 32 + tid; w < wm; w += nthr) v.bad[w] = 0xFFFFFFFFu;  // past the staged bases
    if (tid < 2) {  // slack words unaligned extraction may touch
        v.fA[B / 4 + tid] = 0; v.rA[B / 4 + tid] = 0; v.f2[B / 16 + tid] = 0; v.r2[B / 16 + tid] = 0;
    }
    if (tid < SK_PAD2) { v.f2[-1 - tid] = 0; v.r2[-1 - tid] = 0; }
    // 16 bases per trip: one 128-bit load of raw bytes, 128-bit stores of both ASCII strands, one word
    // each of the 2-bit strands, a halfword of the invalid-base bitmap
    const uint4 *raw128 = reinterpret_cast<const uint4 *>(v.raw);
    uint4 *fA128 = reinterpret_cast<uint4 *>(v.fA), *rA128 = reinterpret_cast<uint4 *>(v.rA);
    uint16_t *badh = reinterpret_cast<uint16_t *>(v.bad);
    const int groups = B / 16;
    for (int g = tid; g < groups; g += nthr) {
        const uint4 raw = raw128[g];
        const Oct o1 = classify8(raw.x, raw.y), o2 = classify8(raw.z, raw.w);
        uint32_t bad16 = o1.bad8 | (o2.bad8 << 8);
        const uint64_t b0 = t0 + (uint64_t)g * 16;
        if (b0 + 16 > sb.n) bad16 |= (b0 >= sb.n) ? 0xFFFFu : (0xFFFFu << (uint32_t)(sb.n - b0)) & 0xFFFFu;
        fA128[g] = make_uint4(o1.fA0, o1.fA1, o2.fA0, o2.fA1);
        const int rg = groups - 1 - g;  // the reverse-complement strand runs the other way
        rA128[rg] = make_uint4(o2.rA0, o2.rA1, o1.rA0, o1.rA1);
        v.f2[g] = o1.f2 | (o2.f2 << 16);
        v.r2[rg] = o2.r2 | (o1.r2 << 16);
        badh[g] = (uint16_t)bad16;
    }
    if (B % 32) {  // B is a multiple of 16: the upper half of the last bad word is past the tile
        if (tid == 0) reinterpret_cast<uint16_t *>(v.bad)[B / 16] = 0xFFFFu;
    }
}

// SK_SHIFTED: copies 1..3 of both ASCII strands (word w of copy c = bytes 4w + c .. 4w + c + 3), after the
// barrier that completes fA / rA.  A k-mer starting at byte s is then words (s >> 2) .. of copy (s & 3).
__device__ __forceinline__ void build_shifted_copies(const TileViews &v, int B) {
    // four words per trip: 128-bit load (+ the next word), three 128-bit stores
    const int quads = (B / 4 + 1 + 3) / 4, stride4 = copy_stride_words(B) / 4;
    for (int q = threadIdx.x; q < 2 * quads; q += blockDim.x) {
        uint32_t *x = (q < quads) ? v.fA : v.rA;
        const int j = (q < quads) ? q : q - quads;
        const uint4 a = reinterpret_cast<const uint4 *>(x)[j];
        const uint32_t n = x[4 * j + 4];  // first word of the next quad (slack words are zeroed)
        uint4 *c = reinterpret_cast<uint4 *>(x);
#pragma unroll
        for (int s = 1; s < 4; s++)
            c[s * stride4 + j] = make_uint4(kb_funnel_r(a.x, a.y, 8 * s), kb_funnel_r(a.y, a.z, 8 * s), kb_funnel_r(a.z, a.w, 8 * s),
                                            kb_funnel_r(a.w, n, 8 * s));
    }
}

// mark the last base of every sequence that ends inside [t0, t0 + B)  (after a barrier that
// follows the zeroing in build_views)
__device__ __forceinline__ void mark_sequence_ends(const TileViews &v, int B, uint64_t t0, const SketchBatch &sb) {
    const int tid = threadIdx.x, nthr = blockDim.x;
    const uint64_t hi = t0 + (uint64_t)B;  // exclusive
    if (sb.offsets == nullptr && sb.read_len == 0) {  // one contiguous sequence ending at n
        if (tid == 0 && sb.n - 1 >= t0 && sb.n - 1 < hi) {
            const uint32_t j = (uint32_t)(sb.n - 1 - t0);
            atomicOr(&v.end[j >> 5], 1u << (j & 31));
        }
    } else if (sb.offsets == nullptr) {
        // one warp does it: the 64-bit division below costs ~150 instructions per WARP, and a tile of reads
        // holds a few dozen read ends at most
        if (tid < 32) {
            const uint64_t L = sb.read_len;
            // ends are at m*L - 1 for m >= 1; first m with m*L - 1 >= t0
            uint64_t m = (t0 + 1 + L - 1) / L;
            if (m == 0) m = 1;
            for (m += tid;; m += 32) {
                const uint64_t e = m * L - 1;
                if (e >= hi || e >= sb.n) break;
                const uint32_t j = (uint32_t)(e - t0);
                atomicOr(&v.end[j >> 5], 1u << (j & 31));
            }
        }
    } else {
        // first sequence s with offsets[s+1] > t0 (its end is the first that can lie in the tile)
        uint64_t a = 0, b = sb.n_seqs;  // invariant: offsets[a'] <= t0 for a' <= a ... search on s+1
        while (a < b) {
            const uint64_t mid = (a + b) >> 1;
            if (sb.offsets[mid + 1] > t0) b = mid; else a = mid + 1;
        }
        for (uint64_t s = a + tid; s < sb.n_seqs; s += nthr) {
            const uint64_t e1 = sb.offsets[s + 1];  // exclusive end, > t0
            if (e1 - 1 >= hi) break;
            const uint32_t j = (uint32_t)(e1 - 1 - t0);
            atomicOr(&v.end[j >> 5], 1u << (j & 31));
        }
    }
}

// sbad[w] for the TILE window starts; reports the first window that the reference would fail on
// (an invalid base inside a window that lies wholly inside one sequence, lib.rs:268-273)
__device__ __forceinline__ void build_start_bitmap(const TileViews &v, uint32_t *sbad, int K, uint64_t t0,
                                                   const SketchBatch &sb, unsigned long long *first_bad) {
    for (int w = threadIdx.x; w < SK_TILE / 32; w += blockDim.x) {
        uint32_t hasbad, crosses;
        if (K <= 64) {
            hasbad = dilate_word(v.bad[w], v.bad[w + 1], v.bad[w + 2], K);
            crosses = dilate_word(v.end[w], v.end[w + 1], v.end[w + 2], K - 1);
        } else {  // generic long k: bit by bit over prefix words
            hasbad = 0; crosses = 0;
            for (int p = 0; p < 32; p++) {
                const int q = w * 32 + p;
                bool hb = false, cr = false;
                for (int j = q; j < q + K; j++) {
                    const uint32_t bit = 1u << (j & 31);
                    hb |= (v.bad[j >> 5] & bit) != 0;
                    if (j < q + K - 1) cr |= (v.end[j >> 5] & bit) != 0;
                }
                hasbad |= (uint32_t)hb << p;
                crosses |= (uint32_t)cr << p;
            }
        }
        // starts at or beyond the limit / the buffer are never used
        const uint64_t q0 = t0 + (uint64_t)w * 32;
        uint32_t beyond = 0;
        if (q0 + 32 > sb.n_limit) beyond = (q0 >= sb.n_limit) ? 0xFFFFFFFFu : (0xFFFFFFFFu << (uint32_t)(sb.n_limit - q0));
        sbad[w] = hasbad | crosses | beyond;
        const uint32_t err = hasbad & ~crosses & ~beyond;
        if (err && first_bad)
            atomicMin(first_bad, (unsigned long long)(sb.pos_base + q0 + (uint32_t)(__ffs(err) - 1)));
    }
}

// Survivors are rare (1 window in 1000 for scaled=1000), so the common path is one predicated
// branch; the threads that do pass aggregate their slot request over whoever is in the branch
// with them (a num sketch that is still filling passes every window: one atomic per warp then).
__device__ __forceinline__ void append_survivor(bool pass, uint64_t h, uint64_t pos0, const SketchBatch &sb,
                                                const SketchOut &out) {
    if (pass) {
        // lane and thread index are read here, inside the rare path, so that no register has to hold
        // them across the k-mer loop; the window start is pos0 + threadIdx.x
        unsigned lane, tid;
        asm volatile("mov.u32 %0, %%laneid;" : "=r"(lane));
        asm volatile("mov.u32 %0, %%tid.x;" : "=r"(tid));
        const unsigned grp = __activemask();
        const int leader = __ffs(grp) - 1;
        unsigned long long base = 0;
        if ((int)lane == leader) base = atomicAdd(out.counter, (unsigned long long)__popc(grp));
        base = __shfl_sync(grp, base, leader);
        const unsigned long long idx = base + __popc(grp & ((1u << lane) - 1u));
        if (idx < out.cap) {
            out.hash[idx] = h;
            if (out.pos) out.pos[idx] = sb.pos_base + pos0 + tid;
        }
    }
}

// ---------------------------------------------------------------------------------------
// fast path: compile-time k-sizes; one launch serves up to three sketches of the same batch
// ---------------------------------------------------------------------------------------
// The k-mer loop of one k-size over a staged tile of B bases: one thread per window start
// i = r * SK_THREADS + tid.  Per-thread constants:
//   2-bit views: word (i >> 4), bit shift 2 * (i & 15); rc(window i) starts at base B - K - i of the
//   reverse-complement views.  ASCII views: a k-mer starting at byte s is words (s >> 2).. of the copy
//   shifted by (s & 3) bytes -- and (s & 3) is the same for all of a thread's windows, because
//   SK_THREADS is a multiple of 32: the r-dependence of every address is a pure word offset.
//   (SK_SHIFTED off: one copy per strand, funnel shifts by 8 * (s & 3); rA then sits (B + 16) bytes after
//   fA (carve_tile), so that one base pointer serves both strands.)
template <int K, int B, int UNROLL>
__device__ __forceinline__ void kmer_loop(const TileViews &v, const uint32_t *sbad, const uint64_t thr, const uint64_t t0,
                                          const SketchBatch &sb, const SketchOut &out) {
    using G = KmerGeom<K>;
    static_assert(SK_THREADS % 32 == 0 && 16 * G::NE - K <= 16 * SK_PAD2, "k-mer loop addressing");
    const int tid = threadIdx.x;
    const int ri0 = B - K - tid, ra0 = B + 16 + ri0;
    // 2-bit k-mers are taken end-aligned (extract2_end): NE words ending at base start + K
    const int ef0 = tid + K - 16 * G::NE, er0 = ri0 + K - 16 * G::NE;  // >= -16 * SK_PAD2
    const uint32_t *qf2 = v.f2 + (ef0 >> 4), *qr2 = v.r2 + (er0 >> 4);  // arithmetic shifts: floor
#if SK_SHIFTED
    constexpr int CS = copy_stride_words(B);  // words between the byte-shifted copies of a strand
    const uint32_t *qfa = v.fA + (tid & 3) * CS + (tid >> 2), *qra = v.rA + (ri0 & 3) * CS + (ri0 >> 2);
    (void)ra0;
#else
    const uint32_t *qfa = v.fA + (tid >> 2), *qra = v.fA + (ra0 >> 2);
    const uint32_t sfa = (uint32_t)tid * 8u, sra = (uint32_t)ra0 * 8u;
#endif
    const uint32_t sf2 = (uint32_t)ef0 * 2u, sr2 = (uint32_t)er0 * 2u;  // funnel shifts use the low 5 bits
    const uint32_t *qsb = sbad + (tid >> 5);
    uint32_t mb = 1u << (tid & 31);
    asm("" : "+r"(mb));  // opaque: keeps the validity test a single LOP3 against a resident mask
    // Prefilter on the high words.  The hash is xs(a) + xs(b) (murmur3_h1_words_parts) and xs keeps the high word, so
    // its high word is hi(a) + hi(b) + carry, carry 0 or 1: h <= thr needs s = hi(a) + hi(b) (mod 2^32) in
    // [0, hi(thr)] or s = 2^32 - 1, i.e. s + 1 <= hi(thr) + 1 (mod 2^32; every s when hi(thr) = 2^32 - 1).  Only the
    // windows that pass finish the hash (two xorshifts, a 64-bit add and compare) and test h <= thr exactly.
    const uint32_t thr_hi = (uint32_t)(thr >> 32);
    uint32_t lim = thr_hi == 0xFFFFFFFFu ? thr_hi : thr_hi + 1u;
    asm("" : "+r"(lim));  // opaque: computed once, not again per window
    // running word pointers: stepped once per UNROLL windows, constant offsets inside
#pragma unroll 1
    for (int r = 0; r < SK_TILE / SK_THREADS; r += UNROLL) {
#pragma unroll
        for (int u = 0; u < UNROLL; u++) {
            const bool valid = (qsb[u * (SK_THREADS / 32)] & mb) == 0;
            uint32_t ef[G::NE], er[G::NE];
            extract2_end<K>(qf2 + u * (SK_THREADS / 16), sf2, ef);
            extract2_end<K>(qr2 - u * (SK_THREADS / 16), sr2, er);  // rc(window i) starts at B - K - i
            const bool use_fw = canonical_is_fw<K>(ef, er);
            uint32_t kw[G::NW];
            const uint32_t *pa = use_fw ? qfa + u * (SK_THREADS / 4) : qra - u * (SK_THREADS / 4);
#if SK_SHIFTED
#pragma unroll
            for (int j = 0; j < G::NW; j++) kw[j] = pa[j];
            kw[G::NW - 1] &= G::TOPA;
#else
            extractAw<K>(pa, use_fw ? sfa : sra, kw);
#endif
            uint64_t a, b;
            murmur3_h1_words_parts<K>(kw, sb.seed, a, b);
            if (valid & ((uint32_t)(a >> 32) + (uint32_t)(b >> 32) + 1u <= lim)) {  // `&`: one test, no early branch
                const uint64_t h = mm_xorshift33(a) + mm_xorshift33(b);
                append_survivor(h <= thr, h, t0 + (uint32_t)((r + u) * SK_THREADS), sb, out);
            }
        }
        qf2 += UNROLL * (SK_THREADS / 16); qr2 -= UNROLL * (SK_THREADS / 16);
        qfa += UNROLL * (SK_THREADS / 4);  qra -= UNROLL * (SK_THREADS / 4);
        qsb += UNROLL * (SK_THREADS / 32);
    }
}

__host__ __device__ constexpr int kmax3(int a, int b, int c) { return a > b ? (a > c ? a : c) : (b > c ? b : c); }

// KB / KC = 0: absent.  The tile (TMA copy, five views, sequence-end bitmap) is staged ONCE and every
// k-size walks it: a multi-k batch (BASELINE cfg2: k = 21, 31, 51 over the same reads) reads each
// base from HBM once and pays the per-base staging work once instead of once per k-size.
template <int KA, int KB, int KC>
__global__ void __launch_bounds__(SK_THREADS, SK_MIN_CTAS) sketch_kernel(const SketchBatch sb, const SketchOuts outs,
                                                                         uint32_t n_tiles) {
    constexpr int B = tile_bases(kmax3(KA, KB, KC));
    extern __shared__ __align__(128) uint8_t s_dyn[];
    __shared__ __align__(8) uint64_t s_bar;
    const TileViews v = carve_tile(s_dyn, B);
    const int tid = threadIdx.x;
    const uint64_t thrA = *outs.o[0].thr;
    const uint64_t thrB = KB ? *outs.o[1].thr : 0;
    const uint64_t thrC = KC ? *outs.o[2].thr : 0;

    // Tiles are handed out dynamically: a CTA's first tile is its block index, every further one
    // comes from an atomic counter.  (With a static round-robin the warp scheduler's fixed priority
    // lets some CTAs run ahead and retire early; the SM then finishes the launch with a third of
    // its warp slots empty -- ncu showed 10.5 of 16 warps per scheduler on average.)
    __shared__ uint32_t s_next;
    if (tid == 0) {
        mbar_init(&s_bar, 1);
        s_next = sb.tile_lo + gridDim.x + atomicAdd(sb.tile_ctr, 1u);
    }
    __syncthreads();
    uint32_t tile = sb.tile_lo + blockIdx.x;
    uint32_t parity = 0;
    if (tid == 0 && tile < n_tiles) {
        const uint64_t t0 = (uint64_t)tile * SK_TILE;
        const uint32_t bytes = tile_copy_bytes(t0, sb.n, B);
        mbar_expect_tx(&s_bar, bytes);
        if (bytes) tma_load_1d(v.raw, sb.buf + t0, bytes, &s_bar);
    }
    while (tile < n_tiles) {
        const uint64_t t0 = (uint64_t)tile * SK_TILE;
        const uint32_t next = s_next;  // written before the last barrier of the previous trip
        uint32_t after_next = 0;
        mbar_wait(&s_bar, parity);
        parity ^= 1u;
        build_views(v, B, t0, sb);
        __syncthreads();  // raw consumed, views + zeroed end bitmap visible
        if (tid == 0) {
            if (next < n_tiles) {  // prefetch: overlaps everything below
                const uint64_t n0 = (uint64_t)next * SK_TILE;
                const uint32_t bytes = tile_copy_bytes(n0, sb.n, B);
                mbar_expect_tx(&s_bar, bytes);
                if (bytes) tma_load_1d(v.raw, sb.buf + n0, bytes, &s_bar);
                after_next = sb.tile_lo + gridDim.x + atomicAdd(sb.tile_ctr, 1u);  // needed one trip from now
            } else {
                after_next = next;
            }
        }
        mark_sequence_ends(v, B, t0, sb);
#if SK_SHIFTED
        build_shifted_copies(v, B);
#endif
        __syncthreads();
        build_start_bitmap(v, v.sbad, KA, t0, sb, outs.first_bad[0]);
        if (KB) build_start_bitmap(v, v.sbad + SK_TILE / 32, KB, t0, sb, outs.first_bad[1]);
        if (KC) build_start_bitmap(v, v.sbad + 2 * (SK_TILE / 32), KC, t0, sb, outs.first_bad[2]);
        __syncthreads();
        // (the fused forms unroll less: three loops unrolled by four no longer fit the instruction cache --
        // ncu showed 11 % `no instruction` stalls)
        constexpr int U = KB ? SK_UNROLL_FUSED : SK_UNROLL;
        kmer_loop<KA, B, U>(v, v.sbad, thrA, t0, sb, outs.o[0]);
        if (KB) kmer_loop<(KB ? KB : KA), B, U>(v, v.sbad + SK_TILE / 32, thrB, t0, sb, outs.o[1]);
        if (KC) kmer_loop<(KC ? KC : KA), B, U>(v, v.sbad + 2 * (SK_TILE / 32), thrC, t0, sb, outs.o[2]);
        if (tid == 0) s_next = after_next;
        __syncthreads();  // views are rebuilt by the next tile
        tile = next;
    }
    if (tid == 0) {  // the last CTA to leave re-arms the counters for the next launch
        __threadfence();
        if (atomicAdd(sb.tile_ctr + 1, 1u) == gridDim.x - 1) {
            sb.tile_ctr[0] = 0;
            sb.tile_ctr[1] = 0;
            __threadfence();
        }
    }
}

// ---------------------------------------------------------------------------------------
// any other k: same staging, byte loops per window
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SK_THREADS) sketch_generic_kernel(const SketchBatch sb, const SketchOut out,
                                                                    uint32_t n_tiles, int K) {
    const int B = SK_TILE + ((K - 1 + 15) / 16) * 16;
    extern __shared__ __align__(128) uint8_t s_dyn[];
    __shared__ __align__(8) uint64_t s_bar;
    const TileViews v = carve_tile(s_dyn, B);
    const int tid = threadIdx.x, lane = tid & 31;
    const uint64_t thr = *out.thr;
    if (tid == 0) mbar_init(&s_bar, 1);
    __syncthreads();
    uint32_t parity = 0;
    for (uint32_t tile = sb.tile_lo + blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const uint64_t t0 = (uint64_t)tile * SK_TILE;
        if (tid == 0) {
            const uint32_t bytes = tile_copy_bytes(t0, sb.n, B);
            mbar_expect_tx(&s_bar, bytes);
            if (bytes) tma_load_1d(v.raw, sb.buf + t0, bytes, &s_bar);
        }
        mbar_wait(&s_bar, parity);
        parity ^= 1u;
        build_views(v, B, t0, sb);
        __syncthreads();
        mark_sequence_ends(v, B, t0, sb);
        __syncthreads();
        build_start_bitmap(v, v.sbad, K, t0, sb, sb.first_bad);
        __syncthreads();
        const uint8_t *fA = reinterpret_cast<const uint8_t *>(v.fA);
        const uint8_t *rA = reinterpret_cast<const uint8_t *>(v.rA);
        for (int r = 0; r < SK_TILE / SK_THREADS; r++) {
            const int i = r * SK_THREADS + tid;
            const bool valid = ((v.sbad[i >> 5] >> (i & 31)) & 1u) == 0;
            uint64_t h = 0;
            if (valid) {
                const uint8_t *f = fA + i;
                const uint8_t *rc = rA + (B - K - i);
                int j = 0;
                while (j < K && f[j] == rc[j]) j++;
                const uint8_t *src = (j < K && f[j] < rc[j]) ? f : rc;  // lib.rs:263-267 (ties -> rc)
                h = murmur3_h1_bytes(src, (uint64_t)K, sb.seed);
            }
            append_survivor(valid && h <= thr, h, t0 + (uint32_t)(r * SK_THREADS), sb, out);
        }
        __syncthreads();
    }
}

bool sketch_has_fast_path(uint32_t K) { return K == 21 || K == 31 || K == 51; }
// distinct fast-path k-sizes in ascending order, two or three of them
bool sketch_multi_supported(const uint32_t *ks, int nk) {
    if (nk < 2 || nk > 3) return false;
    for (int i = 0; i < nk; i++) {
        if (!sketch_has_fast_path(ks[i])) return false;
        if (i && ks[i] <= ks[i - 1]) return false;
    }
    return true;
}

template <int KA, int KB, int KC>
static void launch_fast(const SketchBatch &sb, const SketchOuts &outs, uint32_t n_tiles, unsigned grid, cudaStream_t st) {
    constexpr int NK = 1 + (KB ? 1 : 0) + (KC ? 1 : 0);
    constexpr size_t smem = tile_smem_bytes(tile_bases(kmax3(KA, KB, KC)), NK);
    static bool attr_set = false;
    if (!attr_set) {
        SM_CUDA(cudaFuncSetAttribute(sketch_kernel<KA, KB, KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    sketch_kernel<KA, KB, KC><<<grid, SK_THREADS, smem, st>>>(sb, outs, n_tiles);
}

uint32_t sketch_tile_count(uint64_t n, uint64_t n_limit) {
    const uint64_t span = n_limit < n ? n_limit : n;  // window starts worth visiting
    const uint64_t tiles64 = (span + SK_TILE - 1) / SK_TILE;
    if (tiles64 > 0xFFFFFFFFull) throw_internal("sequence batch too large for one launch");
    return (uint32_t)tiles64;
}
// tiles whose staged bytes (window starts + halo) lie inside the first `bytes_ready` bytes
uint32_t sketch_tiles_ready(uint32_t K, uint64_t bytes_ready) {
    const uint64_t B = SK_TILE + (((uint64_t)K - 1 + 15) / 16) * 16;
    if (bytes_ready < B) return 0;
    return (uint32_t)((bytes_ready - B) / SK_TILE + 1);
}

static unsigned sketch_grid(const SketchBatch &sb, uint32_t tile_hi, int sm_count) {
    unsigned grid = (unsigned)sm_count * SK_CTAS_PER_SM;  // persistent: a multiple of the SM count
    if (grid > tile_hi - sb.tile_lo) grid = tile_hi - sb.tile_lo;
    return grid;
}

void launch_sketch(uint32_t K, const SketchBatch &sb, const SketchOut &out, uint32_t tile_hi, int sm_count,
                   cudaStream_t st) {
    if (sb.n == 0 || sb.n_limit == 0 || K == 0 || tile_hi <= sb.tile_lo) return;
    const uint32_t n_tiles = tile_hi;
    const unsigned grid = sketch_grid(sb, tile_hi, sm_count);
    ProfScope prof(K == 21 ? PROF_SKETCH_K21 : K == 31 ? PROF_SKETCH_K31 : K == 51 ? PROF_SKETCH_K51 : PROF_SKETCH_OTHER, st);
    SketchOuts outs;
    outs.o[0] = out; outs.o[1] = out; outs.o[2] = out;
    outs.first_bad[0] = sb.first_bad; outs.first_bad[1] = nullptr; outs.first_bad[2] = nullptr;
    switch (K) {
    case 21: launch_fast<21, 0, 0>(sb, outs, n_tiles, grid, st); break;
    case 31: launch_fast<31, 0, 0>(sb, outs, n_tiles, grid, st); break;
    case 51: launch_fast<51, 0, 0>(sb, outs, n_tiles, grid, st); break;
    default: {
        if (K > (uint32_t)SK_MAX_GENERIC_K) throw_internal("ksize above 8192 is not supported by the GPU sketcher");
        const int B = SK_TILE + (((int)K - 1 + 15) / 16) * 16;
        const size_t smem = tile_smem_bytes(B);
        SM_CUDA(cudaFuncSetAttribute(sketch_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        sketch_generic_kernel<<<grid, SK_THREADS, smem, st>>>(sb, out, n_tiles, (int)K);
    }
    }
    SM_LAUNCHED();
}

// two or three sketches of the same batch in one launch (sketch_multi_supported(ks, nk)); outs.o[j] /
// outs.first_bad[j] belong to ks[j]; sb.seed and sb.tile_ctr are shared
void launch_sketch_multi(const uint32_t *ks, int nk, const SketchBatch &sb, const SketchOuts &outs, uint32_t tile_hi,
                         int sm_count, cudaStream_t st) {
    if (!sketch_multi_supported(ks, nk)) throw_internal("unsupported k-size combination for the fused sketch kernel");
    if (sb.n == 0 || sb.n_limit == 0 || tile_hi <= sb.tile_lo) return;
    const unsigned grid = sketch_grid(sb, tile_hi, sm_count);
    ProfScope prof(PROF_SKETCH_MULTI, st);
    if (nk == 3) launch_fast<21, 31, 51>(sb, outs, tile_hi, grid, st);
    else if (ks[0] == 21 && ks[1] == 31) launch_fast<21, 31, 0>(sb, outs, tile_hi, grid, st);
    else if (ks[0] == 21 && ks[1] == 51) launch_fast<21, 51, 0>(sb, outs, tile_hi, grid, st);
    else launch_fast<31, 51, 0>(sb, outs, tile_hi, grid, st);
    SM_LAUNCHED();
}

}  // namespace smb200
