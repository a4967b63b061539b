// join.cu -- sparse all-vs-all: find the sketch pairs that share at least one hash with a hash
// table grouped by hash (the probe form: the postings of one side of the block are grouped by hash,
// every hash of the other side looks its run up), so that the merge walk of the reference
// (Intersection, src/lib.rs:515-544, inside intersection_size, lib.rs:470-499) only runs for related
// pairs.  Unrelated pairs have common = 0 and size = min(num, |A| + |B|) by definition, no walk
// needed.  For the untruncated intersection (count_common, lib.rs:428-436; Leaf containment,
// index.rs:146-160) the probe yields the counts directly.  Results are the same integers as the dense
// kernels'.  Sorted (hash, sketch) postings serve only the dense kernel of full num sketches (end of
// this file), which walks ranks of the hashes instead of the hashes.
#include <algorithm>

#include "device.hpp"
#include "kernels.cuh"

namespace smb200 {

static unsigned blocks_for(uint64_t n, unsigned per_block, unsigned cap) {
    uint64_t b = (n + per_block - 1) / per_block;
    if (b == 0) b = 1;
    return (unsigned)(b > cap ? cap : b);
}

// postings of rows [first, first + n_rows): key = hash, val = side << 63 | local row << 32 | position
__global__ void __launch_bounds__(256) postings_kernel(const uint64_t *__restrict__ hashes,
                                                       const uint64_t *__restrict__ offsets, uint64_t first,
                                                       uint64_t n_rows, uint64_t side, uint64_t *__restrict__ keys,
                                                       uint64_t *__restrict__ vals) {
    const int lane = threadIdx.x & 31;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint64_t base = offsets[first];
    for (uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n_rows; r += warps) {
        const uint64_t b = offsets[first + r], e = offsets[first + r + 1];
        for (uint64_t i = b + lane; i < e; i += 32) {
            keys[i - base] = hashes[i];
            vals[i - base] = (side << 63) | (r << 32) | (i - b);
        }
    }
}
void launch_postings(const uint64_t *hashes, const uint64_t *offsets, uint64_t first, uint64_t n_rows, uint64_t side,
                     uint64_t *keys, uint64_t *vals, cudaStream_t st) {
    if (!n_rows) return;
    postings_kernel<<<blocks_for(n_rows * 32, 256, 148 * 16), 256, 0, st>>>(hashes, offsets, first, n_rows, side, keys, vals);
    SM_LAUNCHED();
}

// max over the keys (decides how many radix passes the sort needs)
__global__ void max_u64_kernel(const uint64_t *__restrict__ keys, uint64_t n, unsigned long long *out) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    unsigned long long m = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) m = max(m, (unsigned long long)keys[i]);
    for (int d = 16; d; d >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, d));
    if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}
void launch_max_u64(const uint64_t *keys, uint64_t n, unsigned long long *out, cudaStream_t st) {
    if (!n) return;
    max_u64_kernel<<<blocks_for(n, 256, 148 * 8), 256, 0, st>>>(keys, n, out);
    SM_LAUNCHED();
}

// ---- probe form: the ROW postings are grouped by hash in a hash table; every column hash looks its run up ---
// Used when the row block is much smaller than the column block (a row shard of an all-vs-all matrix,
// a query batch against an index): building the row side costs O(rows) and no sort, which is what lets
// the row-sharded matrix scale with the number of GPUs.
//   group_insert: every row posting claims / finds the slot of its hash (open addressing, linear probing,
//                 atomicCAS) and counts itself there; remembers the slot
//   (exclusive scan of the slot counts = start of each hash's run in `grows`)
//   group_fill:   every row posting writes its local row id into its hash's run
//   probe_group:  one warp per column sketch; each hash finds its slot (an empty slot = no row has it)
//                 and marks (row, column) for every row of the run
// The hash value ~0 cannot be told from an empty slot, so it owns the extra slot T.
constexpr unsigned long long GROUP_EMPTY = ~0ull;
__device__ __forceinline__ uint64_t group_slot0(uint64_t h, int log2_t) { return (h * 0x9E3779B97F4A7C15ull) >> (64 - log2_t); }

__global__ void __launch_bounds__(256) group_insert_kernel(const uint64_t *__restrict__ rh, const uint64_t *__restrict__ ro,
                                                           uint64_t r0, uint64_t nr, unsigned long long *tkey,
                                                           unsigned long long *tcount, uint32_t *slot_of, int log2_t,
                                                           uint32_t *filter, int log2_f, uint32_t split) {
    const int lane = threadIdx.x & 31;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint64_t T = 1ull << log2_t, base = ro[r0];
    // (a sketch is cut into `split` parts, one warp each: a rank's shard of a thousand sketches is otherwise a thousand
    // warps of dependent atomics on a GPU that holds nine thousand)
    for (uint64_t wi = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; wi < nr * split; wi += warps) {
        const uint64_t r = wi / split, part = wi - r * split;
        const uint64_t b0 = ro[r0 + r], len = ro[r0 + r + 1] - b0;
        const uint64_t b = b0 + len * part / split, e = b0 + len * (part + 1) / split;
        for (uint64_t i = b + lane; i < e; i += 32) {
            const unsigned long long h = rh[i];
            uint64_t s;
            if (h == GROUP_EMPTY) {
                s = T;
            } else {
                s = group_slot0(h, log2_t);
                for (;;) {
                    unsigned long long cur = tkey[s];
                    if (cur == GROUP_EMPTY) cur = atomicCAS(&tkey[s], GROUP_EMPTY, h);
                    if (cur == GROUP_EMPTY || cur == h) break;
                    s = (s + 1) & (T - 1);
                }
            }
            atomicAdd(&tcount[s], 1ull);
            slot_of[i - base] = (uint32_t)s;
            if (filter) {  // presence bit (see probe_group_kernel)
                const uint64_t fb = (h * 0xD6E8FEB86659FD93ull) >> (64 - log2_f);
                const uint32_t m = 1u << (fb & 31);
                if (!(filter[fb >> 5] & m)) atomicOr(&filter[fb >> 5], m);
            }
        }
    }
}
__global__ void __launch_bounds__(256) group_fill_kernel(const uint64_t *__restrict__ ro, uint64_t r0, uint64_t nr,
                                                         const uint32_t *__restrict__ slot_of, const uint64_t *__restrict__ toff,
                                                         uint32_t *tcursor, uint32_t *grows, uint32_t split) {
    const int lane = threadIdx.x & 31;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint64_t base = ro[r0];
    for (uint64_t wi = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; wi < nr * split; wi += warps) {
        const uint64_t r = wi / split, part = wi - r * split;
        const uint64_t b0 = ro[r0 + r], len = ro[r0 + r + 1] - b0;
        const uint64_t b = b0 + len * part / split, e = b0 + len * (part + 1) / split;
        for (uint64_t i = b + lane; i < e; i += 32) {
            const uint32_t s = slot_of[i - base];
            grows[toff[s] + atomicAdd(&tcursor[s], 1u)] = (uint32_t)r;
        }
    }
}
// The table is built over one side of the block (the smaller one: "build" side, `grows` holds its local
// sketch ids) and probed with the sketches of the other; BUILD_COLS tells which is which.
// COUNT: atomicAdd into cmat[r * ld + c], else set the pair's bit in the related-pairs bitmap, which is
// PROBE-major (bit = p * n_build + b): a warp works on one probing sketch, so all its bit tests --
// hundreds per pair it ends up marking -- fall into one n_build-bit stretch.
// *incidences += number of (build sketch, probe hash) hits.
template <bool COUNT, bool BUILD_COLS>
__global__ void __launch_bounds__(256) probe_group_kernel(const unsigned long long *__restrict__ tkey,
                                                          const uint64_t *__restrict__ toff, const uint32_t *__restrict__ grows,
                                                          int log2_t, const uint64_t *__restrict__ ph,
                                                          const uint64_t *__restrict__ po, uint64_t p0, uint64_t np, uint32_t *cmat,
                                                          uint64_t ld, unsigned long long *bitmap, uint64_t n_build,
                                                          unsigned long long *incidences, const uint32_t *__restrict__ filter,
                                                          int log2_f, bool smem_rows, uint32_t split) {
    // `filter` (optional): one presence bit per build-side hash in a table small enough to stay in L2.  When
    // the two sides are unrelated collections (a query batch against an index) almost every probing hash is
    // turned away by that one bit instead of a random read in the (much larger) key table.
    const int lane = threadIdx.x & 31;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint64_t T = 1ull << log2_t;
    unsigned long long local = 0;
    // bitmap mode with a build side of up to PROBE_SMEM_ROWS sketches: one shared-memory bitmap per warp
    extern __shared__ uint32_t s_probe[];
    const uint32_t row_words = (uint32_t)((n_build + 31) / 32);
    uint32_t *s_rows = (!COUNT && smem_rows) ? s_probe + (threadIdx.x >> 5) * row_words : nullptr;
    // A probing sketch is cut into `split` parts, one warp each: in a row shard of an all-vs-all matrix only the few
    // sketches related to the shard's rows have any hits, and one warp per sketch left most of the GPU idle while
    // those few warps walked their runs (8 GPUs, cfg3: 1 250 busy warps of 10 000).
    for (uint64_t wi = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; wi < np * split; wi += warps) {
        const uint64_t p = wi / split, part = wi - p * split;
        const uint64_t b0 = po[p0 + p], len = po[p0 + p + 1] - b0;
        const uint64_t b = b0 + len * part / split, e = b0 + len * (part + 1) / split;
        // bit of (p, build sketch 0); computed here, not in the loops: there ptxas spilled in the bitmap instances
        const uint64_t p_bits = p * n_build;
        if (s_rows) {
            for (uint32_t w = lane; w < row_words; w += 32) s_rows[w] = 0;
            __syncwarp();
        }
        for (uint64_t i = b + lane; i < e; i += 32) {
            const unsigned long long h = ph[i];
            if (filter) {
                const uint64_t fb = (h * 0xD6E8FEB86659FD93ull) >> (64 - log2_f);
                if (!((filter[fb >> 5] >> (fb & 31)) & 1u)) continue;
            }
            uint64_t s;
            if (h == GROUP_EMPTY) {
                s = T;
            } else {
                s = group_slot0(h, log2_t);
                for (;;) {
                    const unsigned long long cur = tkey[s];
                    if (cur == h) break;
                    if (cur == GROUP_EMPTY) { s = ~0ull; break; }
                    s = (s + 1) & (T - 1);
                }
                if (s == ~0ull) continue;
            }
            const uint64_t jb = toff[s], je = toff[s + 1];
            local += je - jb;
            uint64_t j = jb;
            if (!COUNT && s_rows) {
                // related rows of this probing sketch are collected in the warp's shared-memory bitmap: the
                // hundreds of repeat hits per pair cost a shared-memory test, not a global one
                // (four row ids per trip, loaded together: the loop is otherwise one dependent L2 load per incidence)
                for (; j + 4 <= je; j += 4) {
                    const uint32_t q0 = __ldg(&grows[j]), q1 = __ldg(&grows[j + 1]), q2 = __ldg(&grows[j + 2]), q3 = __ldg(&grows[j + 3]);
                    const uint32_t m0 = 1u << (q0 & 31), m1 = 1u << (q1 & 31), m2 = 1u << (q2 & 31), m3 = 1u << (q3 & 31);
                    if (!(s_rows[q0 >> 5] & m0)) atomicOr(&s_rows[q0 >> 5], m0);
                    if (!(s_rows[q1 >> 5] & m1)) atomicOr(&s_rows[q1 >> 5], m1);
                    if (!(s_rows[q2 >> 5] & m2)) atomicOr(&s_rows[q2 >> 5], m2);
                    if (!(s_rows[q3 >> 5] & m3)) atomicOr(&s_rows[q3 >> 5], m3);
                }
                for (; j < je; j++) {
                    const uint32_t q = __ldg(&grows[j]);
                    const uint32_t m = 1u << (q & 31);
                    if (!(s_rows[q >> 5] & m)) atomicOr(&s_rows[q >> 5], m);
                }
            }
            for (; j < je; j++) {
                const uint64_t q = grows[j];
                if (COUNT) {
                    atomicAdd(BUILD_COLS ? &cmat[p * ld + q] : &cmat[q * ld + p], 1u);
                } else {
                    const uint64_t bit = p_bits + q;
                    const unsigned long long m = 1ull << (bit & 63);
                    if (!(__ldcg(&bitmap[bit >> 6]) & m)) atomicOr(&bitmap[bit >> 6], m);  // L2 view: atomics land there
                }
            }
        }
        if (s_rows) {  // flush the warp's row set into the probe-major global bitmap (32 rows per word, any alignment)
            __syncwarp();
            for (uint32_t w = lane; w < row_words; w += 32) {
                const unsigned long long v = s_rows[w];
                if (v) {
                    const uint64_t g = p_bits + 32ull * w;
                    const unsigned sh = (unsigned)(g & 63);
                    atomicOr(&bitmap[g >> 6], v << sh);
                    if (sh > 32) atomicOr(&bitmap[(g >> 6) + 1], v >> (64 - sh));
                }
            }
            __syncwarp();
        }
    }
    for (int d = 16; d; d >>= 1) local += __shfl_xor_sync(0xFFFFFFFFu, local, d);
    if (lane == 0 && local) atomicAdd(incidences, local);
}
constexpr uint64_t PROBE_SMEM_ROWS = 65536;  // 8 KB of bitmap per warp, 64 KB per CTA
void launch_group_insert(const uint64_t *rh, const uint64_t *ro, uint64_t r0, uint64_t nr, unsigned long long *tkey,
                         unsigned long long *tcount, uint32_t *slot_of, int log2_t, uint32_t *filter, int log2_f, cudaStream_t st) {
    if (!nr) return;
    const uint32_t split = nr >= 16384 ? 1u : (uint32_t)std::min<uint64_t>(16, (16384 + nr - 1) / nr);
    group_insert_kernel<<<blocks_for(nr * split * 32, 256, 148 * 16), 256, 0, st>>>(rh, ro, r0, nr, tkey, tcount, slot_of, log2_t,
                                                                                   filter, log2_f, split);
    SM_LAUNCHED();
}
void launch_group_fill(const uint64_t *ro, uint64_t r0, uint64_t nr, const uint32_t *slot_of, const uint64_t *toff,
                       uint32_t *tcursor, uint32_t *grows, cudaStream_t st) {
    if (!nr) return;
    const uint32_t split = nr >= 16384 ? 1u : (uint32_t)std::min<uint64_t>(16, (16384 + nr - 1) / nr);
    group_fill_kernel<<<blocks_for(nr * split * 32, 256, 148 * 16), 256, 0, st>>>(ro, r0, nr, slot_of, toff, tcursor, grows, split);
    SM_LAUNCHED();
}
void launch_probe_group(bool count, bool build_cols, const unsigned long long *tkey, const uint64_t *toff, const uint32_t *grows,
                        int log2_t, const uint64_t *ph, const uint64_t *po, uint64_t p0, uint64_t np, uint32_t *cmat, uint64_t ld,
                        unsigned long long *bitmap, uint64_t n_build, unsigned long long *incidences, const uint32_t *filter,
                        int log2_f, cudaStream_t st) {
    if (!np) return;
    ProfScope prof(PROF_PROBE, st);
    const bool smem_rows = !count && n_build <= PROBE_SMEM_ROWS;
    const size_t smem = smem_rows ? 8 * ((n_build + 31) / 32) * 4 : 0;
    // resident CTAs are limited by the shared-memory bitmaps: size the grid to what fits, a multiple of the SM count
    unsigned per_sm = 8;
    if (smem) per_sm = (unsigned)std::max<size_t>(1, std::min<size_t>(8, (200 * 1024) / (smem + 1024)));
    const uint32_t split = np >= 32768 ? 1u : (uint32_t)std::min<uint64_t>(8, (32768 + np - 1) / np);
    const unsigned grid = blocks_for(np * split * 32, 256, 148 * std::max(2u, per_sm * 2));
    static bool attr_set = false;
    if (!attr_set) {
        SM_CUDA(cudaFuncSetAttribute(probe_group_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        SM_CUDA(cudaFuncSetAttribute(probe_group_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        attr_set = true;
    }
#define SM_PROBE(C, B) probe_group_kernel<C, B><<<grid, 256, smem, st>>>(tkey, toff, grows, log2_t, ph, po, p0, np, cmat, ld, bitmap, n_build, incidences, filter, log2_f, smem_rows, split)
    if (count) { if (build_cols) SM_PROBE(true, true); else SM_PROBE(true, false); }
    else { if (build_cols) SM_PROBE(false, true); else SM_PROBE(false, false); }
#undef SM_PROBE
    SM_LAUNCHED();
}

// bitmap -> per-word population counts (u64, for the scan)
__global__ void popc_words_kernel(const unsigned long long *__restrict__ bitmap, uint64_t n_words, uint64_t *counts) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += stride) counts[w] = __popcll(bitmap[w]);
}
void launch_popc_words(const unsigned long long *bitmap, uint64_t n_words, uint64_t *counts, cudaStream_t st) {
    if (!n_words) return;
    popc_words_kernel<<<blocks_for(n_words, 256, 148 * 16), 256, 0, st>>>(bitmap, n_words, counts);
    SM_LAUNCHED();
}
// pairs[pre[w] + k] = index of the k-th set bit of word w (cell id r * nc + c, ascending)
__global__ void expand_bits_kernel(const unsigned long long *__restrict__ bitmap, const uint64_t *__restrict__ pre,
                                   uint64_t n_words, uint64_t *pairs, uint64_t cap) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += stride) {
        unsigned long long m = bitmap[w];
        uint64_t o = pre[w];
        while (m) {
            const int b = __ffsll((long long)m) - 1;
            if (o < cap) pairs[o] = w * 64 + (uint64_t)b;
            o++;
            m &= m - 1;
        }
    }
}
void launch_expand_bits(const unsigned long long *bitmap, const uint64_t *pre, uint64_t n_words, uint64_t *pairs,
                        cudaStream_t st, uint64_t cap) {
    if (!n_words) return;
    expand_bits_kernel<<<blocks_for(n_words, 256, 148 * 16), 256, 0, st>>>(bitmap, pre, n_words, pairs, cap);
    SM_LAUNCHED();
}

// every cell of the block as if the pair were unrelated (mode 0), or finished from the counts (mode 1).
// One CTA row per block row (blockIdx.y strides over rows, threads over columns): no index division, the
// row's length and num are read once per row, writes are coalesced along the row.
__global__ void __launch_bounds__(256) fill_cells_kernel(const uint64_t *__restrict__ ro, const uint32_t *__restrict__ rnum,
                                                         uint64_t r0, uint64_t nr, const uint64_t *__restrict__ co,
                                                         uint64_t c0, uint64_t nc, int mode, const uint32_t *cmat,
                                                         uint64_t cld, uint32_t *common, uint32_t *size, double *ratio,
                                                         uint64_t ld) {
    for (uint64_t i = blockIdx.y; i < nr; i += gridDim.y) {
        const uint32_t na = (uint32_t)(ro[r0 + i + 1] - ro[r0 + i]);
        const uint32_t num = rnum ? rnum[r0 + i] : 0;
        for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < nc; j += (uint64_t)gridDim.x * blockDim.x) {
            uint32_t cm, sz;
            double den;
            if (mode == 0) {
                const uint32_t nb = (uint32_t)(co[c0 + j + 1] - co[c0 + j]);
                const uint64_t uni = (uint64_t)na + nb;
                cm = 0;
                sz = (uint32_t)((num != 0 && uni >= num) ? num : uni);  // lib.rs:391-401
                den = (double)(sz > 1 ? sz : 1);
            } else {
                cm = cmat[i * cld + j];
                sz = na;  // index.rs:152-154: the row (node) sketch is the denominator
                den = (double)sz;
            }
            const size_t at = (size_t)i * ld + j;
            if (common) common[at] = cm;
            if (size) size[at] = sz;
            // 0 / den is +0.0 for every den > 0 (0 / 0 stays NaN below): nearly every cell of a sparse block, and
            // an FP64 division is a ~100-instruction sequence
            if (ratio) ratio[at] = (cm == 0 && den > 0.0) ? 0.0 : (double)cm / den;
        }
    }
}
void launch_fill_cells(const uint64_t *ro, const uint32_t *rnum, uint64_t r0, uint64_t nr, const uint64_t *co, uint64_t c0,
                       uint64_t nc, int mode, const uint32_t *cmat, uint64_t cld, uint32_t *common, uint32_t *size,
                       double *ratio, uint64_t ld, cudaStream_t st) {
    if (!nr || !nc) return;
    ProfScope prof(PROF_FILL, st);
    const unsigned gx = (unsigned)std::min<uint64_t>((nc + 255) / 256, 64);
    const unsigned gy = (unsigned)std::min<uint64_t>(nr, std::max<uint64_t>(1, (148 * 32) / gx));
    fill_cells_kernel<<<dim3(gx, gy), 256, 0, st>>>(ro, rnum, r0, nr, co, c0, nc, mode, cmat, cld, common, size, ratio, ld);
    SM_LAUNCHED();
}

// the reference's merge walk for the listed related pairs only (cell id = i * nc + j)
__global__ void __launch_bounds__(256) walk_pairs_kernel(const uint64_t *__restrict__ pairs, uint64_t n_pairs,
                                                         const uint64_t *__restrict__ rh, const uint64_t *__restrict__ ro,
                                                         const uint32_t *__restrict__ rnum, uint64_t r0,
                                                         const uint64_t *__restrict__ ch, const uint64_t *__restrict__ co,
                                                         uint64_t c0, uint64_t nc, uint32_t *common, uint32_t *size,
                                                         double *ratio, uint64_t ld, const uint64_t *n_dev_a,
                                                         const uint64_t *n_dev_b, uint64_t nr_transposed, bool symmetric) {
    // the pair count either comes from the host or is read here as *n_dev_a + *n_dev_b (the tail of the
    // bitmap scan), capped by n_pairs: the launch then needs no host round trip
    if (n_dev_a) {
        const uint64_t nd = *n_dev_a + *n_dev_b;
        if (nd < n_pairs) n_pairs = nd;
    }
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n_pairs; t += stride) {
        const uint64_t cell = pairs[t];
        uint64_t i, j;
        if (nr_transposed) { j = cell / nr_transposed; i = cell - j * nr_transposed; }  // column-major cell ids (probe join)
        else { i = cell / nc; j = cell - i * nc; }
        // rows and columns are the same sketches with one `num`: compare(a, b) == compare(b, a) (lib.rs:470-508 is
        // symmetric but for self.num), so a pair is walked once and written to both cells
        if (symmetric && i > j) continue;
        const uint64_t ab = ro[r0 + i], bb = co[c0 + j];
        const uint32_t na = (uint32_t)(ro[r0 + i + 1] - ab), nb = (uint32_t)(co[c0 + j + 1] - bb);
        const uint32_t num = rnum ? rnum[r0 + i] : 0;
        const uint32_t limit = num ? num : 0xFFFFFFFFu;
        const uint64_t *a = rh + ab, *b = ch + bb;
        uint32_t x_i = 0, y_j = 0, c = 0, u = 0;
        // lib.rs:470-499 in one pass.  The walk goes in stretches of s = min(left in A, left in B, left of the limit)
        // steps: a step advances either side by at most one element, so inside a stretch neither list can run out and
        // the step needs no bounds test at all -- two 64-bit compares, the count, and per side a predicated
        // "take the element loaded two steps ahead, load the one after" (a row is followed by at least three readable
        // hashes: the next row's, or the slack at the end of the CSR).  Two elements ahead, because the loads come from
        // L2 (~300 cycles) and a step is ~20 instructions: one element ahead left the walk waiting on them
        // (ncu: issue slots 55 % busy, long-scoreboard stalls on top).  Lists of similar length need 2-4 stretches.
        const uint64_t *pa = a, *pb = b;
        uint64_t x = __ldg(pa), y = __ldg(pb);
        uint64_t xn = __ldg(pa + 1), yn = __ldg(pb + 1);
        uint64_t xnn = __ldg(pa + 2), ynn = __ldg(pb + 2);
        for (;;) {
            uint32_t s = min(min(na - x_i, nb - y_j), limit - u);
            if (s == 0) break;
            u += s;
#pragma unroll 2
            for (; s; s--) {
                const bool adv_a = x <= y, adv_b = y <= x;
                c += (adv_a && adv_b);
                if (adv_a) { x = xn; xn = xnn; pa++; xnn = __ldg(pa + 2); }
                if (adv_b) { y = yn; yn = ynn; pb++; ynn = __ldg(pb + 2); }
            }
            x_i = (uint32_t)(pa - a);
            y_j = (uint32_t)(pb - b);
        }
        const uint64_t uni = (uint64_t)u + (na - x_i) + (nb - y_j);
        const uint32_t sz = (uint32_t)((num != 0 && uni >= num) ? num : uni);
        const size_t at = (size_t)i * ld + j;
        const double rt = (double)c / (double)(sz > 1 ? sz : 1);
        if (common) common[at] = c;
        if (size) size[at] = sz;
        if (ratio) ratio[at] = rt;
        if (symmetric && i != j) {
            const size_t ta = (size_t)j * ld + i;
            if (common) common[ta] = c;
            if (size) size[ta] = sz;
            if (ratio) ratio[ta] = rt;
        }
    }
}
void launch_walk_pairs(const uint64_t *pairs, uint64_t n_pairs, const uint64_t *rh, const uint64_t *ro, const uint32_t *rnum,
                       uint64_t r0, const uint64_t *ch, const uint64_t *co, uint64_t c0, uint64_t nc, uint32_t *common,
                       uint32_t *size, double *ratio, uint64_t ld, cudaStream_t st, const uint64_t *n_dev_a,
                       const uint64_t *n_dev_b, uint64_t nr_transposed, bool symmetric) {
    if (!n_pairs) return;
    ProfScope prof(PROF_WALK, st);
    walk_pairs_kernel<<<blocks_for(n_pairs, 256, 148 * 16), 256, 0, st>>>(pairs, n_pairs, rh, ro, rnum, r0, ch, co, c0, nc, common,
                                                                        size, ratio, ld, n_dev_a, n_dev_b, nr_transposed, symmetric);
    SM_LAUNCHED();
}

}  // namespace smb200

// =====================================================================================
// Dense path for FULL num sketches (every sketch of the block holds exactly L = num hashes):
// the hashes are replaced by their dense ranks (u32) among all hashes of the block -- order and
// equality are preserved, so the merge walk sees the same comparisons -- and the walk becomes a
// loop of exactly L steps (the union of two full sketches always has >= num elements, so
// intersection_size stops after num union elements, lib.rs:470-499).
// =====================================================================================
namespace smb200 {

// sorted postings -> rank of every posting's hash, scattered back to sketch order:
// out[(side ? b_base : 0) + row * L + pos] = number of distinct hashes smaller than it
__global__ void __launch_bounds__(256) scatter_ranks_kernel(const uint64_t *__restrict__ keys,
                                                            const uint64_t *__restrict__ vals,
                                                            const uint64_t *__restrict__ pre, uint64_t n, uint32_t L,
                                                            uint64_t b_base, uint32_t *__restrict__ out) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const bool head = (i == 0) || keys[i] != keys[i - 1];
        const uint64_t rank = pre[i] + (head ? 1 : 0) - 1;  // pre = exclusive scan of the head flags
        const uint64_t v = vals[i];
        const uint64_t row = (v >> 32) & 0x7FFFFFFFull, pos = v & 0xFFFFFFFFull;
        out[((v >> 63) ? b_base : 0) + row * L + pos] = (uint32_t)rank;
    }
}
void launch_scatter_ranks(const uint64_t *keys, const uint64_t *vals, const uint64_t *pre, uint64_t n, uint32_t L,
                          uint64_t b_base, uint32_t *out, cudaStream_t st) {
    if (!n) return;
    scatter_ranks_kernel<<<blocks_for(n, 256, 148 * 16), 256, 0, st>>>(keys, vals, pre, n, L, b_base, out);
    SM_LAUNCHED();
}

// CTA = 32 rows x 32 columns = 1024 pairs = 1024 threads.  Both tiles sit in shared memory
// element-major, [element][sketch]: the lane that owns sketch s always touches bank s.  Warp w
// takes the w-th diagonal: lane l walks (row l, column (l + w) mod 32), so within a warp every
// row AND every column is used by exactly one lane -- no bank conflict on either operand, whatever
// the two walk positions are.  One extra all-ones element per sketch stops a finished list.
constexpr int CF_THREADS = 1024;
__global__ void __launch_bounds__(CF_THREADS, 1)
compare_full_kernel(const uint32_t *__restrict__ ra, const uint32_t *__restrict__ rb, uint32_t L, uint64_t nr,
                    uint64_t nc, uint32_t *common, uint32_t *size, double *ratio, uint64_t ld) {
    extern __shared__ __align__(16) uint32_t s_rank[];  // A: (L+1) x 32, then B: (L+1) x 32
    uint32_t *sA = s_rank, *sB = s_rank + (size_t)(L + 1) * 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t row0 = (uint64_t)blockIdx.y * 32, col0 = (uint64_t)blockIdx.x * 32;
    // stage: lane <-> sketch (bank = lane), warp strides over the elements
    {
        const uint64_t r = min(row0 + lane, nr - 1), c = min(col0 + lane, nc - 1);
        const uint32_t *ga = ra + r * L, *gb = rb + c * L;
        for (uint32_t e = warp; e < L; e += CF_THREADS / 32) {
            sA[e * 32 + lane] = __ldg(ga + e);
            sB[e * 32 + lane] = __ldg(gb + e);
        }
        if (warp == 0) { sA[L * 32 + lane] = 0xFFFFFFFFu; sB[L * 32 + lane] = 0xFFFFFFFFu; }
    }
    __syncthreads();
    const int cl = (lane + warp) & 31;
    // walk with two shared-memory byte addresses only: per step two compares, two predicated
    // address bumps, two loads
    const uint32_t a0 = (uint32_t)__cvta_generic_to_shared(sA + lane), b0 = (uint32_t)__cvta_generic_to_shared(sB + cl);
    uint32_t pa = a0, pb = b0;
    uint32_t x, y;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(x) : "r"(pa));
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(y) : "r"(pb));
#pragma unroll 8
    for (uint32_t u = 0; u < L; u++) {  // one union element per step
        if (x <= y) pa += 128;
        if (y <= x) pb += 128;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(x) : "r"(pa));
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(y) : "r"(pb));
    }
    // every step consumes one element of A, of B, or (when equal) one of each: i + j = L + common
    const uint32_t c = ((pa - a0) + (pb - b0)) / 128 - L;
    const uint64_t row = row0 + lane, col = col0 + cl;
    if (row < nr && col < nc) {
        const size_t at = (size_t)row * ld + col;
        if (common) common[at] = c;
        if (size) size[at] = L;
        if (ratio) ratio[at] = (double)c / (double)(L > 1 ? L : 1);
    }
}
bool compare_full_fits(uint32_t L) { return L >= 1 && (size_t)(L + 1) * 32 * 4 * 2 <= 220 * 1024; }
void launch_compare_full(const uint32_t *ra, const uint32_t *rb, uint32_t L, uint64_t nr, uint64_t nc, uint32_t *common,
                         uint32_t *size, double *ratio, uint64_t ld, cudaStream_t st) {
    if (!nr || !nc) return;
    const size_t smem = (size_t)(L + 1) * 32 * 4 * 2;
    SM_CUDA(cudaFuncSetAttribute(compare_full_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((unsigned)((nc + 31) / 32), (unsigned)((nr + 31) / 32));
    if (grid.y > 65535) throw_internal("row block too tall for one launch");
    ProfScope prof(PROF_COMPARE, st);
    compare_full_kernel<<<grid, CF_THREADS, smem, st>>>(ra, rb, L, nr, nc, common, size, ratio, ld);
    SM_LAUNCHED();
}

}  // namespace smb200
