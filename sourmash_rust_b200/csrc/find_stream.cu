// find_stream.cu -- LinearIndex::find (src/index/linear.rs:25-45) over a large index, HBM-bound.
//
// The count |node n query| of every (index sketch, query) cell decides containment (index.rs:146-160) and, for
// sketches without a `num`, similarity (lib.rs:470-508).  One search streams the whole index past the query batch
// once; the index is 10^2-10^3 times larger than the batch (BASELINE config 4: 40 GB against 40 MB), so the
// search can run at the rate HBM delivers the index -- if each index hash costs no more than a few instructions
// and no off-chip access of its own.  The join of collection.cu answers "is this hash in any query" with a read of
// a bit table in L2 (random 32-byte sector per hash: 840 GB/s of index, 13 % of HBM).  Here that test is on chip:
//
//   * the hash range is cut into P equal slices ("partitions"); a sorted sketch meets slice p in ONE contiguous
//     stretch, whose bounds are kept with the index (part_offsets, built once per collection in one pass);
//   * per slice, the query hashes that fall into it go into a Bloom filter of 2^20 bits (two probes): 128 KB,
//     which fits the shared memory of an SM (blocked: one word, three bits per hash; ~0.8 % false positives);
//   * a CTA belongs to one slice (P = SM count / CTAs per slice), holds that slice's filter in shared memory and
//     streams the rows' stretches past it with coalesced loads: per index hash one 32-bit multiply and one
//     shared-memory read; its warps take groups of 32 rows from the slice's counter, no barrier in the loop;
//   * only the hashes the filter lets through (true hits + ~1 % false positives) go to the exact table in global
//     memory (hash -> list of the queries holding it; built slice by slice in shared memory) and add to the count matrix.  They are parked in the
//     warp's shared-memory queue, so that a warp step does not wait for an off-chip table read (with the lookup
//     inline, half of all warp steps stalled on one: 566 GB/s).  Normally the queues are written out to global memory
//     and looked up by a second kernel: the exact table is BUILT on another stream while the index streams (the build
//     is a third of a search at BASELINE config 4).  If the written-out list overflows its buffer (a heavily related
//     index), the block is run again with the lookups done inside the probe kernel, queue by queue.
#include <algorithm>

#include "device.hpp"
#include "kernels.cuh"

namespace smb200 {

namespace {

constexpr int FS_THREADS = 1024;
constexpr int FS_LOG2_F = 20;                              // filter bits per slice
constexpr int FS_LOADS = 4;                                // pipelined loads per row and lane: stretches of up to 128 hashes
constexpr uint32_t FS_FILTER_WORDS = (1u << FS_LOG2_F) / 32;
constexpr unsigned long long FS_EMPTY = ~0ull;

// Blocked Bloom filter: ONE 32-bit multiplicative hash of the folded hash picks a 32-bit word of the slice's filter (its
// top 15 bits) and three bit positions inside that word (its low 15 bits): one shared-memory read and a dozen
// instructions per index hash.  (The hashes are MurmurHash3 outputs; within a slice their high bits are all but
// constant, the low ones uniform.)  At 68 K keys per slice: ~2 keys per word, ~0.8 % false positives.
__device__ __forceinline__ void filter_word_mask(uint64_t h, uint32_t &word, uint32_t &mask) {
    const uint32_t m = ((uint32_t)h ^ (uint32_t)(h >> 32)) * 0x9E3779B1u;
    word = m >> (32 - (FS_LOG2_F - 5));
    mask = (1u << (m & 31)) | (1u << ((m >> 5) & 31)) | (1u << ((m >> 10) & 31));
}
__device__ __forceinline__ bool filter_test(const uint32_t *f, uint64_t h) {
    uint32_t word, mask;
    filter_word_mask(h, word, mask);
    return (f[word] & mask) == mask;
}
// slice of the hash range a hash falls into: monotone in h, P - 1 for the largest hash of the index
// (scale = floor(2^64 * P / (top + 1)), saturated)
__device__ __forceinline__ uint32_t slice_of(uint64_t h, uint64_t scale, uint32_t P) {
    const unsigned long long q = __umul64hi((unsigned long long)h, (unsigned long long)scale);
    return q < (unsigned long long)(P - 1) ? (uint32_t)q : P - 1;
}

// largest hash of the collection (rows are sorted: the last element of each)
__global__ void rows_max_kernel(const uint64_t *__restrict__ h, const uint64_t *__restrict__ off, uint64_t n_rows,
                                unsigned long long *out) {
    unsigned long long m = 0;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += stride) {
        const uint64_t b = off[r], e = off[r + 1];
        if (e > b) m = max(m, (unsigned long long)h[e - 1]);
    }
    for (int d = 16; d; d >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, d));
    if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

// part_off[q * n_rows + r] = number of hashes of row r below slice q (q = 0 .. P): slice p of row r is
// [part_off[p], part_off[p + 1]).  One warp per row, one pass over its hashes.
__global__ void __launch_bounds__(256) part_offsets_kernel(const uint64_t *__restrict__ h, const uint64_t *__restrict__ off,
                                                           uint64_t n_rows, uint64_t scale, uint32_t P, uint32_t *__restrict__ part_off) {
    const int lane = threadIdx.x & 31;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n_rows; r += warps) {
        const uint64_t b = off[r], e = off[r + 1];
        const uint32_t len = (uint32_t)(e - b);
        for (uint32_t i = lane; i < len; i += 32) {
            const int64_t cur = slice_of(h[b + i], scale, P);
            const int64_t prev = i ? (int64_t)slice_of(h[b + i - 1], scale, P) : -1;
            for (int64_t q = prev + 1; q <= cur; q++) part_off[(uint64_t)q * n_rows + r] = i;
        }
        if (lane == 0) {
            const int64_t last = len ? (int64_t)slice_of(h[e - 1], scale, P) : -1;
            for (int64_t q = last + 1; q <= (int64_t)P; q++) part_off[(uint64_t)q * n_rows + r] = len;
        }
    }
}

// Bloom filters of the query hashes, one per slice (global memory; the probe kernel copies a slice's filter into
// shared memory).  Query hashes above the largest hash of the index cannot occur in it: skipped.
__global__ void __launch_bounds__(256) filters_build_kernel(const uint64_t *__restrict__ qh, uint64_t n, uint64_t scale, uint64_t top,
                                                            uint32_t P, uint32_t *filters) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint64_t h = qh[i];
        if (h > top) continue;
        uint32_t word, mask;
        filter_word_mask(h, word, mask);
        atomicOr(&filters[(size_t)slice_of(h, scale, P) * FS_FILTER_WORDS + word], mask);
    }
}

struct StreamArgs {
    const uint64_t *ih, *io;       // index CSR
    uint64_t b0, bn;               // block of index rows
    const uint32_t *part_off;      // [(P + 1)][n_rows_total]
    uint64_t n_rows_total;
    uint32_t P;
    const uint32_t *filters;       // [P][FS_FILTER_WORDS]
    // exact table over the query hashes (qtable_*_kernel): the hash range is cut into QT_SLICES table slices, slice t
    // owns slots [tstart[t], tstart[t + 1]) (twice its keys), open addressing inside; every posting (query hash
    // occurrence) is a node of its hash's list, node i = posting i of the packed query array
    const unsigned long long *tkey;
    const int32_t *thead;          // slot -> first node, -1 = none
    const int32_t *node_next;
    const uint32_t *node_q;        // node -> query id
    const uint32_t *tstart;        // QT_SLICES + 1
    uint64_t tscale, top;          // table slice of h = min(QT_SLICES - 1, mulhi(h, tscale)); no key above top
    uint32_t *cmat;                // [bn][ld] counts; all zero on entry
    uint64_t ld;
    uint32_t *touched_bits;        // bn bits, zero on entry: rows with at least one count
    uint32_t *touched_rows;        // the same rows as a list ...
    unsigned long long *n_touched; // ... of this many entries
    uint32_t *work_ctr;            // P zeroed counters: next group of 32 rows of each slice
    uint32_t ctas_per_slice;
    // deferred mode: the hashes the filter lets through are not looked up by the probe kernel at all (the exact table is
    // being built on another stream meanwhile) but written out; resolve_spill_kernel looks them up afterwards
    uint64_t *spill_hash;          // nullptr = resolve inside the probe kernel
    uint32_t *spill_row;
    unsigned long long *spill_n;   // entries written (may exceed spill_cap: the excess is lost and the host re-runs the block)
    uint64_t spill_cap;
};

// ---- exact table of the query side --------------------------------------------------------------------------------
// Global atomics are the slow way to build a hash table (5 M postings: 0.87 ms, a third of a search).  Instead the hash
// range is cut into QT_SLICES table slices of a few thousand keys; a sorted query meets a slice in one stretch (bounds
// from part_offsets_kernel, as for the index); ONE CTA builds a slice's part of the table in SHARED memory and writes
// it out finished, so that the table needs no memset and no global atomic at all.  A slice too large for shared memory
// (a skewed hash distribution) is built in place with global atomics by the same CTA.
constexpr uint32_t QT_SLICES = 1024;
constexpr uint32_t QT_SMEM_SLOTS = 12288;   // 12288 x (8 + 4) B = 144 KB

__device__ __forceinline__ uint32_t qt_hash32(uint64_t h) { return ((uint32_t)h ^ (uint32_t)(h >> 32)) * 0x85EBCA6Bu; }

// S[t] = sum over the queries of qpo[t][q]  (slot counts follow from differences)
__global__ void __launch_bounds__(128) qt_sums_kernel(const uint32_t *__restrict__ qpo, uint64_t nq, unsigned long long *sums) {
    const uint32_t t = blockIdx.x;
    unsigned long long acc = 0;
    for (uint64_t q = threadIdx.x; q < nq; q += blockDim.x) acc += qpo[(uint64_t)t * nq + q];
    for (int d = 16; d; d >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, d);
    __shared__ unsigned long long part[4];
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) sums[t] = part[0] + part[1] + part[2] + part[3];
}
// tstart[t] = first slot of slice t: every slice gets twice its postings + 32 slots.  Also empties the slot of its own
// at tstart[QT_SLICES] that holds the list of the one hash that looks like an empty slot (~0): it must be empty before
// ANY CTA of qtable_slice_kernel runs, since the last slice's CTA pushes onto it while the others still start up.
__global__ void __launch_bounds__(1024) qt_starts_kernel(const unsigned long long *__restrict__ sums, uint32_t *tstart,
                                                         unsigned long long *tkey, int32_t *thead) {
    __shared__ uint32_t sz[QT_SLICES];
    const uint32_t t = threadIdx.x;
    sz[t] = (uint32_t)(2 * (sums[t + 1] - sums[t]) + 32);
    __syncthreads();
    if (t == 0) {
        uint32_t acc = 0;
        for (uint32_t i = 0; i < QT_SLICES; i++) { tstart[i] = acc; acc += sz[i]; }
        tstart[QT_SLICES] = acc;
        tkey[acc] = FS_EMPTY;
        thead[acc] = -1;
    }
}
template <bool SHARED>
__device__ __forceinline__ void qt_insert(unsigned long long *key, int32_t *head, uint32_t size, unsigned long long h, int32_t node,
                                          int32_t *node_next) {
    uint32_t s = __umulhi(qt_hash32(h), size);
    for (;;) {
        unsigned long long cur = key[s];
        if (cur == FS_EMPTY) cur = atomicCAS(&key[s], FS_EMPTY, h);
        if (cur == FS_EMPTY || cur == h) break;
        s = s + 1 == size ? 0 : s + 1;
    }
    node_next[node] = atomicExch(&head[s], node);
}
__global__ void __launch_bounds__(1024) qtable_slice_kernel(const uint64_t *__restrict__ qh, const uint64_t *__restrict__ qo, uint64_t nq,
                                                           const uint32_t *__restrict__ qpo, const uint32_t *__restrict__ tstart,
                                                           uint64_t top, unsigned long long *tkey, int32_t *thead, int32_t *node_next,
                                                           uint32_t *node_q) {
    extern __shared__ __align__(16) unsigned long long s_key[];
    const uint32_t t = blockIdx.x;
    const uint32_t start = tstart[t], size = tstart[t + 1] - start;
    const bool in_smem = size <= QT_SMEM_SLOTS;
    unsigned long long *key = in_smem ? s_key : tkey + start;
    int32_t *head = in_smem ? reinterpret_cast<int32_t *>(s_key + QT_SMEM_SLOTS) : thead + start;
    for (uint32_t i = threadIdx.x; i < size; i += blockDim.x) { key[i] = FS_EMPTY; head[i] = -1; }
    __syncthreads();
    // a thread takes a query at a time: the (few) postings of that query inside this slice
    for (uint64_t q = threadIdx.x; q < nq; q += blockDim.x) {
        const uint64_t b = qo[q];
        const uint32_t lo = qpo[(uint64_t)t * nq + q], hi = qpo[(uint64_t)(t + 1) * nq + q];
        for (uint32_t i = lo; i < hi; i++) {
            const unsigned long long h = qh[b + i];
            node_q[b + i] = (uint32_t)q;
            if (h > top) { node_next[b + i] = -1; continue; }   // cannot occur in the index
            if (h == FS_EMPTY) { node_next[b + i] = atomicExch(&thead[tstart[QT_SLICES]], (int32_t)(b + i)); continue; }
            if (in_smem) qt_insert<true>(key, head, size, h, (int32_t)(b + i), node_next);
            else qt_insert<false>(key, head, size, h, (int32_t)(b + i), node_next);
        }
    }
    if (in_smem) {
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < size; i += blockDim.x) { tkey[start + i] = key[i]; thead[start + i] = head[i]; }
    }
}

// Exact lookup of one hash the filter let through + count matrix update.  Called by all 32 lanes of a warp (lanes
// without an entry pass have = false); lanes that reach the same (row, query) cell add once.
__device__ __forceinline__ void stream_resolve(const StreamArgs &a, bool have, uint64_t h, uint64_t row) {
    int32_t node = -1;
    if (have && h <= a.top) {
        if (h == FS_EMPTY) {
            node = __ldg(&a.thead[__ldg(&a.tstart[QT_SLICES])]);
        } else {
            const unsigned long long tq = __umul64hi((unsigned long long)h, (unsigned long long)a.tscale);
            const uint32_t t = tq < QT_SLICES - 1 ? (uint32_t)tq : QT_SLICES - 1;
            const uint32_t start = __ldg(&a.tstart[t]), size = __ldg(&a.tstart[t + 1]) - start;
            uint32_t s = __umulhi(qt_hash32(h), size);
            for (;;) {
                const unsigned long long cur = __ldg(&a.tkey[start + s]);
                if (cur == h) { node = __ldg(&a.thead[start + s]); break; }
                if (cur == FS_EMPTY) break;
                s = s + 1 == size ? 0 : s + 1;
            }
        }
    }
    const bool found = node >= 0;
    const unsigned any = __ballot_sync(0xFFFFFFFFu, found);
    if (!any) return;   // nothing but false positives of the filter in this step
    const int lane = threadIdx.x & 31;
    const uint64_t cell = found ? row * a.ld + __ldg(&a.node_q[node]) : (~0ull - lane);
    const unsigned peers = __match_any_sync(0xFFFFFFFFu, cell);
    if (found) {
        if (lane == __ffs(peers) - 1) atomicAdd(&a.cmat[cell], (uint32_t)__popc(peers));
        for (int32_t n = __ldg(&a.node_next[node]); n >= 0; n = __ldg(&a.node_next[n]))   // hash shared by several queries
            atomicAdd(&a.cmat[row * a.ld + __ldg(&a.node_q[n])], 1u);
    }
    // rows that now hold a count: once each into the list the hit pass walks
    const unsigned same_row = __match_any_sync(0xFFFFFFFFu, found ? row : (~0ull - lane));
    if (found && lane == __ffs(same_row) - 1) {
        const uint32_t bit = 1u << (row & 31);
        const uint32_t old = atomicOr(&a.touched_bits[row >> 5], bit);
        if (!(old & bit)) a.touched_rows[atomicAdd(a.n_touched, 1ull)] = (uint32_t)row;
    }
}

// The streaming loop does not wait for the exact table: a hash the filter lets through is parked, with its row, in
// the warp's own shared-memory queue; when the queue is nearly full the warp resolves it, 32 entries per step, while
// the other warps of the CTA keep streaming.
constexpr uint32_t FS_QUEUE = 192;    // entries per warp (hash u64 + row u32): 32 x 192 x 12 B = 72 KB beside the 128 KB filter

__device__ __forceinline__ void queue_drain(const StreamArgs &a, const uint64_t *q_hash, const uint32_t *q_row, uint32_t &cnt) {
    __syncwarp();
    const int lane = threadIdx.x & 31;
    if (a.spill_hash) {   // deferred: one reservation per queue-full, coalesced copies
        unsigned long long at = 0;
        if (lane == 0 && cnt) at = atomicAdd(a.spill_n, (unsigned long long)cnt);
        at = __shfl_sync(0xFFFFFFFFu, at, 0);
        for (uint32_t i = lane; i < cnt; i += 32)
            if (at + i < a.spill_cap) { a.spill_hash[at + i] = q_hash[i]; a.spill_row[at + i] = q_row[i]; }
        __syncwarp();
        cnt = 0;
        return;
    }
    for (uint32_t i0 = 0; i0 < cnt; i0 += 32) {   // warp-uniform
        const bool have = i0 + lane < cnt;
        stream_resolve(a, have, have ? q_hash[i0 + lane] : 0, have ? q_row[i0 + lane] : 0);
    }
    __syncwarp();
    cnt = 0;
}
__device__ __forceinline__ void queue_push(const StreamArgs &a, bool hit, uint64_t h, uint32_t row, uint64_t *q_hash, uint32_t *q_row,
                                           uint32_t &cnt) {
    const unsigned m = __ballot_sync(0xFFFFFFFFu, hit);
    if (!m) return;
    if (hit) {
        const uint32_t at = cnt + __popc(m & ((1u << (threadIdx.x & 31)) - 1));
        q_hash[at] = h;
        q_row[at] = row;
    }
    cnt += __popc(m);
    if (cnt > FS_QUEUE - 32) queue_drain(a, q_hash, q_row, cnt);
}

// the loaded hashes of one row's stretch [cs, ce) against the filter; hits go to the warp's queue
__device__ __forceinline__ void stream_row(const StreamArgs &a, const uint32_t *s_filter, const uint64_t (&h)[FS_LOADS], const uint64_t *seg,
                                           uint32_t cs, uint32_t ce, uint32_t row, uint64_t *q_hash, uint32_t *q_row, uint32_t &q_cnt) {
    const int lane = threadIdx.x & 31;
    bool hit[FS_LOADS];
    bool any = false;
#pragma unroll
    for (int u = 0; u < FS_LOADS; u++) {   // branch-free: a lane beyond the stretch tests hash 0 and drops the answer
        hit[u] = filter_test(s_filter, h[u]) & (cs + lane + 32 * u < ce);
        any |= hit[u];
    }
    if (__any_sync(0xFFFFFFFFu, any)) {
#pragma unroll
        for (int u = 0; u < FS_LOADS; u++) queue_push(a, hit[u], h[u], row, q_hash, q_row, q_cnt);
    }
    for (uint32_t i = cs + 32 * FS_LOADS; i < ce; i += 32) {   // a longer stretch: the rest, one load at a time
        const bool inb = i + lane < ce;
        const uint64_t hh = inb ? __ldcs(seg + i + lane) : 0;
        queue_push(a, inb & filter_test(s_filter, hh), hh, row, q_hash, q_row, q_cnt);
    }
}

// CTA b works on slice b / ctas_per_slice for the whole launch: it loads that slice's filter once and its warps take
// groups of 32 consecutive index rows from the slice's counter until the block of rows is used up -- no CTA-wide
// barrier after the filter is in place, so a warp that is resolving its queue holds nobody up.
__global__ void __launch_bounds__(FS_THREADS, 1) stream_probe_kernel(const StreamArgs a) {
    extern __shared__ __align__(16) uint32_t s_mem[];
    uint32_t *s_filter = s_mem;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint64_t *q_hash = reinterpret_cast<uint64_t *>(s_mem + FS_FILTER_WORDS) + (size_t)warp * FS_QUEUE;
    uint32_t *q_row = reinterpret_cast<uint32_t *>(reinterpret_cast<uint64_t *>(s_mem + FS_FILTER_WORDS) + (size_t)(FS_THREADS / 32) * FS_QUEUE) +
                      (size_t)warp * FS_QUEUE;
    const uint32_t p = blockIdx.x / a.ctas_per_slice;
    if (p >= a.P) return;
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(a.filters + (size_t)p * FS_FILTER_WORDS);
        uint4 *dst = reinterpret_cast<uint4 *>(s_filter);
        for (uint32_t i = threadIdx.x; i < FS_FILTER_WORDS / 4; i += FS_THREADS) dst[i] = __ldg(src + i);
    }
    __syncthreads();
    uint32_t q_cnt = 0;
    const uint32_t *po_lo = a.part_off + (uint64_t)p * a.n_rows_total + a.b0;
    const uint32_t *po_hi = po_lo + a.n_rows_total;
    const uint32_t n_groups = (uint32_t)((a.bn + 31) / 32);
    for (;;) {
        uint32_t grp = 0;
        if (lane == 0) grp = atomicAdd(a.work_ctr + p, 1u);
        grp = __shfl_sync(0xFFFFFFFFu, grp, 0);
        if (grp >= n_groups) break;
        const uint64_t g = (uint64_t)grp * 32;
        // the bounds of 32 consecutive rows arrive with three coalesced loads
        const uint64_t r = g + lane;
        const bool valid = r < a.bn;
        const uint64_t base = valid ? __ldg(&a.io[a.b0 + r]) : 0;
        const uint32_t s = valid ? __ldg(&po_lo[r]) : 0, e = valid ? __ldg(&po_hi[r]) : 0;
        const int n_in = (int)min((uint64_t)32, a.bn - g);
        // One row per step, software-pipelined: the (up to FS_LOADS) loads of row k + 1 are issued before the hashes of
        // row k are tested.  Two steps per trip with the two register sets swapping roles, so that nothing is copied.
        uint64_t ha[FS_LOADS], hb[FS_LOADS];
        const uint64_t *seg_a = a.ih + __shfl_sync(0xFFFFFFFFu, base, 0), *seg_b = seg_a;
        uint32_t sa = __shfl_sync(0xFFFFFFFFu, s, 0), ea = __shfl_sync(0xFFFFFFFFu, e, 0), sb = 0, eb = 0;
#pragma unroll
        for (int u = 0; u < FS_LOADS; u++) ha[u] = (sa + lane + 32 * u < ea) ? __ldcs(seg_a + sa + lane + 32 * u) : 0;
        for (int k = 0; k < n_in; k += 2) {
            // ---- issue row k + 1 into set b, test row k from set a
            {
                const int kn = min(k + 1, n_in - 1);
                seg_b = a.ih + __shfl_sync(0xFFFFFFFFu, base, kn);
                sb = __shfl_sync(0xFFFFFFFFu, s, kn);
                eb = (k + 1 < n_in) ? __shfl_sync(0xFFFFFFFFu, e, kn) : sb;
#pragma unroll
                for (int u = 0; u < FS_LOADS; u++) hb[u] = (sb + lane + 32 * u < eb) ? __ldcs(seg_b + sb + lane + 32 * u) : 0;
                stream_row(a, s_filter, ha, seg_a, sa, ea, (uint32_t)(g + k), q_hash, q_row, q_cnt);
            }
            if (k + 1 >= n_in) break;
            // ---- issue row k + 2 into set a, test row k + 1 from set b
            {
                const int kn = min(k + 2, n_in - 1);
                seg_a = a.ih + __shfl_sync(0xFFFFFFFFu, base, kn);
                sa = __shfl_sync(0xFFFFFFFFu, s, kn);
                ea = (k + 2 < n_in) ? __shfl_sync(0xFFFFFFFFu, e, kn) : sa;
#pragma unroll
                for (int u = 0; u < FS_LOADS; u++) ha[u] = (sa + lane + 32 * u < ea) ? __ldcs(seg_a + sa + lane + 32 * u) : 0;
                stream_row(a, s_filter, hb, seg_b, sb, eb, (uint32_t)(g + k + 1), q_hash, q_row, q_cnt);
            }
        }
    }
    queue_drain(a, q_hash, q_row, q_cnt);
}

// Hits of one block of index rows from the counts: only rows that received a count are looked at (the list the probe
// kernel wrote), and every cell, bit and list entry that is read is cleared again, so that the count matrix, the
// touched-row bitmap and the counters are all-zero for the next block or search without a memset of the whole matrix.
//   containment (index.rs:146-160): count / |node| > threshold;  similarity of sketches without a num (lib.rs:470-508):
//   count / (|node| + |query| - count) > threshold.   found[] receives query * bn + row.
__global__ void __launch_bounds__(256) touched_hits_kernel(uint32_t *cmat, uint64_t bn, uint64_t nq, const uint64_t *__restrict__ row_offsets,
                                                           uint64_t b0, const uint64_t *__restrict__ q_offsets, double threshold,
                                                           uint32_t *touched_bits, const uint32_t *__restrict__ touched_rows,
                                                           const unsigned long long *n_touched, uint64_t *found, uint64_t cap,
                                                           unsigned long long *n_found) {
    const unsigned long long nt = *n_touched;
    for (unsigned long long t = blockIdx.x; t < nt; t += gridDim.x) {
        const uint64_t i = touched_rows[t];
        if (threadIdx.x == 0) touched_bits[i >> 5] = 0;   // (several rows of one word: all of them are in the list)
        const uint64_t la = row_offsets[b0 + i + 1] - row_offsets[b0 + i];
        for (uint64_t j = threadIdx.x; j < nq; j += blockDim.x) {
            const uint32_t cm = cmat[i * nq + j];
            if (cm == 0) continue;
            cmat[i * nq + j] = 0;
            double den = (double)la;
            if (q_offsets) den = (double)(la + (q_offsets[j + 1] - q_offsets[j]) - cm);  // >= 1 when cm >= 1
            if ((double)cm / den > threshold) {
                const unsigned long long at = atomicAdd(n_found, 1ull);
                if (at < cap) found[at] = j * bn + i;
            }
        }
    }
}
__global__ void clear_counter_kernel(unsigned long long *p) { *p = 0; }

// deferred mode: exact lookups of everything the probe kernel wrote out, one entry per thread
__global__ void __launch_bounds__(256) resolve_spill_kernel(const StreamArgs a) {
    const unsigned long long n = min(*a.spill_n, (unsigned long long)a.spill_cap);
    const unsigned long long n_round = (n + 31) / 32 * 32;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_round; i += (unsigned long long)gridDim.x * blockDim.x) {
        const bool have = i < n;   // whole warps stay together: stream_resolve votes
        stream_resolve(a, have, have ? a.spill_hash[i] : 0, have ? a.spill_row[i] : 0);
    }
}

}  // namespace

// ---- host side ---------------------------------------------------------------------------------------------
uint32_t find_stream_partitions(uint64_t n_rows, uint64_t n_hashes, int sm_count) {
    // One CTA per SM and a whole number of CTAs per slice: P = sm_count / c.  Stretches of about 100 hashes (three to
    // four coalesced loads per row and slice: the per-row cost of the loop is spread over more hashes and DRAM sees
    // longer pieces), at most sm_count / 2 slices.
    const uint64_t avg = n_rows ? n_hashes / n_rows : 0;
    const uint32_t want = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)sm_count / 2, avg / 100));
    const uint32_t c = ((uint32_t)sm_count + want - 1) / want;   // CTAs per slice
    return std::max<uint32_t>(1, (uint32_t)sm_count / c);
}

void launch_rows_max(const uint64_t *h, const uint64_t *off, uint64_t n_rows, unsigned long long *out, cudaStream_t st) {
    if (!n_rows) return;
    rows_max_kernel<<<(unsigned)std::min<uint64_t>((n_rows + 255) / 256, 148 * 8), 256, 0, st>>>(h, off, n_rows, out);
    SM_LAUNCHED();
}
uint64_t find_stream_scale(uint64_t top, uint32_t P) {
    const unsigned __int128 q = (((unsigned __int128)P) << 64) / ((unsigned __int128)top + 1);
    return q > (unsigned __int128)~0ull ? ~0ull : (uint64_t)q;
}
void launch_part_offsets(const uint64_t *h, const uint64_t *off, uint64_t n_rows, uint64_t scale, uint32_t P, uint32_t *part_off,
                         cudaStream_t st) {
    if (!n_rows) return;
    part_offsets_kernel<<<(unsigned)std::min<uint64_t>((n_rows * 32 + 255) / 256, 148 * 16), 256, 0, st>>>(h, off, n_rows, scale, P, part_off);
    SM_LAUNCHED();
}
size_t find_stream_filter_bytes(uint32_t P) { return (size_t)P * FS_FILTER_WORDS * 4; }
void launch_filters_build(const uint64_t *qh, uint64_t n, uint64_t scale, uint64_t top, uint32_t P, uint32_t *filters, cudaStream_t st) {
    if (!n) return;
    filters_build_kernel<<<(unsigned)std::min<uint64_t>((n + 255) / 256, 148 * 16), 256, 0, st>>>(qh, n, scale, top, P, filters);
    SM_LAUNCHED();
}
// Exact table of the query side.  qpo: (QT_SLICES + 1) x nq u32 scratch; sums: QT_SLICES + 1 u64 scratch; tstart: QT_SLICES + 1 u32;
// tkey / thead: find_stream_table_slots(n_postings) entries; node_next / node_q: n_postings entries.
size_t find_stream_table_slots(uint64_t n_postings) { return (size_t)(2 * n_postings + 32ull * QT_SLICES + 2); }
uint32_t find_stream_table_slices() { return QT_SLICES; }
void launch_qtable_build(const uint64_t *qh, const uint64_t *qo, uint64_t nq, uint64_t top, uint32_t *qpo, unsigned long long *sums,
                         uint32_t *tstart, unsigned long long *tkey, int32_t *thead, int32_t *node_next, uint32_t *node_q,
                         uint64_t *tscale_out, cudaStream_t st) {
    const uint64_t tscale = find_stream_scale(top, QT_SLICES);
    *tscale_out = tscale;
    ProfScope prof(PROF_SORT, st);
    launch_part_offsets(qh, qo, nq, tscale, QT_SLICES, qpo, st);
    qt_sums_kernel<<<QT_SLICES + 1, 128, 0, st>>>(qpo, nq, sums);
    SM_LAUNCHED();
    qt_starts_kernel<<<1, QT_SLICES, 0, st>>>(sums, tstart, tkey, thead);
    SM_LAUNCHED();
    static bool attr_set = false;
    const size_t smem = (size_t)QT_SMEM_SLOTS * 12;
    if (!attr_set) {
        SM_CUDA(cudaFuncSetAttribute(qtable_slice_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    qtable_slice_kernel<<<QT_SLICES, 1024, smem, st>>>(qh, qo, nq, qpo, tstart, top, tkey, thead, node_next, node_q);
    SM_LAUNCHED();
}
void launch_stream_probe(const uint64_t *ih, const uint64_t *io, uint64_t b0, uint64_t bn, const uint32_t *part_off,
                         uint64_t n_rows_total, uint32_t P, const uint32_t *filters, const unsigned long long *tkey,
                         const int32_t *thead, const int32_t *node_next, const uint32_t *node_q, const uint32_t *tstart, uint64_t tscale,
                         uint64_t top, uint32_t *cmat, uint64_t ld, uint32_t *touched_bits, uint32_t *touched_rows,
                         unsigned long long *n_touched, uint32_t *work_ctr, uint64_t *spill_hash, uint32_t *spill_row,
                         unsigned long long *spill_n, uint64_t spill_cap, int phase, int sm_count, cudaStream_t st) {
    if (!bn) return;
    static bool attr_set = false;
    const size_t smem = (size_t)FS_FILTER_WORDS * 4 + (size_t)(FS_THREADS / 32) * FS_QUEUE * 12;
    if (!attr_set) {
        SM_CUDA(cudaFuncSetAttribute(stream_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    StreamArgs a;
    a.ih = ih; a.io = io; a.b0 = b0; a.bn = bn; a.part_off = part_off; a.n_rows_total = n_rows_total; a.P = P;
    a.filters = filters; a.tkey = tkey; a.thead = thead; a.node_next = node_next; a.node_q = node_q; a.tstart = tstart;
    a.tscale = tscale; a.top = top;
    a.cmat = cmat; a.ld = ld; a.touched_bits = touched_bits; a.touched_rows = touched_rows; a.n_touched = n_touched;
    a.work_ctr = work_ctr;
    a.ctas_per_slice = std::max<uint32_t>(1, (uint32_t)sm_count / P);
    a.spill_hash = spill_hash; a.spill_row = spill_row; a.spill_n = spill_n; a.spill_cap = spill_cap;
    if (phase == 0) {          // stream the index (deferred when spill_hash is given, else resolving as it goes)
        ProfScope prof(PROF_FIND, st);
        stream_probe_kernel<<<P * a.ctas_per_slice, FS_THREADS, smem, st>>>(a);
        SM_LAUNCHED();
    } else {                   // deferred mode, second half: look the written-out hashes up
        ProfScope prof(PROF_PROBE, st);
        resolve_spill_kernel<<<sm_count * 8, 256, 0, st>>>(a);
        SM_LAUNCHED();
    }
}
void launch_touched_hits(uint32_t *cmat, uint64_t bn, uint64_t nq, const uint64_t *row_offsets, uint64_t b0, const uint64_t *q_offsets,
                         double threshold, uint32_t *touched_bits, const uint32_t *touched_rows, unsigned long long *n_touched,
                         uint64_t *found, uint64_t cap, unsigned long long *n_found, int sm_count, cudaStream_t st) {
    touched_hits_kernel<<<sm_count * 8, 256, 0, st>>>(cmat, bn, nq, row_offsets, b0, q_offsets, threshold, touched_bits, touched_rows,
                                                       n_touched, found, cap, n_found);
    SM_LAUNCHED();
    clear_counter_kernel<<<1, 1, 0, st>>>(n_touched);
    SM_LAUNCHED();
}

}  // namespace smb200
