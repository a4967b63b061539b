// nodegraph.cu -- see nodegraph.hpp.  Kernels first, then the host class, then SBT::find.
#include "nodegraph.hpp"

#include <algorithm>
#include <cstring>
#include <memory>
#include <unordered_map>

#include "kernels.cuh"

namespace smb200 {

namespace {

constexpr int NG_THREADS = 256;
constexpr uint64_t NG_TABLE_SHIFT = 56;  // count_many: table index kept in the top byte of the pair's value

__device__ __forceinline__ bool ng_test(const uint32_t *words, const NgTable &t, uint64_t hash) {
    const uint64_t bin = hash % t.len;
    return (words[t.word_off + (bin >> 5)] >> (bin & 31)) & 1u;
}

// one (hash, table) pair per thread, hash-major: key = global bin id of a bin that is still clear
// (total_bits for a bin already set), value = hash index | table << 56
__global__ void ng_pairs_kernel(const uint64_t *hashes, uint64_t n, const uint32_t *words, const NgTable *tabs, uint32_t nt,
                                uint64_t total_bits, uint64_t *keys, uint64_t *vals) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n * nt) return;
    const uint64_t i = j / nt;
    const uint32_t t = (uint32_t)(j % nt);
    const NgTable tb = tabs[t];
    const uint64_t bin = hashes[i] % tb.len;
    const bool set = (words[tb.word_off + (bin >> 5)] >> (bin & 31)) & 1u;
    keys[j] = set ? total_bits : tb.bit_off + bin;
    vals[j] = i | ((uint64_t)t << NG_TABLE_SHIFT);
}
// after the stable sort: the head of every run of equal keys is the FIRST hash of the batch that maps to
// that clear bin -- the one hash for which Nodegraph::count finds `put` returning false there
__global__ void ng_apply_kernel(const uint64_t *keys, const uint64_t *vals, uint64_t m, uint64_t total_bits, uint32_t *words,
                                const NgTable *tabs, uint8_t *is_new, unsigned long long *occupied) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool head = false;
    if (j < m) {
        const uint64_t k = keys[j];
        head = k < total_bits && (j == 0 || keys[j - 1] != k);
        if (head) {
            const uint64_t v = vals[j];
            const NgTable tb = tabs[v >> NG_TABLE_SHIFT];
            const uint64_t bin = k - tb.bit_off;
            atomicOr(&words[tb.word_off + (bin >> 5)], 1u << (bin & 31));
            is_new[v & ((1ull << NG_TABLE_SHIFT) - 1)] = 1;
        }
    }
    const unsigned bal = __ballot_sync(0xFFFFFFFFu, head);
    if ((threadIdx.x & 31) == 0 && bal) atomicAdd(occupied, (unsigned long long)__popc(bal));
}
__global__ void ng_sum_bytes_kernel(const uint8_t *flags, uint64_t n, unsigned long long *out) {
    uint64_t acc = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) acc += flags[i];
    for (int o = 16; o; o >>= 1) acc += __shfl_down_sync(0xFFFFFFFFu, acc, o);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, (unsigned long long)acc);
}
__global__ void ng_get_kernel(const uint64_t *hashes, uint64_t n, const uint32_t *words, const NgTable *tabs, uint32_t nt,
                              uint8_t *present, unsigned long long *matches) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool hit = false;
    if (i < n) {
        const uint64_t h = hashes[i];
        hit = true;
        for (uint32_t t = 0; t < nt && hit; t++) hit = ng_test(words, tabs[t], h);
        if (present) present[i] = hit ? 1 : 0;
    }
    const unsigned bal = __ballot_sync(0xFFFFFFFFu, hit);
    if ((threadIdx.x & 31) == 0 && bal) atomicAdd(matches, (unsigned long long)__popc(bal));
}
// word-wise over the zipped tables: mode 0 = a |= b (only the bits of b below a's table length), mode 1 = popcounts
// of a & b and a | b, mode 2 = *out2 = min(*out2, first table in which b has a set bit at or beyond a's length)
__global__ void ng_words_kernel(uint32_t *a, const NgTable *ta, const uint32_t *b, const NgTable *tb, uint32_t nt, int mode,
                                unsigned long long *out2) {
    unsigned long long n_and = 0, n_or = 0;
    for (uint32_t t = 0; t < nt; t++) {
        const uint64_t wa = (ta[t].len + 31) / 32, wb = (tb[t].len + 31) / 32, lo = wa < wb ? wa : wb, hi = wa < wb ? wb : wa;
        const uint64_t edge = ta[t].len / 32;                            // the word a's table ends in
        const uint32_t below = (1u << (ta[t].len % 32)) - 1u;            // its bits that are inside a's table
        for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < hi; w += (uint64_t)gridDim.x * blockDim.x) {
            const uint32_t x = w < wa ? a[ta[t].word_off + w] : 0u, y = w < wb ? b[tb[t].word_off + w] : 0u;
            if (mode == 0) {
                const uint32_t yi = w == edge ? (y & below) : y;
                if (w < lo && yi) a[ta[t].word_off + w] = x | yi;
            } else if (mode == 2) {
                const uint32_t beyond = w < edge ? 0u : (w == edge ? (y & ~below) : y);
                if (beyond) atomicMin(out2, (unsigned long long)t);
            } else {
                n_and += __popc(x & y);
                n_or += __popc(x | y);
            }
        }
    }
    if (mode == 1) {
        for (int o = 16; o; o >>= 1) {
            n_and += __shfl_down_sync(0xFFFFFFFFu, n_and, o);
            n_or += __shfl_down_sync(0xFFFFFFFFu, n_or, o);
        }
        if ((threadIdx.x & 31) == 0) {
            if (n_and) atomicAdd(out2, n_and);
            if (n_or) atomicAdd(out2 + 1, n_or);
        }
    }
}

// SBT search: one CTA per (query, node): matches[node * nq + query] = sum over the query's hashes of node.get(h)
struct NgView {
    const uint32_t *words;
    const NgTable *tabs;
    uint32_t nt;
};
__global__ void __launch_bounds__(128) sbt_matches_kernel(const uint64_t *q_hashes, const uint64_t *q_offsets, uint64_t q0, uint64_t nq,
                                                          const NgView *nodes, uint32_t *matches) {
    const uint64_t q = blockIdx.x, node = blockIdx.y;
    const NgView nv = nodes[node];
    const uint64_t lo = q_offsets[q0 + q], hi = q_offsets[q0 + q + 1];
    uint32_t acc = 0;
    for (uint64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        const uint64_t h = q_hashes[i];
        bool hit = true;
        for (uint32_t t = 0; t < nv.nt && hit; t++) hit = ng_test(nv.words, nv.tabs[t], h);
        acc += hit;
    }
    __shared__ uint32_t s_acc[4];
    for (int o = 16; o; o >>= 1) acc += __shfl_down_sync(0xFFFFFFFFu, acc, o);
    if ((threadIdx.x & 31) == 0) s_acc[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) matches[node * nq + q] = s_acc[0] + s_acc[1] + s_acc[2] + s_acc[3];
}

int bit_length_u64(uint64_t x) {
    int b = 0;
    while (x) { b++; x >>= 1; }
    return b;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// host class
// ---------------------------------------------------------------------------------------------
Nodegraph::Nodegraph(const uint64_t *tablesizes, size_t n_tables, uint64_t ksize_) : ksize(ksize_) {
    if (n_tables > 255) throw_internal("a Nodegraph holds at most 255 tables (n_tables is one byte in the file format)");
    for (size_t t = 0; t < n_tables; t++) {
        if (tablesizes[t] == 0) throw SourmashError(ERR_PANIC, "sourmash panicked: attempt to calculate the remainder with a divisor of zero");
        NgTable tb;
        tb.len = tablesizes[t];
        tb.word_off = total_words;
        tb.bit_off = total_bits;
        total_words += (tb.len + 31) / 32;
        total_bits += tb.len;
        tables.push_back(tb);
    }
    Context &ctx = Context::get();
    d_words.reserve((total_words + 1) * 4);
    d_tables.reserve((n_tables + 1) * sizeof(NgTable));
    SM_CUDA(cudaMemsetAsync(d_words.p, 0, (total_words + 1) * 4, ctx.stream));
    if (n_tables) SM_CUDA(cudaMemcpyAsync(d_tables.p, tables.data(), n_tables * sizeof(NgTable), cudaMemcpyHostToDevice, ctx.stream));
    ctx.sync();
}

// Nodegraph::from_reader, nodegraph.rs:135-181
Nodegraph *Nodegraph::from_buffer(const uint8_t *d, size_t n) {
    auto fail = [](const char *what) -> void { throw SourmashError(ERR_PANIC, std::string("sourmash panicked: Nodegraph::from_reader: ") + what); };
    if (n < 19) fail("failed to fill whole buffer");
    if (!(d[0] == 0x4f && d[1] == 0x58 && d[2] == 0x4c && d[3] == 0x49)) fail("assertion failed: signature == 0x4f584c49");
    if (d[4] != 0x04) fail("assertion failed: version == 0x04");
    if (d[5] != 0x02) fail("assertion failed: ht_type == 0x02");
    auto le = [&](size_t p, int bytes) { uint64_t v = 0; for (int b = 0; b < bytes; b++) v |= (uint64_t)d[p + b] << (8 * b); return v; };
    const uint64_t ksize = le(6, 4);
    const size_t n_tables = d[10];
    const uint64_t occupied = le(11, 8);
    std::vector<uint64_t> sizes(n_tables);
    size_t q = 19;
    for (size_t t = 0; t < n_tables; t++) {
        if (q + 8 > n) fail("failed to fill whole buffer");
        sizes[t] = le(q, 8);
        if (sizes[t] / 8 + 1 > n - q - 8) fail("failed to fill whole buffer");
        q += 8 + (size_t)(sizes[t] / 8 + 1);
    }
    std::unique_ptr<Nodegraph> ng(new Nodegraph(sizes.data(), n_tables, ksize));
    std::vector<uint32_t> words(ng->total_words + 1, 0);
    size_t p = 19;
    for (size_t t = 0; t < n_tables; t++) {
        const uint64_t tablesize = sizes[t], byte_size = tablesize / 8 + 1;
        p += 8;
        uint32_t *w = words.data() + ng->tables[t].word_off;
        for (uint64_t pos = 0; pos < byte_size; pos++) {
            const uint8_t byte = d[p++];
            if (!byte) continue;
            if (pos * 8 + 7 >= tablesize) {  // FixedBitSet::insert panics beyond the capacity
                for (unsigned i = 0; i < 8; i++)
                    if ((byte >> i) & 1 && pos * 8 + i >= tablesize) fail("index out of bounds");
            }
            w[pos >> 2] |= (uint32_t)byte << (8 * (pos & 3));
        }
    }
    Context &ctx = Context::get();
    if (ng->total_words) SM_CUDA(cudaMemcpyAsync(ng->d_words.p, words.data(), ng->total_words * 4, cudaMemcpyHostToDevice, ctx.stream));
    ctx.sync();
    ng->occupied_bins = occupied;
    ng->unique_kmers = 0;  // "a khmer issue, it doesn't save unique_kmers" (nodegraph.rs:179)
    return ng.release();
}

// Nodegraph::save_to_writer, nodegraph.rs:99-133
size_t Nodegraph::save(uint8_t *out, size_t cap) {
    std::vector<uint32_t> words(total_words + 1, 0);
    Context &ctx = Context::get();
    if (total_words) SM_CUDA(cudaMemcpyAsync(words.data(), d_words.p, total_words * 4, cudaMemcpyDeviceToHost, ctx.stream));
    ctx.sync();
    size_t n = 0;
    auto put8 = [&](uint64_t v) { if (n < cap) out[n] = (uint8_t)v; n++; };
    auto putle = [&](uint64_t v, int bytes) { for (int b = 0; b < bytes; b++) put8(v >> (8 * b)); };
    put8('O'); put8('X'); put8('L'); put8('I');
    put8(4);  // version
    put8(2);  // ht_type
    putle(ksize, 4);
    put8(tables.size());
    putle(occupied_bins, 8);
    for (const NgTable &tb : tables) {
        const uint64_t blocks = (tb.len + 31) / 32;
        putle(tb.len, 8);
        for (uint64_t i = 0; i < blocks; i++) {
            const uint32_t chunk = words[tb.word_off + i];
            if ((i + 1) * 32 <= tb.len) {
                putle(chunk, 4);
            } else {
                const uint64_t rem = tb.len - i * 32;
                const uint64_t remainder = (rem % 8) ? rem / 8 + 1 : rem / 8;
                if (remainder == 0) put8(0);
                else for (uint64_t pos = 0; pos < remainder; pos++) put8((chunk >> (pos * 8)) & 0xff);
            }
        }
    }
    return n;
}

uint64_t Nodegraph::count_many(const uint64_t *hashes, uint64_t n, uint8_t *is_new, bool on_device) {
    if (n == 0) return 0;
    if (tables.empty()) {  // count() sets no bin, so no hash is new
        if (is_new && on_device) {
            Context &ctx = Context::get();
            SM_CUDA(cudaMemsetAsync(is_new, 0, n, ctx.stream));
            ctx.sync();
        } else if (is_new) {
            std::memset(is_new, 0, n);
        }
        return 0;
    }
    if (n >> NG_TABLE_SHIFT) throw_internal("too many hashes in one count_many call");
    Context &ctx = Context::get();
    cudaStream_t st = ctx.stream;
    const uint32_t nt = (uint32_t)tables.size();
    const uint64_t m = n * nt;
    const uint64_t *d_h = hashes;
    if (!on_device) {
        ctx.misc[0].reserve(n * 8);
        SM_CUDA(cudaMemcpyAsync(ctx.misc[0].p, hashes, n * 8, cudaMemcpyHostToDevice, st));
        d_h = ctx.misc[0].as<uint64_t>();
    }
    ctx.join[0].reserve((m + 1) * 8);
    ctx.join[1].reserve((m + 1) * 8);
    ctx.sort_tmp_k.reserve((m + 1) * 8);
    ctx.sort_tmp_v.reserve((m + 1) * 8);
    ctx.scan_tmp.reserve(radix_sort_scan_bytes(m) + 256);
    ctx.misc[1].reserve(n + 16);
    uint64_t *keys = ctx.join[0].as<uint64_t>(), *vals = ctx.join[1].as<uint64_t>();
    uint8_t *d_new = ctx.misc[1].as<uint8_t>();
    SM_CUDA(cudaMemsetAsync(d_new, 0, n, st));
    SM_CUDA(cudaMemsetAsync(ctx.dsc(SC_PAIR0), 0, 16, st));
    ng_pairs_kernel<<<(unsigned)((m + NG_THREADS - 1) / NG_THREADS), NG_THREADS, 0, st>>>(d_h, n, words(), dev_tables(), nt, total_bits,
                                                                                          keys, vals);
    SM_LAUNCHED();
    // stable LSD sort: equal bins keep batch order, so each run starts with its first hash
    radix_sort_pairs(keys, vals, m, ctx.sort_tmp_k.as<uint64_t>(), ctx.sort_tmp_v.as<uint64_t>(), bit_length_u64(total_bits),
                     ctx.scan_tmp.p, ctx.scan_tmp.cap, st);
    ng_apply_kernel<<<(unsigned)((m + NG_THREADS - 1) / NG_THREADS), NG_THREADS, 0, st>>>(keys, vals, m, total_bits, d_words.as<uint32_t>(),
                                                                                          dev_tables(), d_new, ctx.dsc(SC_PAIR0));
    SM_LAUNCHED();
    ng_sum_bytes_kernel<<<(unsigned)std::min<uint64_t>(1024, (n + NG_THREADS - 1) / NG_THREADS), NG_THREADS, 0, st>>>(d_new, n,
                                                                                                                   ctx.dsc(SC_PAIR1));
    SM_LAUNCHED();
    if (is_new) SM_CUDA(cudaMemcpyAsync(is_new, d_new, n, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
    ctx.read_scalars();
    occupied_bins += ctx.h_scalars[SC_PAIR0];
    unique_kmers += ctx.h_scalars[SC_PAIR1];
    return ctx.h_scalars[SC_PAIR1];
}

uint64_t Nodegraph::get_many(const uint64_t *hashes, uint64_t n, uint8_t *present, bool on_device) {
    if (n == 0) return 0;
    Context &ctx = Context::get();
    cudaStream_t st = ctx.stream;
    const uint64_t *d_h = hashes;
    uint8_t *d_p = present;
    if (!on_device) {
        ctx.misc[0].reserve(n * 8);
        SM_CUDA(cudaMemcpyAsync(ctx.misc[0].p, hashes, n * 8, cudaMemcpyHostToDevice, st));
        d_h = ctx.misc[0].as<uint64_t>();
        if (present) {
            ctx.misc[1].reserve(n + 16);
            d_p = ctx.misc[1].as<uint8_t>();
        }
    }
    SM_CUDA(cudaMemsetAsync(ctx.dsc(SC_PAIR0), 0, 8, st));
    ng_get_kernel<<<(unsigned)((n + NG_THREADS - 1) / NG_THREADS), NG_THREADS, 0, st>>>(d_h, n, words(), dev_tables(), (uint32_t)tables.size(),
                                                                                        d_p, ctx.dsc(SC_PAIR0));
    SM_LAUNCHED();
    if (!on_device && present) SM_CUDA(cudaMemcpyAsync(present, d_p, n, cudaMemcpyDeviceToHost, st));
    ctx.read_scalars();
    return ctx.h_scalars[SC_PAIR0];
}

// Nodegraph::update, nodegraph.rs:63-91: tables are zipped; every set bit of `other` is `put` into self.
// (occupied_bins is deliberately left alone there.)  The reference panics at the first set bit of `other` that lies
// beyond self's table (FixedBitSet::put) -- tables in order, bits ascending -- so a LONGER table on the other side is
// fine as long as its tail is clear, and on a panic the earlier tables and the in-range bits of the failing one have
// already been put.
void Nodegraph::update(Nodegraph &other) {
    const uint32_t nt = (uint32_t)std::min(tables.size(), other.tables.size());
    if (!nt) return;
    Context &ctx = Context::get();
    bool longer = false;
    for (uint32_t t = 0; t < nt; t++) longer |= other.tables[t].len > tables[t].len;
    uint32_t nt_ok = nt;
    const unsigned grid = (unsigned)std::min<uint64_t>(2048, (std::max(total_words, other.total_words) + NG_THREADS - 1) / NG_THREADS + 1);
    if (longer) {
        ctx.set_scalar(SC_PAIR0, nt);
        ng_words_kernel<<<grid, NG_THREADS, 0, ctx.stream>>>(d_words.as<uint32_t>(), dev_tables(), other.words(), other.dev_tables(), nt,
                                                               2, ctx.dsc(SC_PAIR0));
        SM_LAUNCHED();
        ctx.read_scalars();
        nt_ok = (uint32_t)ctx.h_scalars[SC_PAIR0];
    }
    ng_words_kernel<<<grid, NG_THREADS, 0, ctx.stream>>>(d_words.as<uint32_t>(), dev_tables(), other.words(), other.dev_tables(),
                                                           std::min(nt, nt_ok + 1), 0, nullptr);
    SM_LAUNCHED();
    ctx.sync();
    if (nt_ok < nt)
        throw SourmashError(ERR_PANIC, "sourmash panicked: Nodegraph::update: put at index beyond the table (tables of different size)");
}

void Nodegraph::and_or_counts(Nodegraph &other, uint64_t *n_and, uint64_t *n_or) {
    const uint32_t nt = (uint32_t)std::min(tables.size(), other.tables.size());
    Context &ctx = Context::get();
    SM_CUDA(cudaMemsetAsync(ctx.dsc(SC_PAIR0), 0, 16, ctx.stream));
    if (nt) {
        const uint64_t w = std::max(total_words, other.total_words);
        ng_words_kernel<<<(unsigned)std::min<uint64_t>(2048, (w + NG_THREADS - 1) / NG_THREADS + 1), NG_THREADS, 0, ctx.stream>>>(
            d_words.as<uint32_t>(), dev_tables(), other.words(), other.dev_tables(), nt, 1, ctx.dsc(SC_PAIR0));
        SM_LAUNCHED();
    }
    ctx.read_scalars();
    *n_and = ctx.h_scalars[SC_PAIR0];
    *n_or = ctx.h_scalars[SC_PAIR1];
}
// nodegraph.rs:199-213
double Nodegraph::similarity(Nodegraph &other) {
    uint64_t x, u;
    and_or_counts(other, &x, &u);
    return (double)x / (double)u;
}
// nodegraph.rs:215-224: the denominator is the summed LENGTH of self's tables
double Nodegraph::containment(Nodegraph &other) {
    uint64_t x, u;
    and_or_counts(other, &x, &u);
    return (double)x / (double)total_bits;
}

// ---------------------------------------------------------------------------------------------
// SBT::find (sbt.rs:147-175) for a whole batch of queries.
// The reference walks the tree once per query and probes one bloom filter at a time.  Here every
// (internal node, query) pair is probed by one kernel launch and every (leaf, query) pair by the
// collection compare kernels; the depth-first walk then only reads those two tables, so its order --
// children pushed 0..d-1 and popped from the back -- and therefore the order of the hits is the
// reference's.
// ---------------------------------------------------------------------------------------------
uint64_t sbt_find(uint32_t d, const uint64_t *node_pos, Nodegraph *const *nodes, const uint64_t *min_n_below, uint64_t n_nodes,
                  const uint64_t *leaf_pos, SketchCollection &leaves, SketchCollection &queries, int mode, double threshold,
                  uint64_t *hit_offsets, uint64_t *hits, uint64_t hits_cap) {
    leaves.check_compatible(queries);
    leaves.finalize();
    queries.finalize();
    const uint64_t nq = queries.n_rows, nl = leaves.n_rows;
    Context &ctx = Context::get();
    cudaStream_t st = ctx.stream;
    std::unordered_map<uint64_t, uint64_t> node_at, leaf_at;
    for (uint64_t i = 0; i < n_nodes; i++) node_at.emplace(node_pos[i], i);  // first entry wins, as a HashMap built from unique keys
    for (uint64_t i = 0; i < nl; i++) leaf_at.emplace(leaf_pos[i], i);

    std::vector<NgView> views(n_nodes);
    for (uint64_t i = 0; i < n_nodes; i++) {
        views[i].words = nodes[i]->words();
        views[i].tabs = nodes[i]->dev_tables();
        views[i].nt = (uint32_t)nodes[i]->tables.size();
    }
    DevBuf d_views;
    if (n_nodes) {
        d_views.reserve(n_nodes * sizeof(NgView));
        SM_CUDA(cudaMemcpyAsync(d_views.p, views.data(), n_nodes * sizeof(NgView), cudaMemcpyHostToDevice, st));
    }
    // query blocks small enough for the two tables to stay modest
    const uint64_t per_query = std::max<uint64_t>(1, n_nodes + nl);
    const uint64_t block_q = std::max<uint64_t>(1, std::min<uint64_t>(nq ? nq : 1, std::min<uint64_t>(65535, (1ull << 26) / per_query)));
    std::vector<uint32_t> h_matches;
    std::vector<double> h_ratio;
    std::vector<uint64_t> stack;
    uint64_t total = 0;
    for (uint64_t q0 = 0; q0 < nq; q0 += block_q) {
        const uint64_t bq = std::min(block_q, nq - q0);
        h_matches.assign(n_nodes * bq, 0);
        h_ratio.assign(nl * bq, 0.0);
        if (n_nodes) {
            ctx.misc[0].reserve(n_nodes * bq * 4);
            dim3 grid((unsigned)bq, (unsigned)n_nodes);
            if (n_nodes > 65535) throw_internal("more than 65535 internal nodes per sbt_find call");
            sbt_matches_kernel<<<grid, 128, 0, st>>>(queries.d_hashes.as<uint64_t>(), queries.d_offsets.as<uint64_t>(), q0, bq,
                                                     d_views.as<NgView>(), ctx.misc[0].as<uint32_t>());
            SM_LAUNCHED();
            SM_CUDA(cudaMemcpyAsync(h_matches.data(), ctx.misc[0].p, n_nodes * bq * 4, cudaMemcpyDeviceToHost, st));
            ctx.sync();
        }
        if (nl) compare_matrix(leaves, 0, nl, queries, q0, bq, mode, nullptr, nullptr, h_ratio.data(), bq, false);
        for (uint64_t q = 0; q < bq; q++) {
            if (hit_offsets) hit_offsets[q0 + q] = total;
            const uint64_t q_size = queries.h_offsets[q0 + q + 1] - queries.h_offsets[q0 + q];
            stack.assign(1, 0);
            while (!stack.empty()) {
                const uint64_t pos = stack.back();
                stack.pop_back();
                auto ni = node_at.find(pos);
                if (ni != node_at.end()) {
                    double v = 0.0;  // sbt.rs:241-243 / 262-264: an empty query sketch compares as 0.0
                    if (q_size) {
                        const double matches = (double)h_matches[ni->second * bq + q];
                        v = mode ? matches / (double)q_size : matches / (double)min_n_below[ni->second];
                    }
                    if (v > threshold)
                        for (uint32_t c = 0; c < d; c++) stack.push_back((uint64_t)d * pos + c + 1);
                    continue;
                }
                auto li = leaf_at.find(pos);
                if (li != leaf_at.end() && h_ratio[li->second * bq + q] > threshold) {
                    if (hits && total < hits_cap) hits[total] = pos;
                    total++;
                }
            }
        }
    }
    if (hit_offsets) hit_offsets[nq] = total;
    return total;
}

}  // namespace smb200
