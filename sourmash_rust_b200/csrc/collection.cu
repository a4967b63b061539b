// collection.cu -- host side of the collection-level operations: CSR packing, the blocked
// all-vs-all matrix and LinearIndex::find over a whole query batch.
#include "collection.hpp"

#include <algorithm>
#include <cstdlib>
#include <memory>

#include "kernels.cuh"

namespace smb200 {

void SketchCollection::push(KmerMinHash &mh) {
    if (!have_params) {
        ksize = mh.ksize; is_protein = mh.is_protein; seed = mh.seed; max_hash = mh.max_hash;
        have_params = true;
    } else {
        if (ksize != mh.ksize) throw SourmashError(ERR_MISMATCH_KSIZES, "different ksizes cannot be compared");
        if (is_protein != mh.is_protein) throw SourmashError(ERR_MISMATCH_DNAPROT, "DNA/prot minhashes cannot be compared");
        if (max_hash != mh.max_hash) throw SourmashError(ERR_MISMATCH_MAXHASH, "mismatch in max_hash; comparison fail");
        if (seed != mh.seed) throw SourmashError(ERR_MISMATCH_SEED, "mismatch in seed; comparison fail");
    }
    const std::vector<uint64_t> &m = mh.mins();
    for (size_t i = 1; i < m.size(); i++)
        if (!(m[i - 1] < m[i])) throw_internal("collection rows must hold strictly ascending mins");
    h_hashes.insert(h_hashes.end(), m.begin(), m.end());
    h_offsets.push_back(h_hashes.size());
    h_nums.push_back(mh.num);
    dirty = true;
    probe_checked = probe_dense_preferred = false;
    parts_valid = false;
}

// slice bounds of every row (find_stream.cu), once per collection content
void SketchCollection::ensure_partitions() {
    finalize();
    if (parts_valid) return;
    Context &ctx = Context::get();
    n_parts = find_stream_partitions(n_rows, n_hashes, ctx.sm_count);
    SM_CUDA(cudaMemsetAsync(ctx.dsc(SC_TMAX), 0, 8, ctx.stream));
    launch_rows_max(d_hashes.as<uint64_t>(), d_offsets.as<uint64_t>(), n_rows, ctx.dsc(SC_TMAX), ctx.stream);
    ctx.read_scalars();
    part_top = ctx.h_scalars[SC_TMAX];
    part_scale = find_stream_scale(part_top, n_parts);
    d_part_off.reserve((size_t)(n_parts + 1) * std::max<uint64_t>(1, n_rows) * 4);
    launch_part_offsets(d_hashes.as<uint64_t>(), d_offsets.as<uint64_t>(), n_rows, part_scale, n_parts, d_part_off.as<uint32_t>(),
                        ctx.stream);
    ctx.sync();
    parts_valid = true;
}

void SketchCollection::finalize() {
    Context &ctx = Context::get();
    ctx.adopt(owner);  // last used from another thread: wait for what that thread queued
    if (!dirty) return;
    n_rows = h_nums.size();
    n_hashes = h_hashes.size();
    d_hashes.reserve((n_hashes + 4) * 8);  // slack: the pair walk reads up to two elements past a row
    d_offsets.reserve((n_rows + 1) * 8);
    d_nums.reserve((n_rows + 1) * 4);
    if (n_hashes) SM_CUDA(cudaMemcpyAsync(d_hashes.p, h_hashes.data(), n_hashes * 8, cudaMemcpyHostToDevice, ctx.stream));
    SM_CUDA(cudaMemcpyAsync(d_offsets.p, h_offsets.data(), (n_rows + 1) * 8, cudaMemcpyHostToDevice, ctx.stream));
    if (n_rows) SM_CUDA(cudaMemcpyAsync(d_nums.p, h_nums.data(), n_rows * 4, cudaMemcpyHostToDevice, ctx.stream));
    ctx.sync();
    max_len = 0;
    for (uint64_t i = 0; i < n_rows; i++) max_len = std::max<uint32_t>(max_len, (uint32_t)(h_offsets[i + 1] - h_offsets[i]));
    dirty = false;
}

SketchCollection *SketchCollection::from_csr(const uint64_t *hashes, const uint64_t *offsets, uint64_t n_rows_, uint32_t num,
                                             uint32_t ksize_, uint64_t seed_, uint64_t max_hash_, bool on_device) {
    Context &ctx = Context::get();
    std::unique_ptr<SketchCollection> c(new SketchCollection());
    ctx.adopt(c->owner);
    c->have_params = true;
    c->ksize = ksize_; c->seed = seed_; c->max_hash = max_hash_; c->is_protein = false;
    c->n_rows = n_rows_;
    c->h_offsets.resize(n_rows_ + 1);
    const cudaMemcpyKind in_kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    if (on_device) {
        SM_CUDA(cudaMemcpyAsync(c->h_offsets.data(), offsets, (n_rows_ + 1) * 8, cudaMemcpyDeviceToHost, ctx.stream));
        ctx.sync();
    } else {
        std::copy(offsets, offsets + n_rows_ + 1, c->h_offsets.begin());
    }
    if (c->h_offsets[0] != 0) throw_internal("CSR offsets must start at 0");
    for (uint64_t i = 0; i < n_rows_; i++) {
        if (c->h_offsets[i + 1] < c->h_offsets[i]) throw_internal("CSR offsets must be non-decreasing");
        if (c->h_offsets[i + 1] - c->h_offsets[i] > 0xFFFFFFFFull) throw_internal("CSR row too long");
        c->max_len = std::max<uint32_t>(c->max_len, (uint32_t)(c->h_offsets[i + 1] - c->h_offsets[i]));
    }
    c->n_hashes = c->h_offsets[n_rows_];
    c->h_nums.assign(n_rows_, num);
    c->d_hashes.reserve((c->n_hashes + 4) * 8);
    c->d_offsets.reserve((n_rows_ + 1) * 8);
    c->d_nums.reserve((n_rows_ + 1) * 4);
    if (c->n_hashes) SM_CUDA(cudaMemcpyAsync(c->d_hashes.p, hashes, c->n_hashes * 8, in_kind, ctx.stream));
    SM_CUDA(cudaMemcpyAsync(c->d_offsets.p, c->h_offsets.data(), (n_rows_ + 1) * 8, cudaMemcpyHostToDevice, ctx.stream));
    if (n_rows_) SM_CUDA(cudaMemcpyAsync(c->d_nums.p, c->h_nums.data(), n_rows_ * 4, cudaMemcpyHostToDevice, ctx.stream));
    // every row strictly ascending (the two-pointer walk is undefined otherwise; SURVEY section 4)
    SM_CUDA(cudaMemsetAsync(ctx.dsc(SC_FLAG), 0, 8, ctx.stream));
    launch_csr_check_sorted(c->d_hashes.as<uint64_t>(), c->d_offsets.as<uint64_t>(), n_rows_, ctx.dsc(SC_FLAG), ctx.stream);
    ctx.read_scalars();
    if (ctx.h_scalars[SC_FLAG]) throw_internal("CSR rows must be strictly ascending");
    c->dirty = false;
    return c.release();
}

bool SketchCollection::uniform_num(uint64_t first, uint64_t n) const {
    for (uint64_t i = 1; i < n; i++)
        if (h_nums[first + i] != h_nums[first]) return false;
    return true;
}

void SketchCollection::check_compatible(const SketchCollection &o) const {
    if (!have_params || !o.have_params) return;
    if (ksize != o.ksize) throw SourmashError(ERR_MISMATCH_KSIZES, "different ksizes cannot be compared");
    if (is_protein != o.is_protein) throw SourmashError(ERR_MISMATCH_DNAPROT, "DNA/prot minhashes cannot be compared");
    if (max_hash != o.max_hash) throw SourmashError(ERR_MISMATCH_MAXHASH, "mismatch in max_hash; comparison fail");
    if (seed != o.seed) throw SourmashError(ERR_MISMATCH_SEED, "mismatch in seed; comparison fail");
}

// every sketch of rows [first, first + n) holds exactly `len` hashes and has num == len
static bool block_is_full(const SketchCollection &c, uint64_t first, uint64_t n, uint32_t *len_out) {
    if (!n) return false;
    const uint64_t len = c.h_offsets[first + 1] - c.h_offsets[first];
    if (len == 0 || len > 0xFFFFFFFFull) return false;
    for (uint64_t i = 0; i < n; i++) {
        if (c.h_offsets[first + i + 1] - c.h_offsets[first + i] != len || c.h_nums[first + i] != len) return false;
    }
    *len_out = (uint32_t)len;
    return true;
}

// cells (index rows x queries) per block of linear_find: SMB200_FIND_BLOCK_MCELLS overrides the default (128 M)
static uint64_t find_block_cells_from_env() {
    const char *e = getenv("SMB200_FIND_BLOCK_MCELLS");
    const uint64_t m = e ? strtoull(e, nullptr, 10) : 128;
    return (m ? m : 1) << 20;
}
static const uint64_t g_find_block_cells = find_block_cells_from_env();
// linear_find's count path: 0 = stream the index (find_stream.cu) when it is large against the query batch,
// 1 = always the general join, 2 = stream whenever the shapes allow it, whatever the sizes (tests), 3 = as 2 with a tiny
// buffer for the written-out filter hits, which forces the re-run with in-kernel lookups (tests).  SMB200_FIND_PATH sets it.
int g_find_path = [] {
    const char *e = getenv("SMB200_FIND_PATH");
    return e ? atoi(e) : 0;
}();
int g_compare_path = 0;  // 0 = choose from the data, 1 = dense kernels, 2 = probe form wherever the block fits it

// The part of the probe-form decision that the compare path and the row collection make: forced sparse always probes;
// by default a block probes unless an earlier probe over the same rows found the dense kernels the better choice.
// The block's size tests come on top (compare_block_device; compare_matrix_allgather decides before the gather).
bool probe_form_allowed(const SketchCollection &rows) {
    return (g_compare_path == 0 && !rows.probe_dense_preferred) || g_compare_path == 2;
}

static int bit_length64(uint64_t x) {
    int b = 0;
    while (x) { b++; x >>= 1; }
    return b;
}

// The hash-grouped postings of a block's build side (join.cu), living in the calling thread's scratch
// (ctx.join[0,1,6,7], sort_tmp_k/v, misc[1]): built either inside compare_block_device or ahead of it --
// compare_matrix_allgather builds the table of a rank's own rows while the other ranks' rows are in flight.
// `side` (optional): the kernels go to that stream instead of the thread's own -- the scratch is still reserved in the
// thread's stream order, `side` starts behind `side_go` recorded there, and the caller makes its stream wait for `side`
// before the table (or the scratch) is touched again.
void join_table_build(Context &ctx, JoinTable &jt, const uint64_t *bh, const uint64_t *bo, uint64_t b0, uint64_t n_build,
                      uint64_t n_bp, bool with_filter, cudaStream_t side, cudaEvent_t side_go) {
    cudaStream_t st = ctx.stream;
    // slots: the power of two at or above 1.5 x the postings (postings of one hash share a slot, so the load is
    // below 0.67 whatever the data; the memsets and the scan over the slots are a third of the build at 5 M postings)
    int log2_t = 12;
    while ((1ull << log2_t) < n_bp + n_bp / 2) log2_t++;
    const uint64_t T = 1ull << log2_t;
    ctx.join[0].reserve((T + 2) * 8);
    ctx.join[1].reserve((T + 2) * 8);
    ctx.sort_tmp_k.reserve((T + 2) * 8);
    ctx.sort_tmp_v.reserve((T + 2) * 4);
    ctx.join[6].reserve((n_bp + 1) * 4);
    ctx.join[7].reserve((n_bp + 1) * 4);
    ctx.scan_tmp.reserve(scan_tmp_bytes(T + 2) + 256);
    // presence filter in front of the key table (16 bits per build-side hash, 2^20 .. 2^30 bits)
    int log2_f = 20;
    while (log2_f < 30 && (1ull << log2_f) < 16 * n_bp) log2_f++;
    uint32_t *filter = nullptr;
    if (with_filter) {
        ctx.misc[1].reserve((1ull << log2_f) / 8 + 256);
        filter = ctx.misc[1].as<uint32_t>();
    }
    unsigned long long *tkey = ctx.join[0].as<unsigned long long>(), *tcount = ctx.join[1].as<unsigned long long>();
    uint64_t *toff = ctx.sort_tmp_k.as<uint64_t>();
    uint32_t *tcursor = ctx.sort_tmp_v.as<uint32_t>(), *slot_of = ctx.join[6].as<uint32_t>(), *grows = ctx.join[7].as<uint32_t>();
    if (side) {
        SM_CUDA(cudaEventRecord(side_go, ctx.stream));
        SM_CUDA(cudaStreamWaitEvent(side, side_go, 0));
        st = side;
    }
    {
        ProfScope prof(PROF_SORT, st);
        SM_CUDA(cudaMemsetAsync(tkey, 0xFF, (T + 1) * 8, st));
        SM_CUDA(cudaMemsetAsync(tcount, 0, (T + 2) * 8, st));
        SM_CUDA(cudaMemsetAsync(tcursor, 0, (T + 1) * 4, st));
        if (filter) SM_CUDA(cudaMemsetAsync(filter, 0, (1ull << log2_f) / 8, st));
        launch_group_insert(bh, bo, b0, n_build, tkey, tcount, slot_of, log2_t, filter, log2_f, st);
        scan_exclusive_u64(reinterpret_cast<uint64_t *>(tcount), toff, T + 2, ctx.scan_tmp.p, st);
        launch_group_fill(bo, b0, n_build, slot_of, toff, tcursor, grows, st);
    }
    jt.valid = true;
    jt.ctx_id = ctx.id;
    jt.bh = bh; jt.bo = bo; jt.b0 = b0; jt.n_build = n_build; jt.n_bp = n_bp;
    jt.log2_t = log2_t; jt.log2_f = log2_f; jt.has_filter = filter != nullptr;
}

// One block of the matrix into DEVICE outputs.  A large enough block takes the probe form of the join
// (only pairs sharing a hash are walked) unless an earlier probe over the same rows found the dense
// kernels the better choice; any other block is walked densely, on ranks when every sketch is full.
// Same integers either way.
void compare_block_device(SketchCollection &rows, uint64_t r0, uint64_t nr, SketchCollection &cols, uint64_t c0,
                          uint64_t nc, int mode, uint32_t *common, uint32_t *size, double *ratio, uint64_t ld,
                          const JoinTable *prebuilt, cudaEvent_t cols_ready) {
    Context &ctx = Context::get();
    cudaStream_t st = ctx.stream;
    const uint64_t *rh = rows.d_hashes.as<uint64_t>(), *ro = rows.d_offsets.as<uint64_t>();
    const uint64_t *ch = cols.d_hashes.as<uint64_t>(), *co = cols.d_offsets.as<uint64_t>();
    const uint32_t *rnum = rows.d_nums.as<uint32_t>();
    // rows and columns from the same collection with the row range inside the column range (the
    // all-vs-all case, whole or row-sharded): one postings set serves both sides
    const bool shared = (&rows == &cols) && r0 >= c0 && r0 + nr <= c0 + nc;
    const uint64_t n_r = shared ? 0 : rows.h_offsets[r0 + nr] - rows.h_offsets[r0];
    const uint64_t n_c = cols.h_offsets[c0 + nc] - cols.h_offsets[c0];
    const uint64_t n = n_r + n_c;
    const bool force_dense = g_compare_path == 1, force_sparse = g_compare_path == 2;
    const bool big = n > 0 && nr * nc >= 4096 && nr < (1ull << 31) && nc < (1ull << 31);
    // full num sketches (Jaccard): the dense walk can run on 32-bit ranks with a fixed trip count
    uint32_t L = 0, Lc = 0;
    const bool full = mode == 0 && big && block_is_full(rows, r0, nr, &L) && block_is_full(cols, c0, nc, &Lc) && L == Lc &&
                      compare_full_fits(L);
    // Probe form of the join (the sparse path): the postings of the smaller side are grouped by hash in a
    // hash table and every hash of the other side looks its run up -- O(build side) to build, no sort, and
    // no host round trip anywhere in the block as long as the pair list fits the cell count.  A row shard
    // of the all-vs-all matrix therefore costs its share of the rows, which is what lets the matrix scale
    // over GPUs.  An empty build side gives an empty table: every cell is then written as unrelated.
    const uint64_t n_rp = rows.h_offsets[r0 + nr] - rows.h_offsets[r0];
    // When is the dense walk the better choice?  It costs about (|row| + |column|) / 2 steps per cell; the
    // probe form costs one bitmap test per incidence plus the walk of the related pairs.  Measured at
    // num = 500 the break-even was 8 incidences per cell, i.e. one per ~60 walk steps; scale with the
    // sketch sizes (scaled sketches of 5 000 hashes: 80 per cell).
    const double avg_len = 0.5 * ((double)(rows.h_offsets[r0 + nr] - rows.h_offsets[r0]) / (double)nr + (double)n_c / (double)nc);
    const uint64_t dense_if_above = (uint64_t)((double)nr * (double)nc * std::max(1.0, avg_len / 60.0));
    // the table goes over the side with fewer hashes (a query batch against an index block: the queries)
    const bool build_cols = n_c < n_rp;
    const uint64_t n_bp = build_cols ? n_c : n_rp, n_build = build_cols ? nc : nr;
    const uint64_t *bh = build_cols ? ch : rh, *bo = build_cols ? co : ro, *ph = build_cols ? rh : ch, *po = build_cols ? ro : co;
    const uint64_t b0 = build_cols ? c0 : r0, p0 = build_cols ? r0 : c0, n_probe = build_cols ? nr : nc;
    const bool probe = !force_dense && n > 0 && (force_sparse || big) && nr < (1ull << 31) && nc < (1ull << 31) &&
                       n_bp < (1ull << 31) && probe_form_allowed(rows);
    // Column hashes still in flight: the probe form with the table over the ROWS waits for them right before its probe
    // launch (what it queues first needs the rows and the column offsets only); everything else needs them now.
    cudaEvent_t probe_waits = nullptr;
    if (probe && !build_cols) probe_waits = cols_ready;
    else if (cols_ready) SM_CUDA(cudaStreamWaitEvent(st, cols_ready, 0));
    if (probe) {
        // the table: handed in (built over exactly this block's build side, on this thread's scratch) or built here;
        // with a presence filter in front of it when the probing side is a different, larger collection
        JoinTable own;
        const JoinTable *jt = prebuilt;
        if (!(jt && jt->valid && jt->ctx_id == ctx.id && jt->bh == bh && jt->bo == bo && jt->b0 == b0 && jt->n_build == n_build &&
              jt->n_bp == n_bp)) {
            const uint64_t n_pp = build_cols ? n_rp : n_c;
            join_table_build(ctx, own, bh, bo, b0, n_build, n_bp, (&rows != &cols) && n_pp >= 4 * n_bp);
            jt = &own;
        }
        const int log2_t = jt->log2_t, log2_f = jt->log2_f;
        const uint64_t n_words = (nr * nc + 63) / 64;
        ctx.scan_tmp.reserve(scan_tmp_bytes(n_words) + 256);
        const uint32_t *filter = jt->has_filter ? ctx.misc[1].as<uint32_t>() : nullptr;
        const unsigned long long *tkey = ctx.join[0].as<unsigned long long>();
        const uint64_t *toff = ctx.sort_tmp_k.as<uint64_t>();
        const uint32_t *grows = ctx.join[7].as<uint32_t>();
        SM_CUDA(cudaMemsetAsync(ctx.dsc(SC_CNT), 0, 8, st));
        ProfScope prof(PROF_COMPARE, st);
        if (mode == 1) {
            uint32_t *cmat = common;
            uint64_t cld = ld;
            if (!cmat) {
                ctx.join[2].reserve(nr * nc * 4 + 256);
                cmat = ctx.join[2].as<uint32_t>();
                cld = nc;
            }
            SM_CUDA(cudaMemset2DAsync(cmat, cld * 4, 0, nc * 4, nr, st));
            if (probe_waits) SM_CUDA(cudaStreamWaitEvent(st, probe_waits, 0));
            launch_probe_group(true, build_cols, tkey, toff, grows, log2_t, ph, po, p0, n_probe, cmat, cld, nullptr, n_build,
                               ctx.dsc(SC_CNT), filter, log2_f, st);
            if (size || ratio || cmat != common)  // (counts only, straight into the caller's matrix: nothing left to do)
                launch_fill_cells(ro, rnum, r0, nr, co, c0, nc, 1, cmat, cld, common, size, ratio, ld, st);
        } else {
            ctx.join[2].reserve((n_words + 1) * 8);
            ctx.join[3].reserve((n_words + 1) * 8);
            ctx.join[4].reserve((n_words + 1) * 8);
            unsigned long long *bitmap = ctx.join[2].as<unsigned long long>();
            uint64_t *counts = ctx.join[3].as<uint64_t>(), *pre = ctx.join[4].as<uint64_t>();
            SM_CUDA(cudaMemsetAsync(bitmap, 0, n_words * 8, st));
            // (the unrelated-pair values need row lengths only: written first, they overlap a transfer the probe waits for)
            launch_fill_cells(ro, rnum, r0, nr, co, c0, nc, 0, nullptr, 0, common, size, ratio, ld, st);  // as if unrelated
            if (probe_waits) SM_CUDA(cudaStreamWaitEvent(st, probe_waits, 0));
            launch_probe_group(false, build_cols, tkey, toff, grows, log2_t, ph, po, p0, n_probe, nullptr, 0, bitmap, n_build,
                               ctx.dsc(SC_CNT), filter, log2_f, st);
            launch_popc_words(bitmap, n_words, counts, st);
            scan_exclusive_u64(counts, pre, n_words, ctx.scan_tmp.p, st);
            // the pair list can hold every cell of a block of up to 2^26 cells: then the walk reads its
            // count on the device and nothing waits for the host; larger blocks size the list first
            uint64_t cap = nr * nc;
            if (cap > (1ull << 26)) {
                uint64_t tail[2];
                ctx.fetch2(pre + (n_words - 1), counts + (n_words - 1), tail);
                cap = tail[0] + tail[1];
            }
            if (cap) {
                ctx.join[5].reserve((cap + 1) * 8);
                launch_expand_bits(bitmap, pre, n_words, ctx.join[5].as<uint64_t>(), st, cap);
                // the whole square of ONE collection whose sketches share a `num`: each unordered pair is walked once
                const bool symmetric = (&rows == &cols) && r0 == c0 && nr == nc && rows.uniform_num(r0, nr);
                launch_walk_pairs(ctx.join[5].as<uint64_t>(), cap, rh, ro, rnum, r0, ch, co, c0, nc, common, size, ratio, ld, st,
                                  pre + (n_words - 1), counts + (n_words - 1), build_cols ? 0 : nr, symmetric);  // probe-major cell ids
            }
        }
        // The probe path is exact whatever the data; whether the dense kernels would have been faster
        // (mostly-related collections) is learned once per row collection, from its first block.
        if (!rows.probe_checked && !force_sparse) {
            ctx.read_scalars();
            rows.probe_checked = true;
            rows.probe_dense_preferred = ctx.h_scalars[SC_CNT] > dense_if_above;
        }
        return;
    }
    if (!full) {
        launch_compare_cross(rh, ro, rnum, r0, nr, ch, co, c0, nc, mode, common, size, ratio, ld, cols.max_len, ctx.sm_count, st);
        return;
    }
    // full num sketches: every hash is replaced by its rank among the block's hashes, from the sorted postings
    // (head flags -> scan -> scatter back to sketch order)
    ctx.join[0].reserve((n + 1) * 8);
    ctx.join[1].reserve((n + 1) * 8);
    uint64_t *keys = ctx.join[0].as<uint64_t>(), *vals = ctx.join[1].as<uint64_t>();
    {
        ProfScope prof(PROF_SORT, st);
        ctx.sort_tmp_k.reserve((n + 1) * 8);
        ctx.sort_tmp_v.reserve((n + 1) * 8);
        ctx.scan_tmp.reserve(std::max(radix_sort_scan_bytes(n), scan_tmp_bytes(n)) + 256);
        if (!shared) launch_postings(rh, ro, r0, nr, 0, keys, vals, st);
        launch_postings(ch, co, c0, nc, shared ? 0 : 1, keys + n_r, vals + n_r, st);
        SM_CUDA(cudaMemsetAsync(ctx.dsc(SC_TMAX), 0, 8, st));
        launch_max_u64(keys, n, ctx.dsc(SC_TMAX), st);
        ctx.read_scalars();
        radix_sort_pairs(keys, vals, n, ctx.sort_tmp_k.as<uint64_t>(), ctx.sort_tmp_v.as<uint64_t>(),
                         std::max(1, bit_length64(ctx.h_scalars[SC_TMAX])), ctx.scan_tmp.p, ctx.scan_tmp.cap, st);
    }
    ctx.join[2].reserve((n + 1) * 8);
    ctx.join[3].reserve((n + 1) * 8);
    ctx.join[6].reserve((n + 1) * 4);
    uint64_t *flags = ctx.join[2].as<uint64_t>(), *pre = ctx.join[3].as<uint64_t>();
    uint32_t *ranks = ctx.join[6].as<uint32_t>();
    launch_heads(keys, n, flags, st);
    scan_exclusive_u64(flags, pre, n, ctx.scan_tmp.p, st);
    launch_scatter_ranks(keys, vals, pre, n, L, n_r, ranks, st);
    const uint32_t *rb = ranks + n_r;                                  // column sketches
    const uint32_t *ra = shared ? rb + (r0 - c0) * (uint64_t)L : ranks;  // row sketches
    launch_compare_full(ra, rb, L, nr, nc, common, size, ratio, ld, st);
}

void compare_matrix(SketchCollection &rows, uint64_t r0, uint64_t nr, SketchCollection &cols, uint64_t c0, uint64_t nc,
                    int mode, uint32_t *common, uint32_t *size, double *ratio, uint64_t ld, bool out_on_device) {
    rows.check_compatible(cols);
    rows.finalize();
    cols.finalize();
    if (r0 + nr > rows.n_rows || c0 + nc > cols.n_rows) throw_internal("compare block outside the collections");
    if (nr == 0 || nc == 0) return;
    if (ld < nc) throw_internal("ld smaller than the block width");
    Context &ctx = Context::get();
    cudaStream_t st = ctx.stream;
    if (out_on_device) {
        compare_block_device(rows, r0, nr, cols, c0, nc, mode, common, size, ratio, ld);
        ctx.sync();
        return;
    }
    // host output: row blocks of up to 2^25 cells through two sets of device scratch; the copy of
    // block b back to the host (copy stream) overlaps the kernels of block b + 1 (library stream)
    const uint64_t block_rows = std::max<uint64_t>(1, std::min<uint64_t>(nr, (1ull << 25) / nc));
    DevBuf *bc[2] = {&ctx.misc[5], &ctx.misc[2]}, *bs[2] = {&ctx.misc[6], &ctx.misc[3]}, *br[2] = {&ctx.misc[7], &ctx.misc[4]};
    const int n_sets = nr > block_rows ? 2 : 1;
    for (int k = 0; k < n_sets; k++) {
        if (common) bc[k]->reserve(block_rows * nc * 4);
        if (size) bs[k]->reserve(block_rows * nc * 4);
        if (ratio) br[k]->reserve(block_rows * nc * 8);
    }
    cudaEvent_t *ev_done = ctx.ev_done, *ev_free = ctx.ev_free;
    cudaStream_t cs = ctx.copy_stream;
    auto copy_back = [&](void *dst, uint64_t dst_ld_bytes, const void *src, uint64_t row_bytes, uint64_t n_rows_blk) {
        if (dst_ld_bytes == row_bytes)  // contiguous: one linear copy
            SM_CUDA(cudaMemcpyAsync(dst, src, row_bytes * n_rows_blk, cudaMemcpyDeviceToHost, cs));
        else
            SM_CUDA(cudaMemcpy2DAsync(dst, dst_ld_bytes, src, row_bytes, row_bytes, n_rows_blk, cudaMemcpyDeviceToHost, cs));
    };
    uint64_t blk = 0;
    for (uint64_t b0 = 0; b0 < nr; b0 += block_rows, blk++) {
        const uint64_t bn = std::min(block_rows, nr - b0);
        const int k = (int)(blk & 1);
        if (blk >= 2) SM_CUDA(cudaStreamWaitEvent(st, ev_free[k], 0));  // this set's previous copy has left
        compare_block_device(rows, r0 + b0, bn, cols, c0, nc, mode, common ? bc[k]->as<uint32_t>() : nullptr,
                             size ? bs[k]->as<uint32_t>() : nullptr, ratio ? br[k]->as<double>() : nullptr, nc);
        SM_CUDA(cudaEventRecord(ev_done[k], st));
        SM_CUDA(cudaStreamWaitEvent(cs, ev_done[k], 0));
        if (common) copy_back(common + b0 * ld, ld * 4, bc[k]->p, nc * 4, bn);
        if (size) copy_back(size + b0 * ld, ld * 4, bs[k]->p, nc * 4, bn);
        if (ratio) copy_back(ratio + b0 * ld, ld * 8, br[k]->p, nc * 8, bn);
        SM_CUDA(cudaEventRecord(ev_free[k], cs));
    }
    SM_CUDA(cudaStreamSynchronize(cs));
    ctx.sync();
}

// Leaf-pairing pass of scaffold (src/index/sbt.rs:356-381).  The reference runs count_common of the
// popped leaf against every remaining leaf -- O(N^2) intersections; here the whole count matrix
// comes from one compare_block_device call and the pass itself is a scan of its rows.
uint64_t scaffold_pairs(SketchCollection &c, uint64_t *pairs_first, uint64_t *pairs_second) {
    c.finalize();
    const uint64_t n = c.n_rows;
    if (n == 0) return 0;
    Context &ctx = Context::get();
    std::vector<uint32_t> common((size_t)n * n);
    {
        ctx.misc[5].reserve(n * n * 4 + 256);
        compare_block_device(c, 0, n, c, 0, n, 1, ctx.misc[5].as<uint32_t>(), nullptr, nullptr, n);
        SM_CUDA(cudaMemcpyAsync(common.data(), ctx.misc[5].p, n * n * 4, cudaMemcpyDeviceToHost, ctx.stream));
        ctx.sync();
    }
    std::vector<uint64_t> alive(n);
    for (uint64_t i = 0; i < n; i++) alive[i] = i;
    uint64_t n_pairs = 0;
    while (!alive.empty()) {
        const uint64_t next = alive.back();
        alive.pop_back();
        if (alive.empty()) {
            pairs_first[n_pairs] = next;
            pairs_second[n_pairs++] = ~0ull;
            break;
        }
        const uint32_t *row = common.data() + (size_t)next * n;
        size_t similar_pos = 0;
        uint32_t current_max = 0;
        for (size_t pos = 0; pos < alive.size(); pos++) {
            const uint32_t cm = row[alive[pos]];
            if (cm > current_max) { current_max = cm; similar_pos = pos; }  // strict: the first maximum wins
        }
        pairs_first[n_pairs] = next;
        pairs_second[n_pairs++] = alive[similar_pos];
        alive.erase(alive.begin() + (std::ptrdiff_t)similar_pos);
    }
    return n_pairs;
}

uint64_t linear_find(SketchCollection &index, SketchCollection &queries, int mode, double threshold, uint64_t *hit_offsets,
                     uint64_t *hits, uint64_t hits_cap) {
    std::vector<std::vector<uint64_t>> per_query = linear_find_lists(index, queries, mode, threshold);
    const uint64_t nq = per_query.size();
    uint64_t total = 0;
    for (uint64_t q = 0; q < nq; q++) {
        if (hit_offsets) hit_offsets[q] = total;
        for (uint64_t id : per_query[q]) {
            if (hits && total < hits_cap) hits[total] = id;
            total++;
        }
    }
    if (hit_offsets) hit_offsets[nq] = total;
    return total;
}

std::vector<std::vector<uint64_t>> linear_find_lists(SketchCollection &index, SketchCollection &queries, int mode, double threshold) {
    index.check_compatible(queries);
    index.finalize();
    queries.finalize();
    const uint64_t ni = index.n_rows, nq = queries.n_rows;
    std::vector<std::vector<uint64_t>> per_query(nq);
    if (ni && nq) {
        Context &ctx = Context::get();
        cudaStream_t st = ctx.stream;
        const uint64_t block_rows = std::max<uint64_t>(1, std::min<uint64_t>(ni, (g_find_block_cells) / nq));
        const uint64_t cells = block_rows * nq;
        std::vector<uint64_t> cellbuf;
        // Containment with a threshold >= 0: a cell can only hit when the pair shares a hash, and the join leaves
        // the shared-hash COUNT of every cell in a u32 matrix.  One pass over that matrix picks the hits (count
        // > 0 and count / |node| > threshold); the f64 ratio matrix, the flag matrix, its scan and the compaction
        // of the general path (7 GB of traffic per 128 M cells) are never materialised.
        // Similarity takes the same path when no index sketch has a `num` (scaled sketches): lib.rs:470-499 with
        // self.num == 0 gives common = |A n B| and size = |A u B| = |A| + |B| - common, both known from the count.
        bool index_unbounded = true;
        for (uint32_t v : index.h_nums) index_unbounded &= v == 0;
        const bool count_sim = mode == 0 && index_unbounded;
        const bool count_path = (mode == 1 || count_sim) && threshold >= 0.0;
        // a large index against a (much) smaller query batch: stream the index at HBM rate (find_stream.cu); the query
        // table's slot numbers (twice the query hashes + 32 per table slice) are u32
        const bool stream = count_path && g_find_path != 1 && queries.n_hashes > 0 && queries.n_hashes < (1ull << 31) &&
                            find_stream_table_slots(queries.n_hashes) <= (1ull << 32) && nq < (1ull << 31) &&
                            index.max_len < (1u << 31) &&
                            (g_find_path >= 2 || (index.n_hashes >= 4 * queries.n_hashes && index.n_hashes >= (1ull << 22)));
        uint32_t *q_tstart = nullptr;
        uint64_t q_tscale = 0;
        if (stream) index.ensure_partitions();
        ctx.misc[3].reserve((cells + 1) * 8);      // flags, [query][index row] / the hit list of the count paths
        if (!stream) ctx.misc[2].reserve(cells * 8);  // ratio or counts, [index row][query]
        if (!count_path) {
            ctx.misc[4].reserve((cells + 1) * 8);  // scan
            ctx.misc[5].reserve((cells + 1) * 8);  // compacted cell ids
        }
        for (uint64_t b0 = 0; count_path && b0 < ni; b0 += block_rows) {
            const uint64_t bn = std::min(block_rows, ni - b0);
            uint32_t *cmat = ctx.misc[2].as<uint32_t>();  // cells * 8 bytes reserved: room for the u32 counts
            uint64_t *found = ctx.misc[3].as<uint64_t>();
            if (stream) {
                // the index streams past per-slice Bloom filters of the query hashes held in shared memory (find_stream.cu)
                if (b0 == 0) {   // the query side: exact table + filters, once per search
                    const size_t slots = find_stream_table_slots(queries.n_hashes);
                    const uint32_t ts = find_stream_table_slices();
                    ctx.join[0].reserve(slots * 8);                                   // keys
                    ctx.join[1].reserve(slots * 4);                                   // list heads
                    ctx.join[6].reserve((queries.n_hashes + 1) * 4);                  // node -> next
                    ctx.join[7].reserve((queries.n_hashes + 1) * 4);                  // node -> query
                    ctx.join[2].reserve(((size_t)ts + 1) * (nq + 1) * 4);             // where each query meets each table slice
                    ctx.join[3].reserve(((size_t)ts + 2) * 8 + ((size_t)ts + 2) * 4); // sums, then slice starts
                    q_tstart = reinterpret_cast<uint32_t *>(ctx.join[3].as<unsigned long long>() + ts + 2);
                    launch_qtable_build(queries.d_hashes.as<uint64_t>(), queries.d_offsets.as<uint64_t>(), nq, index.part_top,
                                        ctx.join[2].as<uint32_t>(), ctx.join[3].as<unsigned long long>(), q_tstart,
                                        ctx.join[0].as<unsigned long long>(), ctx.join[1].as<int32_t>(), ctx.join[6].as<int32_t>(),
                                        ctx.join[7].as<uint32_t>(), &q_tscale, st);
                    ctx.misc[6].reserve(find_stream_filter_bytes(index.n_parts) + (size_t)index.n_parts * 4 + 256);
                    SM_CUDA(cudaMemsetAsync(ctx.misc[6].p, 0, find_stream_filter_bytes(index.n_parts), st));
                    launch_filters_build(queries.d_hashes.as<uint64_t>(), queries.n_hashes, index.part_scale, index.part_top,
                                         index.n_parts, ctx.misc[6].as<uint32_t>(), st);
                    // count matrix / touched-row bitmap: zero from the last search, or zeroed now
                    const size_t c_bytes = (size_t)block_rows * nq * 4, b_bytes = ((size_t)block_rows + 31) / 32 * 4 + 4;
                    const bool grow = ctx.find_cmat.cap < c_bytes || ctx.find_bits.cap < b_bytes;
                    ctx.find_cmat.reserve(c_bytes);
                    ctx.find_bits.reserve(b_bytes);
                    ctx.find_rows.reserve((size_t)block_rows * 4 + 4);
                    if (grow || !ctx.find_clean) {
                        SM_CUDA(cudaMemsetAsync(ctx.find_cmat.p, 0, ctx.find_cmat.cap, st));
                        SM_CUDA(cudaMemsetAsync(ctx.find_bits.p, 0, ctx.find_bits.cap, st));
                        SM_CUDA(cudaMemsetAsync(ctx.dsc(SC_TOUCHED), 0, 8, st));
                    }
                    ctx.find_clean = false;   // until this search has cleaned up after itself
                }
                uint32_t *work_ctr = ctx.misc[6].as<uint32_t>() + find_stream_filter_bytes(index.n_parts) / 4;  // behind the filters
                SM_CUDA(cudaMemsetAsync(work_ctr, 0, (size_t)index.n_parts * 4, st));
                // written-out filter hits: room for one in eight index hashes of the block (false positives are ~1 %)
                const uint64_t blk_hashes = index.h_offsets[b0 + bn] - index.h_offsets[b0];
                const uint64_t spill_cap = g_find_path == 3 ? 64 : std::min<uint64_t>(std::max<uint64_t>(blk_hashes / 8, 1ull << 20), 1ull << 27);
                ctx.misc[4].reserve((spill_cap + 1) * 8);
                ctx.misc[5].reserve((spill_cap + 1) * 4);
                SM_CUDA(cudaMemsetAsync(ctx.dsc(SC_SPILL), 0, 8, st));
                auto probe = [&](bool deferred, int phase) {
                    launch_stream_probe(index.d_hashes.as<uint64_t>(), index.d_offsets.as<uint64_t>(), b0, bn, index.d_part_off.as<uint32_t>(),
                                        index.n_rows, index.n_parts, ctx.misc[6].as<uint32_t>(), ctx.join[0].as<unsigned long long>(),
                                        ctx.join[1].as<int32_t>(), ctx.join[6].as<int32_t>(), ctx.join[7].as<uint32_t>(), q_tstart, q_tscale,
                                        index.part_top, ctx.find_cmat.as<uint32_t>(), nq, ctx.find_bits.as<uint32_t>(), ctx.find_rows.as<uint32_t>(),
                                        ctx.dsc(SC_TOUCHED), work_ctr, deferred ? ctx.misc[4].as<uint64_t>() : nullptr, ctx.misc[5].as<uint32_t>(),
                                        ctx.dsc(SC_SPILL), spill_cap, phase, ctx.sm_count, st);
                };
                auto hit_pass = [&]() {
                    SM_CUDA(cudaMemsetAsync(ctx.dsc(SC_CNT), 0, 8, st));
                    launch_touched_hits(ctx.find_cmat.as<uint32_t>(), bn, nq, index.d_offsets.as<uint64_t>(), b0,
                                        count_sim ? queries.d_offsets.as<uint64_t>() : nullptr, threshold, ctx.find_bits.as<uint32_t>(),
                                        ctx.find_rows.as<uint32_t>(), ctx.dsc(SC_TOUCHED), found, cells, ctx.dsc(SC_CNT), ctx.sm_count, st);
                };
                probe(true, 0);
                probe(true, 1);
                hit_pass();
                ctx.read_scalars();
                if (ctx.h_scalars[SC_SPILL] > spill_cap) {
                    // more filter hits than the buffer holds (a heavily related index): the counts were partial (the hit pass
                    // has wiped them again) -- once more, with the lookups inside the probe kernel
                    SM_CUDA(cudaMemsetAsync(work_ctr, 0, (size_t)index.n_parts * 4, st));
                    probe(false, 0);
                    hit_pass();
                    ctx.read_scalars();
                }
            } else {
                compare_block_device(index, b0, bn, queries, 0, nq, 1, cmat, nullptr, nullptr, nq);
                SM_CUDA(cudaMemsetAsync(ctx.dsc(SC_CNT), 0, 8, st));
                launch_count_hits(cmat, bn, nq, index.d_offsets.as<uint64_t>(), b0, count_sim ? queries.d_offsets.as<uint64_t>() : nullptr,
                                  threshold, found, cells, ctx.dsc(SC_CNT), st);
                ctx.read_scalars();
            }
            const uint64_t n_hit = ctx.h_scalars[SC_CNT];
            if (n_hit > cells) throw_internal("linear_find: hit list overflow");
            cellbuf.resize(n_hit);
            if (n_hit) {
                SM_CUDA(cudaMemcpyAsync(cellbuf.data(), found, n_hit * 8, cudaMemcpyDeviceToHost, st));
                ctx.sync();
            }
            std::sort(cellbuf.begin(), cellbuf.end());  // cell id = query * bn + row: per query, ascending index id
            for (uint64_t cell : cellbuf) per_query[cell / bn].push_back(b0 + cell % bn);
        }
        if (stream) ctx.find_clean = true;   // every block's hit pass has cleared what its probe wrote
        for (uint64_t b0 = 0; !count_path && b0 < ni; b0 += block_rows) {
            const uint64_t bn = std::min(block_rows, ni - b0);
            const uint64_t n_cells = bn * nq;
            compare_block_device(index, b0, bn, queries, 0, nq, mode, nullptr, nullptr, ctx.misc[2].as<double>(), nq);
            ctx.scan_tmp.reserve(scan_tmp_bytes(cells) + 256);
            launch_threshold_flags_t(ctx.misc[2].as<double>(), bn, nq, threshold, ctx.misc[3].as<uint64_t>(), st);
            scan_exclusive_u64(ctx.misc[3].as<uint64_t>(), ctx.misc[4].as<uint64_t>(), n_cells, ctx.scan_tmp.p, st);
            launch_compact_indices(ctx.misc[3].as<uint64_t>(), ctx.misc[4].as<uint64_t>(), n_cells, ctx.misc[5].as<uint64_t>(), st);
            // number of hits = scan[last] + flag[last]
            uint64_t tail[2];
            SM_CUDA(cudaMemcpyAsync(&tail[0], ctx.misc[4].as<uint64_t>() + (n_cells - 1), 8, cudaMemcpyDeviceToHost, st));
            SM_CUDA(cudaMemcpyAsync(&tail[1], ctx.misc[3].as<uint64_t>() + (n_cells - 1), 8, cudaMemcpyDeviceToHost, st));
            ctx.sync();
            const uint64_t n_hit = tail[0] + tail[1];
            cellbuf.resize(n_hit);
            if (n_hit) {
                SM_CUDA(cudaMemcpyAsync(cellbuf.data(), ctx.misc[5].p, n_hit * 8, cudaMemcpyDeviceToHost, st));
                ctx.sync();
            }
            for (uint64_t cell : cellbuf) per_query[cell / bn].push_back(b0 + cell % bn);  // ascending index id per query
        }
    }
    return per_query;
}

}  // namespace smb200
