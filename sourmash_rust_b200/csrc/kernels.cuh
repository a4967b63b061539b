// Launchers of every hand-written sm_100a kernel in the library.
// All take the stream explicitly; none synchronise.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace smb200 {

// ---- sketch.cu --------------------------------------------------------------------------
#ifndef SK_TILE_V          // overridable for kernel A/B builds (tests/manual/build_variant.py)
#define SK_TILE_V 4096
#endif
#ifndef SK_THREADS_V
#define SK_THREADS_V 256
#endif
#ifndef SK_CTAS_V
#define SK_CTAS_V 5   // 42 KB of tile views per CTA (byte-shifted ASCII copies): five fit the 227 KB of an SM
#endif
constexpr int SK_TILE = SK_TILE_V;          // window starts per tile
constexpr int SK_THREADS = SK_THREADS_V;    // SK_TILE / SK_THREADS windows per thread per tile
constexpr int SK_CTAS_PER_SM = SK_CTAS_V;   // resident persistent CTAs per SM
constexpr int SK_MAX_GENERIC_K = 8192;

// A batch of sequences resident in device memory as one ASCII buffer.
//   offsets == nullptr && read_len == 0 : one sequence buf[0, n)
//   offsets == nullptr && read_len  > 0 : n / read_len fixed-length sequences, back to back
//   offsets != nullptr                  : sequence s = buf[offsets[s], offsets[s+1]), s < n_seqs
// buf must be 16-byte aligned and readable up to n rounded up to 16 bytes.
struct SketchBatch {
    const uint8_t *buf;
    uint64_t n;        // bytes in the batch
    uint64_t n_limit;  // window starts >= n_limit are ignored (force=false replay up to the first bad k-mer)
    const uint64_t *offsets;
    uint64_t n_seqs;
    uint32_t read_len;
    uint32_t tile_lo;  // first tile this launch covers
    uint64_t seed;
    uint64_t pos_base;                  // added to the window start in out.pos / first_bad
    unsigned long long *first_bad;      // nullable: atomicMin of the first window add_sequence fails on
    uint32_t *tile_ctr;                 // two zeroed words: dynamic tile counter + finished-CTA counter (the last
                                        // CTA of a launch zeroes both again); launches sharing it must be ordered
};
// Survivors (hash <= *thr) are appended through *counter; entries beyond cap are dropped but
// still counted, so the host can detect the overflow and re-run with a larger buffer.
struct SketchOut {
    const uint64_t *thr;
    uint64_t *hash;
    uint64_t *pos;  // nullable
    uint64_t cap;
    unsigned long long *counter;
};
struct SketchOuts {  // per k-size outputs of a fused multi-k launch
    SketchOut o[3];
    unsigned long long *first_bad[3];  // nullable
};
uint32_t sketch_tile_count(uint64_t n, uint64_t n_limit);
uint32_t sketch_tiles_ready(uint32_t K, uint64_t bytes_ready);
// tiles [sb.tile_lo, tile_hi)
void launch_sketch(uint32_t K, const SketchBatch &sb, const SketchOut &out, uint32_t tile_hi, int sm_count,
                   cudaStream_t st);
bool sketch_has_fast_path(uint32_t K);
bool sketch_multi_supported(const uint32_t *ks, int nk);
void launch_sketch_multi(const uint32_t *ks, int nk, const SketchBatch &sb, const SketchOuts &outs, uint32_t tile_hi,
                         int sm_count, cudaStream_t st);

// ---- protein.cu: 6-frame translated sketching (reference src/lib.rs:275-302) --------------------
struct ProteinBatch {
    const uint8_t *buf;
    uint64_t n;
    const uint64_t *offsets;
    uint64_t n_seqs;
    uint32_t read_len;
    uint32_t ksize;
    uint64_t seed;
};
uint64_t protein_slots(uint64_t n_bytes, uint64_t n_seqs);
// aa, comp: protein_slots + 1 bytes; flags, pre: protein_slots + 1 u64; scan_tmp: scan_tmp_bytes(protein_slots + 1)
void launch_protein_sketch(const ProteinBatch &pb, const SketchOut &out, uint8_t *aa, uint8_t *comp, uint64_t *flags,
                           uint64_t *pre, void *scan_tmp, cudaStream_t st);

// ---- sortops.cu -------------------------------------------------------------------------
// keep[i] = hashes[i] passing the state-independent gate (h <= max_hash || max_hash == 0) and
// h <= *thr; compacted (order NOT preserved) into out via *counter.
void launch_filter_hashes(const uint64_t *hashes, uint64_t n, uint64_t max_hash, const uint64_t *thr,
                          uint64_t *out_hash, uint64_t *out_pos, unsigned long long *counter, cudaStream_t st);
// LSD radix sort on key bits [0, end_bit); vals may be null.  Result ends in keys/vals.
void radix_sort_pairs(uint64_t *keys, uint64_t *vals, uint64_t n, uint64_t *tmp_keys, uint64_t *tmp_vals,
                      int end_bit, void *scan_tmp, size_t scan_tmp_bytes, cudaStream_t st);
size_t radix_sort_scan_bytes(uint64_t n);
// Exclusive prefix sum (u64), in place allowed.  tmp must hold scan_tmp_bytes(n).
void scan_exclusive_u64(const uint64_t *in, uint64_t *out, uint64_t n, void *tmp, cudaStream_t st);
size_t scan_tmp_bytes(uint64_t n);
// Run-length reduce of a sorted key array: unique keys -> ukeys, sum of vals (or run lengths if
// vals == null) -> usums (must be zeroed by the callee), number of runs -> *n_unique.
// idx_tmp: n u64 of scratch.
void reduce_by_key(const uint64_t *keys, const uint64_t *vals, uint64_t n, uint64_t *ukeys, uint64_t *usums,
                   unsigned long long *n_unique, uint64_t *idx_tmp, void *scan_tmp, cudaStream_t st);
// min over vals per run (first-occurrence positions); umins pre-filled with ~0 by the callee.
void min_by_key(const uint64_t *keys, const uint64_t *vals, uint64_t n, const uint64_t *idx, uint64_t *umins,
                cudaStream_t st);
void launch_fill_u64(uint64_t *p, uint64_t v, uint64_t n, cudaStream_t st);
// 1 if keys[0..n) is strictly ascending
void launch_check_sorted(const uint64_t *keys, uint64_t n, unsigned long long *not_sorted_flag, cudaStream_t st);
// num+abundance quirk (lib.rs:206-208): see minhash.cu
// (x is read from device memory: the largest element of the freshly merged sketch)
void launch_first_new_max(const uint64_t *ukeys, const uint64_t *ufirst, uint64_t nu, const uint64_t *old_keys,
                          uint64_t n_old, const uint64_t *x, unsigned long long *t_max_plus1, cudaStream_t st);
void launch_count_key_upto(const uint64_t *keys, const uint64_t *pos, uint64_t n, const uint64_t *x,
                           const unsigned long long *t_max_plus1, unsigned long long *count, cudaStream_t st);
void launch_fix_max_abund(uint64_t *abund_x, const uint64_t *ukeys, const uint64_t *ucounts, uint64_t nu,
                          const uint64_t *x, const unsigned long long *count_upto, cudaStream_t st);
// fast fold of scaled-sketch candidates (minhash.cu: ingest): candidates already in the sorted state bump
// their abundance in place, the others are appended to news[] (capacity nc) through *n_news
void launch_fold_match(const uint64_t *cand, uint64_t nc, const uint64_t *mins, uint64_t na, uint64_t *abunds /*nullable*/,
                       uint64_t *news, unsigned long long *n_news, cudaStream_t st);
// n_news <= fold_small_limit() new hashes: one CTA sorts and run-length reduces them (ukeys, ucnt, *n_unique),
// then state and new keys are merged by rank into out_k / out_v (out_v nullable; abunds nullable)
int fold_small_limit();
void launch_fold_small(const uint64_t *news, uint32_t n_news, const uint64_t *mins, const uint64_t *abunds, uint64_t na,
                       uint64_t *ukeys, uint64_t *ucnt, unsigned long long *n_unique, uint64_t *out_k, uint64_t *out_v,
                       cudaStream_t st);
// ordered replay of add_hash (lib.rs:192-245) for non-standard parameter combinations
void launch_replay_add_hash(const uint64_t *events, uint64_t n_events, uint32_t num, uint64_t max_hash,
                            uint64_t *mins, uint64_t *abunds /*nullable*/, unsigned long long *len_io,
                            cudaStream_t st);

// ---- compare.cu -------------------------------------------------------------------------
// One pair: out[0] = |A∩B|, out[1] = |A∩B∩bottom_num(A∪B)| (== out[0] when num == 0),
// out[2] = |combined| = min(num, |A∪B|) or |A∪B| (lib.rs:428-436, 470-499).
void launch_pair_stats(const uint64_t *a, uint64_t na, const uint64_t *b, uint64_t nb, uint32_t num,
                       unsigned long long *out3, cudaStream_t st);
// flags[i] = 1 if a[i] occurs in b (both sorted, distinct)
void launch_mark_common(const uint64_t *a, uint64_t na, const uint64_t *b, uint64_t nb, uint64_t *flags,
                        cudaStream_t st);
// out[i - pre[i]] = vals[i] for every unflagged i (pre = exclusive scan of flags)
void launch_compact_unflagged(const uint64_t *vals, const uint64_t *flags, const uint64_t *pre, uint64_t n,
                              uint64_t *out, cudaStream_t st);
// out[pre[i]] = vals[i] for every flagged i with pre[i] < limit
void launch_compact_flagged(const uint64_t *vals, const uint64_t *flags, const uint64_t *pre, uint64_t n, uint64_t limit,
                            uint64_t *out, cudaStream_t st);

// CSR collections of sorted sketches: hashes[offsets[i] .. offsets[i+1]).
// Block rows [r0, r0+nr) of the row collection x cols [c0, c0+nc) of the column collection; writes
// common/size (u32) and/or ratio (f64) at out[(i - r0) * ld + (j - c0)].
// mode 0: KmerMinHash::compare -- common = |A∩B∩bottom_num(A∪B)|, size = |combined|, num = row_nums[i]
//         (lib.rs:470-508); ratio = common / max(1, size).
// mode 1: count_common with size = |row| (Leaf containment, index.rs:146-160); ratio = common/|row|.
void launch_compare_cross(const uint64_t *row_hashes, const uint64_t *row_offsets, const uint32_t *row_nums,
                          uint64_t r0, uint64_t nr, const uint64_t *col_hashes, const uint64_t *col_offsets,
                          uint64_t c0, uint64_t nc, int mode, uint32_t *common, uint32_t *size, double *ratio,
                          uint64_t ld, uint32_t max_col_len, int sm_count, cudaStream_t st);
// hits of a linear search: flags[j * nr + i] = ratio[i * nq + j] > threshold (strict '>',
// search.rs:3-9; NaN never hits) -- transposed so that each query's hits are contiguous and in
// index order
void launch_threshold_flags_t(const double *ratio, uint64_t nr, uint64_t nq, double threshold, uint64_t *flags,
                              cudaStream_t st);
// linear_find's containment fast path: hits straight from the u32 count matrix (see compare.cu)
// (q_offsets: the queries' CSR offsets for the similarity form over num == 0 sketches, else nullptr)
void launch_count_hits(const uint32_t *cmat, uint64_t nr, uint64_t nq, const uint64_t *row_offsets, uint64_t r0,
                       const uint64_t *q_offsets, double threshold, uint64_t *found, uint64_t cap, unsigned long long *n_found,
                       cudaStream_t st);
// *flag = 1 if some CSR row is not strictly ascending
void launch_csr_check_sorted(const uint64_t *hashes, const uint64_t *offsets, uint64_t n_rows, unsigned long long *flag,
                             cudaStream_t st);
// out[pre[i]] = i for flagged i (ascending)
void launch_compact_indices(const uint64_t *flags, const uint64_t *pre, uint64_t n, uint64_t *out,
                            cudaStream_t st);

// ---- join.cu: sparse all-vs-all through an inverted index (see the file header) ----------------
void launch_postings(const uint64_t *hashes, const uint64_t *offsets, uint64_t first, uint64_t n_rows, uint64_t side,
                     uint64_t *keys, uint64_t *vals, cudaStream_t st);
void launch_max_u64(const uint64_t *keys, uint64_t n, unsigned long long *out, cudaStream_t st);
// probe form of the join (join.cu): row postings grouped by hash in a hash table of 2^log2_t (+1) slots
//   tkey  (2^log2_t + 1) u64, preset to ~0;  tcount (2^log2_t + 2) u64, zeroed;  tcursor (2^log2_t + 1) u32, zeroed
//   slot_of, grows: one u32 per row posting;  toff = exclusive scan of tcount over 2^log2_t + 2 entries
void launch_group_insert(const uint64_t *rh, const uint64_t *ro, uint64_t r0, uint64_t nr, unsigned long long *tkey,
                         unsigned long long *tcount, uint32_t *slot_of, int log2_t, uint32_t *filter /*nullable, zeroed, 2^log2_f bits*/,
                         int log2_f, cudaStream_t st);
void launch_group_fill(const uint64_t *ro, uint64_t r0, uint64_t nr, const uint32_t *slot_of, const uint64_t *toff,
                       uint32_t *tcursor, uint32_t *grows, cudaStream_t st);
// the table was built over the rows (build_cols = false) or the columns of the block; the other side's
// sketches [p0, p0 + np) probe it.  count: counts into cmat[r * ld + c], else related-pairs bitmap with
// bit = probe sketch * n_build + build sketch; *incidences += hits.
void launch_probe_group(bool count, bool build_cols, const unsigned long long *tkey, const uint64_t *toff, const uint32_t *grows,
                        int log2_t, const uint64_t *ph, const uint64_t *po, uint64_t p0, uint64_t np, uint32_t *cmat, uint64_t ld,
                        unsigned long long *bitmap, uint64_t n_build, unsigned long long *incidences,
                        const uint32_t *filter /*nullable: presence bits filled by launch_group_insert*/, int log2_f, cudaStream_t st);
void launch_popc_words(const unsigned long long *bitmap, uint64_t n_words, uint64_t *counts, cudaStream_t st);
void launch_expand_bits(const unsigned long long *bitmap, const uint64_t *pre, uint64_t n_words, uint64_t *pairs,
                        cudaStream_t st, uint64_t cap = ~0ull);
void launch_fill_cells(const uint64_t *ro, const uint32_t *rnum, uint64_t r0, uint64_t nr, const uint64_t *co, uint64_t c0,
                       uint64_t nc, int mode, const uint32_t *cmat, uint64_t cld, uint32_t *common, uint32_t *size,
                       double *ratio, uint64_t ld, cudaStream_t st);
void launch_walk_pairs(const uint64_t *pairs, uint64_t n_pairs, const uint64_t *rh, const uint64_t *ro, const uint32_t *rnum,
                       uint64_t r0, const uint64_t *ch, const uint64_t *co, uint64_t c0, uint64_t nc, uint32_t *common,
                       uint32_t *size, double *ratio, uint64_t ld, cudaStream_t st, const uint64_t *n_dev_a = nullptr,
                       const uint64_t *n_dev_b = nullptr, uint64_t nr_transposed = 0, bool symmetric = false);

// ---- find_stream.cu: LinearIndex::find over a large index at HBM rate (see the file header) -----------------
uint32_t find_stream_partitions(uint64_t n_rows, uint64_t n_hashes, int sm_count);   // slices of the hash range (SM count / k)
void launch_rows_max(const uint64_t *h, const uint64_t *off, uint64_t n_rows, unsigned long long *out /*zeroed*/, cudaStream_t st);
// part_off: (P + 1) x n_rows u32, slice-major: row r meets slice p in [part_off[p][r], part_off[p + 1][r])
// slice of h = min(P - 1, mulhi(h, scale)), scale = floor(2^64 * P / (top + 1)): monotone, so a sorted row meets a slice in one stretch
uint64_t find_stream_scale(uint64_t top, uint32_t P);
void launch_part_offsets(const uint64_t *h, const uint64_t *off, uint64_t n_rows, uint64_t scale, uint32_t P, uint32_t *part_off,
                         cudaStream_t st);
size_t find_stream_filter_bytes(uint32_t P);
void launch_filters_build(const uint64_t *qh, uint64_t n, uint64_t scale, uint64_t top, uint32_t P, uint32_t *filters /*zeroed*/,
                          cudaStream_t st);
// exact table of the query side: hash -> list of its postings (node i = posting i of the packed query array), built per
// table slice in shared memory.  qpo: (slices + 1) x nq u32 scratch; sums: slices + 1 u64 scratch; tstart: slices + 1 u32;
// tkey (u64) / thead (i32): find_stream_table_slots(n_postings) entries; node_next (i32) / node_q (u32): n_postings entries
size_t find_stream_table_slots(uint64_t n_postings);
uint32_t find_stream_table_slices();
void launch_qtable_build(const uint64_t *qh, const uint64_t *qo, uint64_t nq, uint64_t top, uint32_t *qpo, unsigned long long *sums,
                         uint32_t *tstart, unsigned long long *tkey, int32_t *thead, int32_t *node_next, uint32_t *node_q,
                         uint64_t *tscale_out, cudaStream_t st);
// counts of shared hashes of index rows [b0, b0 + bn) x queries into cmat[(row - b0) * ld + query]; cmat, touched_bits
// (bn bits), *n_touched and the P work counters must be zero on entry; rows that received a count are listed in touched_rows
void launch_stream_probe(const uint64_t *ih, const uint64_t *io, uint64_t b0, uint64_t bn, const uint32_t *part_off,
                         uint64_t n_rows_total, uint32_t P, const uint32_t *filters, const unsigned long long *tkey,
                         const int32_t *thead, const int32_t *node_next, const uint32_t *node_q, const uint32_t *tstart, uint64_t tscale,
                         uint64_t top, uint32_t *cmat, uint64_t ld, uint32_t *touched_bits, uint32_t *touched_rows, unsigned long long *n_touched,
                         uint32_t *work_ctr, uint64_t *spill_hash /*nullable: resolve inside the kernel*/, uint32_t *spill_row,
                         unsigned long long *spill_n /*zeroed*/, uint64_t spill_cap, int phase /*0 = stream, 1 = resolve the spill*/,
                         int sm_count, cudaStream_t st);
// hits (query * bn + row) from the counts of the touched rows; clears every cell, bit and counter it reads
void launch_touched_hits(uint32_t *cmat, uint64_t bn, uint64_t nq, const uint64_t *row_offsets, uint64_t b0, const uint64_t *q_offsets,
                         double threshold, uint32_t *touched_bits, const uint32_t *touched_rows, unsigned long long *n_touched,
                         uint64_t *found, uint64_t cap, unsigned long long *n_found, int sm_count, cudaStream_t st);

// dense path for full num sketches: dense u32 ranks + fixed-length walk (join.cu)
void launch_scatter_ranks(const uint64_t *keys, const uint64_t *vals, const uint64_t *pre, uint64_t n, uint32_t L,
                          uint64_t b_base, uint32_t *out, cudaStream_t st);
bool compare_full_fits(uint32_t L);
void launch_compare_full(const uint32_t *ra, const uint32_t *rb, uint32_t L, uint64_t nr, uint64_t nc, uint32_t *common,
                         uint32_t *size, double *ratio, uint64_t ld, cudaStream_t st);
void launch_heads(const uint64_t *keys, uint64_t n, uint64_t *flags, cudaStream_t st);

// integer-pipe microbenchmark (bench.py: measured INT32 issue peak); returns via out[0] a checksum
void launch_int_peak(uint32_t *out, int iters, int blocks, int mode, cudaStream_t st);

}  // namespace smb200
