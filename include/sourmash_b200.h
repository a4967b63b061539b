/*
 * sourmash_b200.h -- batch extension of the sourmash C ABI for the B200 build.
 *
 * The reference ABI (sourmash.h) is per object: one sequence per kmerminhash_add_sequence call,
 * one pair per kmerminhash_compare call.  The workloads this build exists for (10^8 reads,
 * 10^4..10^6 sketches) need one call per BATCH, so that a single kernel launch covers it.  Every
 * function below is defined as a loop over reference calls, and cites them; results are
 * bit-identical to running that loop against the reference.
 *
 * Error convention: as sourmash.h (thread-local last error, zero return value).
 * Threading: as the reference (src/utils.rs:14-16) -- no library-wide lock.  Every host thread that calls in
 * gets its own CUDA stream and scratch; distinct handles may be driven from distinct threads at the same
 * time, and a handle may move between threads (the new thread waits for what the old one queued).
 * Pointers marked [host|device] are host pointers unless the call's `on_device` flag is set, in
 * which case they are device pointers of the library's device (see smgpu_set_device) and no
 * host<->device copy is made.
 */
#ifndef SOURMASH_B200_EXT_H
#define SOURMASH_B200_EXT_H

#include "sourmash.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- device ---------------------------------------------------------------------------------- */
/* Select the CUDA device this process uses (one process per GPU).  Must precede the first call
 * that touches the GPU; default is the calling thread's current device. */
void smgpu_set_device(int32_t device);
/* device ordinal in use (creates the context), SM count through *sm_count when non-NULL */
int32_t smgpu_device(int32_t *sm_count);
/* kernels this library has launched so far in this process */
uint64_t smgpu_launch_count(void);
/* the CUDA stream (cudaStream_t, as an integer) the kernels launched from the CALLING THREAD go to: lets a
 * caller bracket its calls with its own CUDA events */
uint64_t smgpu_stream(void);
/* per-kernel device timing with CUDA events on that stream: kinds 0/1/2 = sketch kernel k=21/31/51,
 * 3 = sketch kernel other k, 4 = compare matrix kernel.  read() waits for the recorded events and
 * returns the accumulated milliseconds and launch count (optionally resetting them). */
void smgpu_profile_enable(bool on);
void smgpu_profile_read(int32_t kind, double *ms, uint64_t *launches, bool reset);
/* integer-pipe microbenchmark: thread-instructions per second of a dependent-chain kernel
 * (mode 0 = IMAD only, 1 = LOP3/SHF only, 2 = both interleaved) -- the measured roofline
 * denominator of the sketch kernel */
double smgpu_int_peak(int32_t mode, int32_t iters, int32_t blocks);
/* page-locked host memory for batch buffers (host->device copies from it run at full PCIe rate
 * and overlap with the kernels) */
void *smgpu_alloc_pinned(uintptr_t bytes);
void smgpu_free_pinned(void *ptr);
/* frees what kmerminhash_get_mins / kmerminhash_get_abunds returned (reference: leaked, ffi.rs:97-122) */
void kmerminhash_slice_free(const uint64_t *ptr);

/* ---- names and results the crate has but src/ffi.rs does not export ---------------------------------- */
/* north_star's names: jaccard = KmerMinHash::compare (src/lib.rs:501-508);
 * containment = |ptr n other| / |ptr|, the sketch `ptr` in the role of the node of
 * Leaf::containment (src/index.rs:146-160; 0/0 = NaN).  Errors as kmerminhash_compare / _count_common. */
double kmerminhash_jaccard(KmerMinHash *ptr, const KmerMinHash *other);
double kmerminhash_containment(KmerMinHash *ptr, const KmerMinHash *other);
/* KmerMinHash::intersection (src/lib.rs:438-468): the hashes common to both sketches that are also among
 * combined = bottom_num(ptr u other), ascending; *n_common = how many, *size (nullable) = |combined|.
 * (kmerminhash_intersection, src/ffi.rs:292-309, returns only |combined|.)  The returned array is the
 * caller's: kmerminhash_slice_free.  On error: NULL, *n_common untouched. */
const uint64_t *kmerminhash_intersection_hashes(KmerMinHash *ptr, const KmerMinHash *other, uintptr_t *n_common,
                                                uint64_t *size);

/* ---- batch sketching ------------------------------------------------------------------------- */
/* for s in 0..n_seqs: for m in 0..n_mhs: kmerminhash_add_sequence(mhs[m], buf[offsets[s]..offsets[s+1]], force)
 * (src/ffi.rs:55-70 -> src/lib.rs:252-274), sequences NOT NUL-terminated.  n_mhs <= 6, and no sketch may
 * appear twice in mhs (such a call is refused and changes no sketch).
 * With force == false, each sketch keeps the k-mers that precede ITS first invalid k-mer in batch
 * order and SOURMASH_ERROR_CODE_INVALID_D_N_A is recorded.
 * A device `buf` must be 16-byte aligned and readable up to offsets[n_seqs] rounded up to 16. */
void kmerminhash_add_sequences(KmerMinHash *const *mhs, uintptr_t n_mhs, const char *buf /*[host|device]*/,
                               const uint64_t *offsets /*[host|device], n_seqs + 1 */, uint64_t n_seqs,
                               bool force, bool on_device);
/* same for n_reads fixed-length reads stored back to back (no offsets array) */
void kmerminhash_add_reads(KmerMinHash *const *mhs, uintptr_t n_mhs, const char *buf /*[host|device]*/,
                           uint64_t n_reads, uint32_t read_len, bool force, bool on_device);
/* NOT A REFERENCE FORMAT -- an input format of this build only.  The same as kmerminhash_add_reads for reads stored
 * 2 bits per base: A = 0, C = 1, G = 2, T = 3; base i of a read in bits 2*(i % 4) .. 2*(i % 4) + 1 of its byte i / 4;
 * every read starts on a byte boundary ((read_len + 3) / 4 bytes per read, padding bits ignored).  A quarter of the
 * bytes cross PCIe; the device expands them to the ASCII the kernels read, behind the copy.  Results are those of
 * kmerminhash_add_reads over the ASCII form.  (No invalid bases can be expressed, so no error can arise.) */
void kmerminhash_add_reads_2bit(KmerMinHash *const *mhs, uintptr_t n_mhs, const uint8_t *packed /*[host|device]*/,
                                uint64_t n_reads, uint32_t read_len, bool on_device);
/* replace the sketch content: equivalent to a fresh sketch followed by n kmerminhash_mins_push and
 * n_abunds kmerminhash_abunds_push calls (src/ffi.rs:143-150,179-188); abunds may be NULL */
void kmerminhash_set_mins(KmerMinHash *ptr, const uint64_t *mins, uintptr_t n, const uint64_t *abunds,
                          uintptr_t n_abunds);
/* copy the sorted mins (and abundances when `abunds` is non-NULL and tracked) into caller memory
 * of kmerminhash_get_mins_size elements; returns the element count */
uintptr_t kmerminhash_copy_mins(KmerMinHash *ptr, uint64_t *mins /*[host|device]*/,
                                uint64_t *abunds /*[host|device]*/, bool on_device);
/* hex md5 of ksize + mins as stored in the Signature JSON (src/lib.rs:72-77,86) */
SourmashStr kmerminhash_md5sum(KmerMinHash *ptr);

/* ---- sketch collections: packed CSR of sorted u64 hashes in HBM ------------------------------- */
typedef struct SketchCollection SketchCollection;
SketchCollection *smgpu_collection_new(void);
void smgpu_collection_free(SketchCollection *c);
/* append a copy of the sketch's mins as the next row (the sketch must hold sorted, distinct mins) */
void smgpu_collection_push(SketchCollection *c, KmerMinHash *mh);
/* the same for the first sketch of each of n loaded signatures, in one call: the rows a
 * LinearIndex<Leaf<Signature>> holds after `insert` of each (src/index/linear.rs:33-36; a leaf compares through
 * signatures[0], src/index.rs:131-160).  A signature without a sketch is an error, as the reference panics on it. */
void smgpu_collection_push_signatures(SketchCollection *c, Signature *const *sigs, uintptr_t n);
/* adopt a ready CSR: row i = hashes[offsets[i] .. offsets[i+1]); every row sorted ascending and
 * distinct (checked); all rows share (num, ksize, is_protein = false, seed, max_hash) */
SketchCollection *smgpu_collection_from_csr(const uint64_t *hashes /*[host|device]*/,
                                            const uint64_t *offsets /*[host|device], n_rows + 1 */,
                                            uint64_t n_rows, uint32_t num, uint32_t ksize, uint64_t seed,
                                            uint64_t max_hash, bool on_device);
/* One fresh sketch per sequence, pushed in order:
 *   for s in 0..n_seqs { mh = kmerminhash_new(num, ksize, false, seed, max_hash, false);
 *                        kmerminhash_add_sequence(mh, buf[offsets[s]..offsets[s+1]], force = true);
 *                        smgpu_collection_push(c, mh) }
 * (src/lib.rs:142-174, 252-274) -- the sketching half of "sketch N genomes, compare them all" -- in ONE
 * pass over the batch instead of N calls.  Either num > 0 (bottom-num sketches) or max_hash > 0 (scaled);
 * DNA only; invalid k-mers are skipped (force = true).  A device `buf` must be 16-byte aligned and readable
 * up to offsets[n_seqs] rounded up to 16 (the kernel's bulk copies move whole 16-byte groups). */
SketchCollection *smgpu_sketch_collection(const char *buf /*[host|device]*/, const uint64_t *offsets /*[host|device], n_seqs + 1 */,
                                          uint64_t n_seqs, uint32_t num, uint32_t ksize, uint64_t seed, uint64_t max_hash,
                                          bool on_device);
/* One collection per template, each holding one fresh sketch per sequence:
 *   for s in 0..n_seqs: for m in 0..n_templates:
 *     mh = kmerminhash_new(num_m, ksize_m, is_protein_m, seed_m, max_hash_m, false);
 *     kmerminhash_add_sequence(mh, buf[offsets[s]..offsets[s+1]], force = true);
 *     smgpu_collection_push(out[m], mh)
 * in ONE pass over the batch: a host batch crosses PCIe once, DNA templates with distinct k in {21, 31, 51}
 * and one seed share the fused launch of smgpu_fuse_multi_k, and protein templates share one six-frame
 * translation of the batch.  out[m] equals smgpu_sketch_collection with template m's parameters (protein:
 * the rows of per-sequence protein sketches).
 * A template is a KmerMinHash handle of which only num, ksize, is_protein, seed and max_hash are read (its
 * content is neither read nor changed).  1 <= n_templates <= 6; each template has num > 0 or max_hash > 0,
 * not both; DNA ksize 1 to 8192, protein ksize at least 3 (the per-object errors); seeds may differ and a
 * template may appear twice (two equal collections).  A template that tracks abundance is refused:
 * collections hold no abundances.  Input as smgpu_sketch_collection.  out has n_templates entries and
 * receives collections the caller frees; on any error every out[m] is NULL. */
void smgpu_sketch_collections(const char *buf /*[host|device]*/, const uint64_t *offsets /*[host|device], n_seqs + 1 */,
                              uint64_t n_seqs, KmerMinHash *const *templates, uintptr_t n_templates, bool on_device,
                              SketchCollection **out /* n_templates, caller frees each */);
uint64_t smgpu_collection_len(SketchCollection *c);
/* copy the packed rows to the host: hashes (capacity = the returned total) and offsets (n_rows + 1);
 * either may be NULL (call once with NULLs for the size) */
uint64_t smgpu_collection_copy(SketchCollection *c, uint64_t *hashes, uint64_t *offsets);
/* device pointers of the packed arrays (valid until the collection is modified or freed) and the
 * total number of hashes -- what a multi-GPU caller all-gathers */
uint64_t smgpu_collection_csr(SketchCollection *c, const uint64_t **hashes_dev, const uint64_t **offsets_dev);

/* Block [r0, r0+nr) x [c0, c0+nc) of the all-vs-all matrix, element (i, j) at out[(i-r0)*ld + (j-c0)].
 * mode 0: rows[i].compare(cols[j])  -- common = |A n B n bottom_num(A u B)|, size = |bottom_num(A u B)|,
 *         ratio = common / max(1, size)                       (src/lib.rs:470-508)
 * mode 1: Leaf containment with the ROW as the node -- common = |A n B|, size = |A|, ratio = common/size
 *         (src/index.rs:146-160; 0/0 = NaN)
 * Any of common / size / ratio may be NULL.  Incompatible collections record the same error as
 * kmerminhash_compare (src/lib.rs:176-190) and write nothing. */
void smgpu_compare_matrix(SketchCollection *rows, uint64_t r0, uint64_t nr, SketchCollection *cols, uint64_t c0,
                          uint64_t nc, int32_t mode, uint32_t *common /*[host|device]*/,
                          uint32_t *size /*[host|device]*/, double *ratio /*[host|device]*/, uint64_t ld,
                          bool out_on_device);
/* The leaf-pairing pass of `scaffold` (src/index/sbt.rs:356-381): repeatedly take the LAST remaining
 * row, pair it with the first remaining row that has the strictly largest count_common with it
 * (the first remaining row when all counts are 0), remove both.  pairs_first[p] / pairs_second[p]
 * (host, capacity (n + 1) / 2) receive the row ids of pair p in processing order; pairs_second is
 * UINT64_MAX for an unpaired last row.  Returns the number of pairs.  The N x N count_common
 * matrix behind it is one smgpu_compare_matrix(mode 1) block. */
uint64_t smgpu_scaffold_pairs(SketchCollection *c, uint64_t *pairs_first, uint64_t *pairs_second);
/* How smgpu_compare_matrix / smgpu_linear_find walk a block: 0 (default) decides from the data --
 * a hash table over the smaller side of the block (a row shard of an all-vs-all matrix: its own
 * rows, so the shard costs its share of the rows) finds the pairs that share at least one hash,
 * and only those are walked; when the first such block over a row collection finds the
 * (pair, shared hash) incidences many against the dense work, later blocks over those rows go
 * to the dense kernels.  1 forces the dense kernels, 2 forces the hash-table path wherever the
 * block fits it (a build side below 2^31 hashes).  Any other value selects 0.  Results are
 * identical. */
void smgpu_compare_path(int32_t path);
/* How smgpu_linear_find counts shared hashes when a count decides the hit (containment; similarity of sketches
 * without a num): 0 (default) = an index that is large against the query batch is STREAMED once past per-slice
 * Bloom filters of the query hashes held in shared memory (the search then runs at the rate HBM delivers the
 * index), anything smaller goes through the join of smgpu_compare_matrix; 1 = always the join; 2 = stream whenever
 * the shapes allow it; 3 = as 2 with a tiny buffer for the deferred lookups, which exercises the re-run of a
 * block whose hits overflow it (tests).  Results are identical. */
void smgpu_find_path(int32_t path);
/* Batch sketching of several k-sizes over the same sequences (smgpu_add_* with more than one
 * handle, smgpu_sketch_collections with more than one template): on (default) = sketches with
 * distinct k in {21, 31, 51} and one seed share a fused launch that stages each tile of bases once;
 * off = one launch per sketch or template.  Results are identical. */
void smgpu_fuse_multi_k(bool on);
/* LinearIndex::find (src/index/linear.rs:25-45) for every row of `queries` against `index`:
 * mode 0 = search_minhashes (node.similarity(query) > threshold), mode 1 =
 * search_minhashes_containment (node.containment(query) > threshold) (src/index/search.rs:3-9).
 * hit_offsets (n_queries + 1, host) receives the CSR offsets of the per-query hit lists; hits
 * (host, capacity hits_cap) the index row ids in insertion order.  Returns the total number of
 * hits (which may exceed hits_cap: only the first hits_cap are stored). */
uint64_t smgpu_linear_find(SketchCollection *index, SketchCollection *queries, int32_t mode, double threshold,
                           uint64_t *hit_offsets, uint64_t *hits, uint64_t hits_cap);

/* ---- multi-GPU: one process per GPU, the exchange steps over NCCL inside the library ------------------------
 * The reference is single-process (SURVEY 5); what shards is algebra (SURVEY 8(e)): partial sketches combine by
 * KmerMinHash::merge, matrix rows are independent, a partitioned LinearIndex concatenates its parts' hits.
 * NCCL is bound at run time (libnccl.so.2; the copy the host program already loaded, if any).  The 128-byte id
 * is made on one rank and handed to the others by the host program's own channel (MPI_Bcast, a file, ...);
 * every function below marked "collective" must be called by all ranks, in the same order.  Without a
 * communicator the collectives act as in a world of one rank (and NCCL is never loaded). */
#define SMGPU_COMM_ID_BYTES 128
void smgpu_comm_unique_id(uint8_t *id128);                                   /* ncclGetUniqueId */
void smgpu_comm_init(const uint8_t *id128, int32_t rank, int32_t world);     /* collective; after smgpu_set_device */
void smgpu_comm_destroy(void);
int32_t smgpu_comm_rank(void);
int32_t smgpu_comm_world(void);
int32_t smgpu_comm_nccl_version(void);
/* collective: a new collection holding every rank's rows in rank order (rank 0's rows first).  Each rank has
 * checked its own rows (sorted, distinct) when it built `local`; the gathered rows are not checked again. */
SketchCollection *smgpu_collection_allgather(SketchCollection *local);
/* collective: this rank's row block of the all-vs-all matrix -- rows of `local` x the rows of ALL ranks -- as
 * smgpu_compare_matrix(local, 0, n_local, all, 0, n_all, ...) would give it, where all =
 * smgpu_collection_allgather(local), which is also what is returned (caller frees).  The hash table of the join is
 * built over the local rows while the other ranks' rows are in flight over NVLink. */
SketchCollection *smgpu_compare_matrix_allgather(SketchCollection *local, int32_t mode, uint32_t *common /*[host|device]*/,
                                                 uint32_t *size /*[host|device]*/, double *ratio /*[host|device]*/,
                                                 uint64_t ld, bool out_on_device);
/* collective: every rank holds a partial sketch of one sample (its share of the reads); afterwards every rank
 * holds  s_0.merge(s_1).merge(s_2)...  (src/lib.rs:307-403: set union, abundances summed), s_r = rank r's sketch */
void smgpu_comm_allmerge(KmerMinHash *ptr);
/* collective: smgpu_linear_find over an index partitioned by rank (rank r's rows follow those of ranks < r; the
 * query batch is the same on every rank).  Every rank receives the hit lists of the whole index, ids global, in
 * insertion order (src/index/linear.rs:34-44). */
uint64_t smgpu_linear_find_sharded(SketchCollection *index_part, SketchCollection *queries, int32_t mode, double threshold,
                                   uint64_t *hit_offsets, uint64_t *hits, uint64_t hits_cap);

/* ---- Nodegraph (khmer bloom filter) and SBT search: src/index/nodegraph.rs, src/index/sbt.rs ------ */
/* The reference keeps these behind its Rust API only (no extern "C" in src/ffi.rs); the functions
 * below give them the same C-ABI shape as the rest of this header.  Bitsets live in HBM. */
typedef struct Nodegraph Nodegraph;
/* Nodegraph::new(tablesizes, ksize) (nodegraph.rs:20-32); at most 255 tables */
Nodegraph *smgpu_nodegraph_new(const uint64_t *tablesizes, uintptr_t n_tables, uint64_t ksize);
void smgpu_nodegraph_free(Nodegraph *ng);
/* Nodegraph::from_reader over a khmer "OXLI" version-4 Nodegraph file image (nodegraph.rs:135-181);
 * a failed assertion / short read records a Panic error */
Nodegraph *smgpu_nodegraph_from_buffer(const uint8_t *data, uintptr_t len);
/* Nodegraph::save_to_writer (nodegraph.rs:99-133): returns the number of bytes of the file image and
 * writes it when cap is large enough */
uintptr_t smgpu_nodegraph_save(Nodegraph *ng, uint8_t *out, uintptr_t cap);
/* for i in 0..n: is_new[i] = ng.count(hashes[i]) (nodegraph.rs:34-50), in that order -- a bin set by an
 * earlier hash of the batch is not new for a later one.  Returns the number of new k-mers;
 * is_new may be NULL. */
uint64_t smgpu_nodegraph_count_many(Nodegraph *ng, const uint64_t *hashes /*[host|device]*/, uint64_t n,
                                    uint8_t *is_new /*[host|device]*/, bool on_device);
/* sum over i of ng.get(hashes[i]) (nodegraph.rs:52-60); present[i] = that value, may be NULL */
uint64_t smgpu_nodegraph_get_many(Nodegraph *ng, const uint64_t *hashes /*[host|device]*/, uint64_t n,
                                  uint8_t *present /*[host|device]*/, bool on_device);
/* sum of ng.get(h) over the sketch's mins: the numerator of Node<Nodegraph> x Leaf<Signature>
 * similarity / containment (sbt.rs:245,266) */
uint64_t smgpu_nodegraph_matches(Nodegraph *ng, KmerMinHash *mh);
/* Nodegraph::update (nodegraph.rs:63-91): ng |= other, table by table */
void smgpu_nodegraph_update(Nodegraph *ng, Nodegraph *other);
/* Nodegraph::similarity / containment (nodegraph.rs:199-224) */
double smgpu_nodegraph_similarity(Nodegraph *ng, Nodegraph *other);
double smgpu_nodegraph_containment(Nodegraph *ng, Nodegraph *other);
/* tablesizes() into out (capacity cap); returns the number of tables */
uintptr_t smgpu_nodegraph_tablesizes(Nodegraph *ng, uint64_t *out, uintptr_t cap);
uint64_t smgpu_nodegraph_ksize(Nodegraph *ng);
uint64_t smgpu_nodegraph_n_occupied_bins(Nodegraph *ng);
uint64_t smgpu_nodegraph_unique_kmers(Nodegraph *ng);
/* SBT::find (sbt.rs:147-175) for every row of `queries`, with search_minhashes (mode 0) or
 * search_minhashes_containment (mode 1) (search.rs:3-9).  The tree is given by position (root 0,
 * children of p at d*p+1 .. d*p+d): internal node i sits at node_positions[i] with bloom filter
 * nodes[i] and metadata min_n_below[i]; leaf i (row i of `leaves`) at leaf_positions[i].
 * Internal nodes compare as sbt.rs:233-277 (matches / min_n_below, matches / |query|), leaves as
 * index.rs:131-160.  hit_offsets (n_queries + 1, host) / hits (host, capacity hits_cap) receive, per
 * query, the POSITIONS of the matching leaves in the order the reference's depth-first walk
 * reaches them.  Returns the total number of hits. */
uint64_t smgpu_sbt_find(uint32_t d, const uint64_t *node_positions, Nodegraph *const *nodes, const uint64_t *min_n_below,
                        uint64_t n_nodes, const uint64_t *leaf_positions, SketchCollection *leaves,
                        SketchCollection *queries, int32_t mode, double threshold, uint64_t *hit_offsets, uint64_t *hits,
                        uint64_t hits_cap);

#ifdef __cplusplus
}
#endif
#endif /* SOURMASH_B200_EXT_H */
