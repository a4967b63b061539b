// SketchCollection -- many sketches packed as one CSR array of sorted u64 hashes in HBM: the
// operand layout of the all-vs-all compare and linear-search kernels (compare.cu).
// Replaces, for whole collections, the reference's Vec<Leaf<Signature>> walked pair by pair
// (src/index/linear.rs:25-45, src/index.rs:131-160).
#pragma once
#include <memory>
#include <vector>

#include "minhash.hpp"

namespace smb200 {

struct SketchCollection {
    // parameters every row shares (checked on push; compared by check_compatible)
    bool have_params = false;
    uint32_t ksize = 0;
    bool is_protein = false;
    uint64_t seed = 0, max_hash = 0;
    // rows pushed one sketch at a time are staged on the host and uploaded on first use
    std::vector<uint64_t> h_hashes;
    std::vector<uint64_t> h_offsets{0};
    std::vector<uint32_t> h_nums;
    bool dirty = false;
    // device CSR
    DevBuf d_hashes, d_offsets, d_nums;
    uint64_t n_rows = 0, n_hashes = 0;
    uint32_t max_len = 0;
    // compare path bookkeeping (collection.cu): has a block with these rows gone through the probe form of
    // the join yet, and did it find so many incidences that the dense kernels are the better choice
    bool probe_checked = false, probe_dense_preferred = false;
    // find_stream.cu: where each (sorted) row meets each of n_parts equal slices of the hash range [0, part_top];
    // built on the first large search over this collection, kept until it changes
    DevBuf d_part_off;
    uint32_t n_parts = 0;
    uint64_t part_top = 0, part_scale = 0;
    bool parts_valid = false;
    void ensure_partitions();
    std::mutex mu;      // as KmerMinHash::mu
    StreamOwner owner;  // thread context that last queued work on the device arrays (finalize() re-homes)

    void push(KmerMinHash &mh);
    static SketchCollection *from_csr(const uint64_t *hashes, const uint64_t *offsets, uint64_t n_rows, uint32_t num,
                                      uint32_t ksize, uint64_t seed, uint64_t max_hash, bool on_device);
    void finalize();  // upload staged rows
    void check_compatible(const SketchCollection &other) const;  // lib.rs:176-190
    bool uniform_num(uint64_t first, uint64_t n) const;          // rows [first, first + n) share one `num`
};

// one fresh sketch per sequence of the batch, in one pass (sketch_many.cu); see include/sourmash_b200.h
SketchCollection *sketch_collection(const uint8_t *buf, const uint64_t *offsets, uint64_t n_seqs, uint32_t num, uint32_t ksize,
                                    uint64_t seed, uint64_t max_hash, bool on_device);
// the same for 1 to 6 parameter sets over one batch: one collection per entry of ps, in that order
std::vector<std::unique_ptr<SketchCollection>> sketch_collections(const uint8_t *buf, const uint64_t *offsets, uint64_t n_seqs,
                                                                  const std::vector<SketchParams> &ps, bool on_device);

// see collection.cu: join_table_build
struct JoinTable {
    bool valid = false;
    uint64_t ctx_id = 0;
    const uint64_t *bh = nullptr, *bo = nullptr;
    uint64_t b0 = 0, n_build = 0, n_bp = 0;
    int log2_t = 0, log2_f = 0;
    bool has_filter = false;
};
void join_table_build(Context &ctx, JoinTable &jt, const uint64_t *bh, const uint64_t *bo, uint64_t b0, uint64_t n_build,
                      uint64_t n_bp, bool with_filter, cudaStream_t side = nullptr, cudaEvent_t side_go = nullptr);
// one block of the matrix into device outputs (common / size / ratio may be null).  `cols_ready` (optional): the column
// hashes are in device memory once this event has passed on the calling thread's stream (null: they already are); their
// offsets and nums are valid from the start (a gathered collection still in flight, comm.cu).
void compare_block_device(SketchCollection &rows, uint64_t r0, uint64_t nr, SketchCollection &cols, uint64_t c0, uint64_t nc,
                          int mode, uint32_t *common, uint32_t *size, double *ratio, uint64_t ld,
                          const JoinTable *prebuilt = nullptr, cudaEvent_t cols_ready = nullptr);

extern int g_compare_path;
extern int g_find_path;
// see collection.cu
bool probe_form_allowed(const SketchCollection &rows);
// see include/sourmash_b200.h
void compare_matrix(SketchCollection &rows, uint64_t r0, uint64_t nr, SketchCollection &cols, uint64_t c0, uint64_t nc,
                    int mode, uint32_t *common, uint32_t *size, double *ratio, uint64_t ld, bool out_on_device);
uint64_t scaffold_pairs(SketchCollection &c, uint64_t *pairs_first, uint64_t *pairs_second);
// per query: the index row ids that hit, ascending (= insertion order)
std::vector<std::vector<uint64_t>> linear_find_lists(SketchCollection &index, SketchCollection &queries, int mode, double threshold);
uint64_t linear_find(SketchCollection &index, SketchCollection &queries, int mode, double threshold,
                     uint64_t *hit_offsets, uint64_t *hits, uint64_t hits_cap);

}  // namespace smb200
