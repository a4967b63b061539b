// KmerMinHash -- host-side mirror of the reference's sketch type (src/lib.rs:37-513), with
// the same method names, argument meaning and error behaviour, whose state lives in HBM and
// whose work runs as CUDA kernels (sketch.cu / sortops.cu / compare.cu).
//
// There is no CPU implementation of the sketching or comparison arithmetic in this class:
// if no CUDA device is usable every operation throws SourmashError(Internal).  The only host
// arithmetic is the scalar MurmurHash3 of a single word (add_word / hash_murmur), which is a
// scalar call in the reference ABI as well.
#pragma once
#include <stdint.h>

#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "device.hpp"

namespace smb200 {

// add_sequences: share one fused launch among the fast-path k-sizes of a batch (smgpu_fuse_multi_k)
extern bool g_fuse_multi_k;
// host batches are copied to the device in chunks of this size, overlapped with the kernels (minhash.cu)
extern uint64_t g_h2d_chunk_bytes;

// what KmerMinHash::new takes apart from track_abundance
struct SketchParams {
    uint32_t num, ksize;
    bool is_protein;
    uint64_t seed, max_hash;
};
// Several sketches over one batch: those that share one fused launch (sketch.cu) -- with g_fuse_multi_k on, DNA
// sketches of distinct fast-path k-sizes and the seed of the first of them, at most three -- in ascending k.
// Empty unless at least two qualify.
std::vector<int> fused_members(const std::vector<SketchParams> &ps);

// A batch of sequences as the caller holds it (host or device memory).
//   offsets == nullptr && read_len == 0 : one sequence of n_bytes
//   offsets == nullptr && read_len  > 0 : n_seqs reads of read_len bytes, back to back
//   offsets != nullptr                  : n_seqs + 1 offsets into buf (same memory space as buf)
struct SeqBatch {
    const uint8_t *buf = nullptr;
    const uint64_t *offsets = nullptr;
    uint64_t n_seqs = 0;
    uint32_t read_len = 0;
    uint64_t n_bytes = 0;
    bool on_device = false;
    // NON-REFERENCE input format (kmerminhash_add_reads_2bit): fixed-length reads, 2 bits per base (A=0 C=1 G=2 T=3;
    // base i of a read in bits 2*(i%4).. of its byte i/4; every read starts on a byte boundary).  When set, `buf` is
    // unused and n_bytes = n_seqs * read_len is the size of the ASCII form the device expands it into.
    const uint8_t *packed2 = nullptr;
};

// Host-side stage of deferred add_sequence calls (minhash.cu, "deferral of short sequences"): the bytes of the
// sequences back to back (plain or page-locked memory) and their end offsets.
struct SeqStage {
    uint8_t *p = nullptr;
    size_t n = 0, cap = 0;
    size_t accounted = 0;  // bytes this stage has added to the process-wide total of deferred bytes
    bool pinned = false;
    std::vector<uint64_t> offsets{0};
    SeqStage() = default;
    SeqStage(const SeqStage &) = delete;
    SeqStage &operator=(const SeqStage &) = delete;
    ~SeqStage();
    void grow(size_t len);
    void drop();
};

class KmerMinHash {
  public:
    // fields of the reference struct (lib.rs:37-46); mins/abunds live on the device
    uint32_t num;
    uint32_t ksize;
    bool is_protein;
    uint64_t seed;
    uint64_t max_hash;
    std::mutex mu;  // held by the C ABI around every call that is handed this sketch (ffi.cpp, "Locking")

    // KmerMinHash::new (lib.rs:142-174)
    KmerMinHash(uint32_t num, uint32_t ksize, bool is_protein, uint64_t seed, uint64_t max_hash,
                bool track_abundance);
    // KmerMinHash::default (lib.rs:48-60)
    static KmerMinHash *make_default() { return new KmerMinHash(1000, 21, false, 42, 0, false); }
    KmerMinHash *clone();
    ~KmerMinHash();
    KmerMinHash(const KmerMinHash &) = delete;
    KmerMinHash &operator=(const KmerMinHash &) = delete;

    void check_compatible(const KmerMinHash &other) const;            // lib.rs:176-190
    void add_hash(uint64_t hash);                                      // lib.rs:192-245
    void add_word(const uint8_t *word, size_t len);                    // lib.rs:247-250
    void add_sequence(const uint8_t *seq, size_t len, bool force);     // lib.rs:252-305 (DNA arm)
    void merge(KmerMinHash &other);                                    // lib.rs:307-403
    void add_from(KmerMinHash &other);                                 // lib.rs:405-410
    void add_many(const uint64_t *hashes, size_t n);                   // lib.rs:412-417
    uint64_t count_common(KmerMinHash &other);                         // lib.rs:428-436
    std::pair<uint64_t, uint64_t> intersection_size(KmerMinHash &other);  // lib.rs:470-499
    // the common hashes themselves, ascending, and |combined| (lib.rs:438-468)
    std::pair<std::vector<uint64_t>, uint64_t> intersection(KmerMinHash &other);
    double compare(KmerMinHash &other);                                // lib.rs:501-508
    // Leaf<Signature>::similarity / containment with this sketch as the node (index.rs:131-160)
    double similarity(KmerMinHash &other) { return compare(other); }
    double containment(KmerMinHash &other);
    size_t size();                                                     // lib.rs:510-512

    // ---- batch extension: many add_sequence calls (and several sketches) in one pass --------
    // Equivalent to `for s in batch: for mh in mhs: mh.add_sequence(s, force)`, except that on
    // an invalid k-mer with force == false every sketch keeps what the reference would have added
    // up to ITS first failing k-mer and the error of the first failing sketch is thrown.
    static void add_sequences(KmerMinHash *const *mhs, int n_mhs, const SeqBatch &batch, bool force);

    // ---- raw state access (ffi.rs:97-188) ----------------------------------------------------
    bool track_abundance() const { return has_abunds_; }
    const std::vector<uint64_t> &mins();     // host copy (synchronises)
    const std::vector<uint64_t> &abunds();   // host copy (empty when not tracking)
    void mins_push(uint64_t v);              // raw append, bypasses ordering (ffi.rs:143-150)
    void abunds_push(uint64_t v);            // ffi.rs:179-188
    // device view (flushes pending work); valid until the next mutating call
    const uint64_t *device_mins(size_t *n);
    const uint64_t *device_abunds(size_t *n);
    void set_from_host(const uint64_t *mins, size_t n, const uint64_t *abunds, size_t n_abunds);
    void take_state_of(KmerMinHash &other);  // mins / abundances (and whether they are tracked) move over; parameters must match
    std::string md5sum();                    // lib.rs:72-77,86
    bool equals(KmerMinHash &other);         // derived PartialEq (lib.rs:37)

  private:
    bool has_abunds_;
    // canonical state on the device (valid when dev_valid_)
    DevBuf d_mins_, d_abunds_;
    DevBuf d_mins_alt_, d_abunds_alt_;  // output side of the next merge (swapped in by commit)
    size_t n_mins_ = 0, n_abunds_ = 0;
    // host mirror (valid when host_valid_)
    std::vector<uint64_t> h_mins_, h_abunds_;
    bool host_valid_ = true, dev_valid_ = true;
    // strict ascending order of mins: 1 yes, 0 no, -1 unknown (raw pushes)
    int sorted_ = 1;
    // add_hash events not yet ingested (stream order)
    std::vector<uint64_t> pending_;
    // small sequences of add_sequence calls not yet sketched (host side, call order; see add_sequence).  At most
    // one of pending_ / seq_stage_ is non-empty at any time, so call order between the two kinds is kept.
    SeqStage seq_stage_;
    void flush_sequences(bool stage_full = false);
    // survivors of the sketch kernel not yet merged into the state (scaled sketches merge lazily)
    DevBuf d_cand_hash_, d_cand_pos_;
    uint64_t n_cand_ = 0;
    // per-handle device scalars: [0] candidate counter, [1] threshold, [2] first failing window
    DevBuf d_hs_;

    StreamOwner owner_;  // thread context that last queued device work on this sketch
    Context &home();

    enum Mode { MODE_SCALED, MODE_NUM, MODE_REPLAY };
    Mode mode() const;
    bool want_pos() const { return mode() == MODE_REPLAY || (mode() == MODE_NUM && has_abunds_); }
    unsigned long long *hs(int i);
    void flush();          // pending_ + candidates -> canonical device state; gives scratch back to the pool
    void flush_pending();
    void ensure_dev();
    void ensure_host();
    void require_sorted(const char *what);
    void reserve_candidates(Context &ctx, uint64_t extra);
    bool ingest(Context &ctx, bool thr_is_estimate, uint64_t thr_value = ~0ull);
    void replay(Context &ctx, const uint64_t *d_events, uint64_t n_events);
    void commit(DevBuf &mins, DevBuf &abunds, size_t n_mins, size_t n_abunds);
};

// add_sequence calls on short valid sequences are collected on the host and sketched as one batch
// (SMB200_DEFER_SEQ=0 switches this off)
extern bool g_defer_small_sequences;

// host scalar hash (ffi.rs:15-24)
uint64_t hash_murmur_host(const uint8_t *kmer, size_t len, uint64_t seed);

}  // namespace smb200
