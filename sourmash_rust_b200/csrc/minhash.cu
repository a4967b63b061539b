// minhash.cu -- KmerMinHash host class: owns the sketch state in HBM and drives the kernels.
//
// How the reference's per-hash state machine (add_hash, src/lib.rs:192-245) is reproduced for a
// whole batch of hashes at once:
//   scaled sketch (num == 0, max_hash > 0): the result is the set of distinct hashes <= max_hash
//       with their occurrence counts -- order independent.  Survivors of the sketch kernel are
//       appended to a per-sketch candidate list and folded into the sorted state lazily
//       (concatenate + radix sort + run-length reduce).
//   num sketch (num > 0, max_hash == 0): the result is the `num` smallest distinct hashes.
//       The kernel filters with a threshold (the current largest element once the sketch is full,
//       otherwise an estimate that is verified and widened if it kept too few), then the same
//       sort/reduce and a truncation.  With abundance tracking the reference does NOT count
//       re-occurrences of the largest element of a full sketch (lib.rs:206-208); that is restored
//       exactly from first-occurrence positions (see ingest()).
//   any other combination (both set, or neither): order dependent in the reference, so the
//       survivors are replayed in stream order by a single-CTA kernel (launch_replay_add_hash).
#include "minhash.hpp"

#include <atomic>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "kernels.cuh"
#include "md5.hpp"
#include "murmur3.cuh"

namespace smb200 {

bool g_fuse_multi_k = true;
static uint64_t h2d_chunk_from_env() {
    const char *e = getenv("SMB200_H2D_CHUNK_MB");
    uint64_t mb = e ? strtoull(e, nullptr, 10) : 8;
    return (mb ? mb : 1) << 20;
}
uint64_t g_h2d_chunk_bytes = h2d_chunk_from_env();  // SMB200_H2D_CHUNK_MB overrides the 8 MiB default

static const uint64_t U64_MAX = ~0ull;
static const uint64_t LAZY_CANDIDATES = 1ull << 22;  // scaled sketches fold their candidates in past this

uint64_t hash_murmur_host(const uint8_t *kmer, size_t len, uint64_t seed) {
    return murmur3_h1_bytes(kmer, (uint64_t)len, seed);
}

// small device helpers ------------------------------------------------------------------------
__global__ void set_u64_kernel(unsigned long long *p, unsigned long long v) { *p = v; }
static void set_u64(unsigned long long *p, unsigned long long v, cudaStream_t st) {
    set_u64_kernel<<<1, 1, 0, st>>>(p, v);
    SM_LAUNCHED();
}
// thr = largest kept element when the sketch is full, else `fallback`
__global__ void thr_from_state_kernel(unsigned long long *thr, const uint64_t *mins, uint64_t n_mins, uint32_t num,
                                      unsigned long long fallback) {
    *thr = (num != 0 && n_mins >= num) ? mins[num - 1] : fallback;
}
__global__ void iota_ones_kernel(uint64_t *v, uint64_t n) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) v[i] = 1;
}

// 2-bit packed reads -> ASCII (kmerminhash_add_reads_2bit): 16 output bytes per thread, reads [r0, r1)
__global__ void __launch_bounds__(256) unpack_2bit_kernel(const uint8_t *__restrict__ packed, uint8_t *__restrict__ ascii, uint64_t r0,
                                                          uint64_t r1, uint32_t read_len) {
    const uint32_t bpr = (read_len + 3) / 4;
    const uint64_t o_lo = r0 * read_len, o_hi = r1 * read_len;   // output byte range; o_lo is what the caller aligned to 16
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x * 16;
    for (uint64_t o = (o_lo & ~15ull) + ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16; o < o_hi; o += stride) {
        uint64_t r = o / read_len;
        uint32_t i = (uint32_t)(o - r * read_len);
        uint32_t w[4] = {0, 0, 0, 0};
#pragma unroll
        for (int b = 0; b < 16; b++) {
            const uint64_t ob = o + b;
            uint32_t ch = 0;
            if (ob >= o_lo && ob < o_hi) {
                const uint32_t code = (packed[r * bpr + (i >> 2)] >> (2 * (i & 3))) & 3u;
                ch = (0x54474341u >> (8 * code)) & 0xFFu;   // "ACGT"
            }
            w[b >> 2] |= ch << (8 * (b & 3));
            if (++i == read_len) { i = 0; r++; }
        }
        if (o >= o_lo && o + 16 <= o_hi) {
            *reinterpret_cast<uint4 *>(ascii + o) = make_uint4(w[0], w[1], w[2], w[3]);
        } else {   // a group cut by the range: its bytes one by one (the neighbours belong to another launch)
            for (int b = 0; b < 16; b++)
                if (o + b >= o_lo && o + b < o_hi) ascii[o + b] = (uint8_t)(w[b >> 2] >> (8 * (b & 3)));
        }
    }
}

static int bit_length(uint64_t x) {
    int b = 0;
    while (x) { b++; x >>= 1; }
    return b;
}

// ---------------------------------------------------------------------------------------------
KmerMinHash::KmerMinHash(uint32_t num_, uint32_t ksize_, bool is_protein_, uint64_t seed_, uint64_t max_hash_,
                         bool track_abundance)
    : num(num_), ksize(ksize_), is_protein(is_protein_), seed(seed_), max_hash(max_hash_),
      has_abunds_(track_abundance) {}

// Bytes of deferred add_sequence calls waiting in all sketches together (see "deferral of short sequences" below):
// many live sketches (10^5 genomes, one handle each) must not pile up host memory without bound -- above
// kDeferTotalCap a sketch flushes on every call until others have drained.
static std::atomic<size_t> g_seq_pending_total{0};

KmerMinHash::~KmerMinHash() {}

KmerMinHash *KmerMinHash::clone() {
    flush();
    KmerMinHash *c = new KmerMinHash(num, ksize, is_protein, seed, max_hash, has_abunds_);
    c->sorted_ = sorted_;
    if (host_valid_) {
        c->h_mins_ = h_mins_;
        c->h_abunds_ = h_abunds_;
        c->host_valid_ = true;
        c->dev_valid_ = false;
        c->n_mins_ = h_mins_.size();
        c->n_abunds_ = h_abunds_.size();
    } else {
        Context &ctx = home();
        ctx.adopt(c->owner_);
        c->d_mins_.reserve((n_mins_ + 1) * 8);
        c->d_abunds_.reserve((n_abunds_ + 1) * 8);
        if (n_mins_) SM_CUDA(cudaMemcpyAsync(c->d_mins_.p, d_mins_.p, n_mins_ * 8, cudaMemcpyDeviceToDevice, ctx.stream));
        if (n_abunds_) SM_CUDA(cudaMemcpyAsync(c->d_abunds_.p, d_abunds_.p, n_abunds_ * 8, cudaMemcpyDeviceToDevice, ctx.stream));
        ctx.sync();
        c->n_mins_ = n_mins_;
        c->n_abunds_ = n_abunds_;
        c->host_valid_ = false;
        c->dev_valid_ = true;
    }
    return c;
}

// This thread's context, after waiting for whatever another thread may have left queued on this sketch.
Context &KmerMinHash::home() {
    Context &c = Context::get();
    c.adopt(owner_);
    return c;
}

KmerMinHash::Mode KmerMinHash::mode() const {
    if (num == 0 && max_hash != 0) return MODE_SCALED;
    if (num != 0 && max_hash == 0) return MODE_NUM;
    return MODE_REPLAY;
}

unsigned long long *KmerMinHash::hs(int i) {
    if (!d_hs_.p) {
        d_hs_.reserve(64);
        SM_CUDA(cudaMemsetAsync(d_hs_.p, 0, 64, home().stream));
    }
    return d_hs_.as<unsigned long long>() + i;
}

void KmerMinHash::check_compatible(const KmerMinHash &other) const {
    if (ksize != other.ksize) throw SourmashError(ERR_MISMATCH_KSIZES, "different ksizes cannot be compared");
    if (is_protein != other.is_protein) throw SourmashError(ERR_MISMATCH_DNAPROT, "DNA/prot minhashes cannot be compared");
    if (max_hash != other.max_hash) throw SourmashError(ERR_MISMATCH_MAXHASH, "mismatch in max_hash; comparison fail");
    if (seed != other.seed) throw SourmashError(ERR_MISMATCH_SEED, "mismatch in seed; comparison fail");
}

// ---- host <-> device mirrors ------------------------------------------------------------------
void KmerMinHash::ensure_dev() {
    Context &ctx = home();
    if (dev_valid_) return;
    n_mins_ = h_mins_.size();
    n_abunds_ = h_abunds_.size();
    d_mins_.reserve((n_mins_ + 1) * 8);
    d_abunds_.reserve((n_abunds_ + 1) * 8);
    if (n_mins_) SM_CUDA(cudaMemcpyAsync(d_mins_.p, h_mins_.data(), n_mins_ * 8, cudaMemcpyHostToDevice, ctx.stream));
    if (n_abunds_) SM_CUDA(cudaMemcpyAsync(d_abunds_.p, h_abunds_.data(), n_abunds_ * 8, cudaMemcpyHostToDevice, ctx.stream));
    ctx.sync();
    dev_valid_ = true;
}

void KmerMinHash::ensure_host() {
    flush();
    if (host_valid_) return;
    Context &ctx = home();
    h_mins_.resize(n_mins_);
    h_abunds_.resize(n_abunds_);
    if (n_mins_) SM_CUDA(cudaMemcpyAsync(h_mins_.data(), d_mins_.p, n_mins_ * 8, cudaMemcpyDeviceToHost, ctx.stream));
    if (n_abunds_) SM_CUDA(cudaMemcpyAsync(h_abunds_.data(), d_abunds_.p, n_abunds_ * 8, cudaMemcpyDeviceToHost, ctx.stream));
    ctx.sync();
    host_valid_ = true;
}

void KmerMinHash::require_sorted(const char *what) {
    if (sorted_ == 1) return;
    ensure_dev();
    if (sorted_ == -1) {
        Context &ctx = home();
        set_u64(ctx.dsc(SC_FLAG), 0, ctx.stream);
        launch_check_sorted(d_mins_.as<uint64_t>(), n_mins_, ctx.dsc(SC_FLAG), ctx.stream);
        ctx.read_scalars();
        sorted_ = ctx.h_scalars[SC_FLAG] ? 0 : 1;
    }
    if (sorted_ == 0)
        throw_internal(std::string(what) + ": mins are not strictly ascending (raw mins_push of unsorted data); "
                       "the reference's binary search / two-pointer walk is undefined on such input");
}

const std::vector<uint64_t> &KmerMinHash::mins() { ensure_host(); return h_mins_; }
const std::vector<uint64_t> &KmerMinHash::abunds() { ensure_host(); return h_abunds_; }
size_t KmerMinHash::size() { flush(); return dev_valid_ ? n_mins_ : h_mins_.size(); }

void KmerMinHash::mins_push(uint64_t v) {
    ensure_host();
    if (sorted_ == 1 && !h_mins_.empty() && !(h_mins_.back() < v)) sorted_ = -1;
    h_mins_.push_back(v);
    dev_valid_ = false;
}
void KmerMinHash::abunds_push(uint64_t v) {
    if (!has_abunds_) return;  // ffi.rs:179-188: only when tracking
    ensure_host();
    h_abunds_.push_back(v);
    dev_valid_ = false;
}
void KmerMinHash::set_from_host(const uint64_t *mins_in, size_t n, const uint64_t *abunds_in, size_t n_abunds) {
    pending_.clear();
    seq_stage_.drop();
    n_cand_ = 0;
    h_mins_.assign(mins_in, mins_in + n);
    if (abunds_in) h_abunds_.assign(abunds_in, abunds_in + n_abunds); else h_abunds_.clear();
    host_valid_ = true;
    dev_valid_ = false;
    sorted_ = std::is_sorted(h_mins_.begin(), h_mins_.end(), [](uint64_t a, uint64_t b) { return a <= b; }) ? 1 : 0;
    if (n < 2) sorted_ = 1;
}
void KmerMinHash::take_state_of(KmerMinHash &o) {
    check_compatible(o);
    o.flush();
    Context &ctx = home();
    ctx.adopt(o.owner_);
    pending_.clear();
    seq_stage_.drop();
    n_cand_ = 0;
    has_abunds_ = o.has_abunds_;
    std::swap(d_mins_, o.d_mins_);
    std::swap(d_abunds_, o.d_abunds_);
    h_mins_.swap(o.h_mins_);
    h_abunds_.swap(o.h_abunds_);
    n_mins_ = o.n_mins_; n_abunds_ = o.n_abunds_;
    host_valid_ = o.host_valid_; dev_valid_ = o.dev_valid_;
    sorted_ = o.sorted_;
    o.n_mins_ = o.n_abunds_ = 0;
    o.h_mins_.clear(); o.h_abunds_.clear();
    o.host_valid_ = true; o.dev_valid_ = false;
}
const uint64_t *KmerMinHash::device_mins(size_t *n) {
    flush(); ensure_dev();
    *n = n_mins_;
    return d_mins_.as<uint64_t>();
}
const uint64_t *KmerMinHash::device_abunds(size_t *n) {
    flush(); ensure_dev();
    *n = n_abunds_;
    return has_abunds_ ? d_abunds_.as<uint64_t>() : nullptr;
}

std::string KmerMinHash::md5sum() {
    ensure_host();
    Md5 ctx;
    ctx.update(std::to_string(ksize));
    for (uint64_t m : h_mins_) ctx.update(std::to_string(m));
    return ctx.hex();
}

bool KmerMinHash::equals(KmerMinHash &o) {
    ensure_host(); o.ensure_host();
    return num == o.num && ksize == o.ksize && is_protein == o.is_protein && seed == o.seed && max_hash == o.max_hash &&
           h_mins_ == o.h_mins_ && has_abunds_ == o.has_abunds_ && (!has_abunds_ || h_abunds_ == o.h_abunds_);
}

// ---- single-hash entry points -----------------------------------------------------------------
void KmerMinHash::add_hash(uint64_t hash) {
    flush_sequences();  // deferred sequences came first
    pending_.push_back(hash);
}
void KmerMinHash::add_word(const uint8_t *word, size_t len) { add_hash(hash_murmur_host(word, len, seed)); }
void KmerMinHash::add_many(const uint64_t *hashes, size_t n) {
    flush_sequences();
    pending_.insert(pending_.end(), hashes, hashes + n);
}
void KmerMinHash::add_from(KmerMinHash &other) {
    flush_sequences();
    const std::vector<uint64_t> &m = other.mins();
    pending_.insert(pending_.end(), m.begin(), m.end());
}

void KmerMinHash::commit(DevBuf &mins, DevBuf &abunds, size_t n_mins, size_t n_abunds) {
    std::swap(d_mins_, mins);
    if (has_abunds_) std::swap(d_abunds_, abunds);
    n_mins_ = n_mins;
    n_abunds_ = has_abunds_ ? n_abunds : 0;
    dev_valid_ = true;
    host_valid_ = false;
    sorted_ = 1;
}

void KmerMinHash::reserve_candidates(Context &ctx, uint64_t total) {
    const size_t bytes = (size_t)(total + 64) * 8;
    d_cand_hash_.reserve(bytes, ctx.stream, n_cand_ > 0, (size_t)n_cand_ * 8);
    if (want_pos()) d_cand_pos_.reserve(bytes, ctx.stream, n_cand_ > 0, (size_t)n_cand_ * 8);
}

void KmerMinHash::replay(Context &ctx, const uint64_t *d_events, uint64_t n_events) {
    if (!n_events) return;
    ensure_dev();
    require_sorted("add_hash");
    if (has_abunds_ && n_abunds_ != n_mins_) throw_internal("abundances out of step with mins");
    d_mins_.reserve((n_mins_ + n_events + 1) * 8, ctx.stream, true, n_mins_ * 8);
    if (has_abunds_) d_abunds_.reserve((n_mins_ + n_events + 1) * 8, ctx.stream, true, n_abunds_ * 8);
    set_u64(ctx.dsc(SC_LEN), n_mins_, ctx.stream);
    launch_replay_add_hash(d_events, n_events, num, max_hash, d_mins_.as<uint64_t>(),
                           has_abunds_ ? d_abunds_.as<uint64_t>() : nullptr, ctx.dsc(SC_LEN), ctx.stream);
    ctx.read_scalars();
    n_mins_ = ctx.h_scalars[SC_LEN];
    n_abunds_ = has_abunds_ ? n_mins_ : 0;
    host_valid_ = false;
}

// add_hash events buffered on the host -> candidates (or straight replay)
void KmerMinHash::flush_pending() {
    flush_sequences();
    if (pending_.empty()) return;
    Context &ctx = home();
    ensure_dev();
    const uint64_t n = pending_.size();
    ctx.misc[7].reserve((n + 1) * 8);
    uint64_t *d_events = ctx.misc[7].as<uint64_t>();
    SM_CUDA(cudaMemcpyAsync(d_events, pending_.data(), n * 8, cudaMemcpyHostToDevice, ctx.stream));
    ctx.sync();
    std::vector<uint64_t>().swap(pending_);
    if (mode() == MODE_REPLAY) {
        replay(ctx, d_events, n);
        return;
    }
    require_sorted("add_hash");
    if (mode() == MODE_NUM && n_cand_) ingest(ctx, false);
    reserve_candidates(ctx, n_cand_ + n);
    set_u64(hs(0), n_cand_, ctx.stream);
    thr_from_state_kernel<<<1, 1, 0, ctx.stream>>>(hs(1), d_mins_.as<uint64_t>(), n_mins_, num,
                                                   mode() == MODE_SCALED ? max_hash : U64_MAX);
    SM_LAUNCHED();
    // the counter starts at n_cand_, so the survivors land behind the candidates already held
    launch_filter_hashes(d_events, n, max_hash, reinterpret_cast<const uint64_t *>(hs(1)), d_cand_hash_.as<uint64_t>(),
                         want_pos() ? d_cand_pos_.as<uint64_t>() : nullptr, hs(0), ctx.stream);
    SM_CUDA(cudaMemcpyAsync(ctx.h_scalars + SC_CAND0, hs(0), 8, cudaMemcpyDeviceToHost, ctx.stream));
    ctx.sync();
    n_cand_ = ctx.h_scalars[SC_CAND0];
    if (mode() == MODE_NUM || n_cand_ > LAZY_CANDIDATES) ingest(ctx, false);
}

void KmerMinHash::flush() {
    flush_pending();
    if (n_cand_) ingest(home(), false);
    // Many sketches may be alive at once (10^4..10^6): scratch that dwarfs the sketch itself goes back
    // to the stream-ordered pool (the next batch gets it again in microseconds); scratch of the same
    // order as the state stays, so a sketch that is read between batches does not churn.
    const size_t keep = 16 * std::max<size_t>((n_mins_ + n_abunds_) * 8, 16 * 1024);
    if (d_cand_hash_.cap > keep) d_cand_hash_.release();
    if (d_cand_pos_.cap > keep) d_cand_pos_.release();
    if (d_mins_alt_.cap > keep) d_mins_alt_.release();
    if (d_abunds_alt_.cap > keep) d_abunds_alt_.release();
}

// ---------------------------------------------------------------------------------------------
// candidates -> state.  Returns false (nothing committed, candidates dropped) when the threshold
// was an estimate and turned out too tight to fill a num sketch.
// ---------------------------------------------------------------------------------------------
bool KmerMinHash::ingest(Context &ctx, bool thr_is_estimate, uint64_t thr_value) {
    const uint64_t nc = n_cand_;
    n_cand_ = 0;
    if (nc == 0) return !(mode() == MODE_NUM && thr_is_estimate && n_mins_ < num);  // nothing kept: estimate too tight?
    ensure_dev();
    require_sorted("add_hash");
    if (has_abunds_ && n_abunds_ != n_mins_) throw_internal("abundances out of step with mins");
    cudaStream_t st = ctx.stream;
    const Mode m = mode();
    const bool quirk = (m == MODE_NUM && has_abunds_);
    const uint64_t na = n_mins_;
    const int key_bits = (m == MODE_SCALED) ? bit_length(max_hash) : 64;

    uint64_t *cand = d_cand_hash_.as<uint64_t>();
    uint64_t *cpos = d_cand_pos_.as<uint64_t>();
    uint64_t nc_generic = nc;  // candidates the sort-based union below still has to take
    if (m == MODE_SCALED && na > 0) {
        // Fast path: a scaled sketch that has already seen the sample holds nearly every candidate.  Look
        // each one up in the sorted state (abundance += 1 in place); only the hashes that are new go on.
        ctx.misc[6].reserve((nc + 1) * 8);
        uint64_t *news = ctx.misc[6].as<uint64_t>();
        SM_CUDA(cudaMemsetAsync(ctx.dsc(SC_NUNIQ), 0, 8, st));
        launch_fold_match(cand, nc, d_mins_.as<uint64_t>(), na, has_abunds_ ? d_abunds_.as<uint64_t>() : nullptr, news,
                          ctx.dsc(SC_NUNIQ), st);
        ctx.read_scalars();
        const uint64_t n_news = ctx.h_scalars[SC_NUNIQ];
        host_valid_ = false;
        if (n_news == 0) return true;
        if (n_news <= (uint64_t)fold_small_limit()) {
            // few new hashes: one CTA sorts them, then a merge by rank
            ctx.misc[3].reserve((n_news + 1) * 8);
            ctx.misc[4].reserve((n_news + 1) * 8);
            d_mins_alt_.reserve((na + n_news + 1) * 8);
            if (has_abunds_) d_abunds_alt_.reserve((na + n_news + 1) * 8);
            launch_fold_small(news, (uint32_t)n_news, d_mins_.as<uint64_t>(), has_abunds_ ? d_abunds_.as<uint64_t>() : nullptr, na,
                              ctx.misc[3].as<uint64_t>(), ctx.misc[4].as<uint64_t>(), ctx.dsc(SC_NUNIQ),
                              d_mins_alt_.as<uint64_t>(), has_abunds_ ? d_abunds_alt_.as<uint64_t>() : nullptr, st);
            ctx.read_scalars();
            const uint64_t n_out = na + ctx.h_scalars[SC_NUNIQ];
            commit(d_mins_alt_, d_abunds_alt_, n_out, n_out);
            return true;
        }
        // many new hashes: they are the candidates of the generic union (the matched ones are already counted)
        SM_CUDA(cudaMemcpyAsync(cand, news, n_news * 8, cudaMemcpyDeviceToDevice, st));
        nc_generic = n_news;
    }
    const uint64_t n_max = na + nc_generic;
    ctx.sort_tmp_k.reserve((n_max + 1) * 8);
    ctx.sort_tmp_v.reserve((n_max + 1) * 8);
    ctx.scan_tmp.reserve(std::max(radix_sort_scan_bytes(n_max), scan_tmp_bytes(n_max)) + 256);
    for (int i = 0; i < 6; i++) ctx.misc[i].reserve((n_max + 1) * 8);
    uint64_t *cat_k = ctx.misc[0].as<uint64_t>(), *cat_v = ctx.misc[1].as<uint64_t>();
    uint64_t *idx = ctx.misc[2].as<uint64_t>();
    uint64_t *ukeys = ctx.misc[3].as<uint64_t>(), *ucnt = ctx.misc[4].as<uint64_t>(), *ufirst = ctx.misc[5].as<uint64_t>();

    // second operand of the union: the candidates themselves, or (quirk) their run-length form
    const uint64_t *b_keys = cand;
    const uint64_t *b_vals = nullptr;  // nullptr = every entry counts 1
    uint64_t nb = nc_generic;
    if (quirk) {
        radix_sort_pairs(cand, cpos, nc, ctx.sort_tmp_k.as<uint64_t>(), ctx.sort_tmp_v.as<uint64_t>(), key_bits,
                         ctx.scan_tmp.p, ctx.scan_tmp.cap, st);
        reduce_by_key(cand, nullptr, nc, ukeys, ucnt, ctx.dsc(SC_NUNIQ), idx, ctx.scan_tmp.p, st);
        launch_fill_u64(ufirst, U64_MAX, nc, st);
        min_by_key(cand, cpos, nc, idx, ufirst, st);
        ctx.read_scalars();
        nb = ctx.h_scalars[SC_NUNIQ];
        b_keys = ukeys;
        b_vals = ucnt;
    }
    // concatenate state and second operand
    const uint64_t n_cat = na + nb;
    if (na) SM_CUDA(cudaMemcpyAsync(cat_k, d_mins_.p, na * 8, cudaMemcpyDeviceToDevice, st));
    SM_CUDA(cudaMemcpyAsync(cat_k + na, b_keys, nb * 8, cudaMemcpyDeviceToDevice, st));
    if (has_abunds_) {
        if (na) SM_CUDA(cudaMemcpyAsync(cat_v, d_abunds_.p, na * 8, cudaMemcpyDeviceToDevice, st));
        if (b_vals) SM_CUDA(cudaMemcpyAsync(cat_v + na, b_vals, nb * 8, cudaMemcpyDeviceToDevice, st));
        else {
            iota_ones_kernel<<<(unsigned)std::min<uint64_t>((nb + 255) / 256, 148 * 16), 256, 0, st>>>(cat_v + na, nb);
            SM_LAUNCHED();
        }
    }
    radix_sort_pairs(cat_k, has_abunds_ ? cat_v : nullptr, n_cat, ctx.sort_tmp_k.as<uint64_t>(),
                     ctx.sort_tmp_v.as<uint64_t>(), key_bits, ctx.scan_tmp.p, ctx.scan_tmp.cap, st);
    DevBuf &out_k = d_mins_alt_, &out_v = d_abunds_alt_;
    out_k.reserve((n_cat + 1) * 8);
    out_v.reserve((n_cat + 1) * 8);
    uint64_t *idx2 = quirk ? ctx.sort_tmp_k.as<uint64_t>() : idx;  // idx still holds the candidates' run ids
    reduce_by_key(cat_k, has_abunds_ ? cat_v : nullptr, n_cat, out_k.as<uint64_t>(), out_v.as<uint64_t>(),
                  ctx.dsc(SC_NUNIQ), idx2, ctx.scan_tmp.p, st);
    ctx.read_scalars();
    const uint64_t n_new = ctx.h_scalars[SC_NUNIQ];
    if (m == MODE_NUM && thr_is_estimate) {
        // The kernel kept only the batch's hashes <= thr_value.  The union is the true bottom-num exactly when its
        // num-th smallest element is <= thr_value: every hash that was filtered away is larger than that.  Counting
        // distinct elements alone is not enough -- elements of the OLD state above the estimate count too, and
        // would hide batch hashes between the estimate and them.
        if (n_new < num) return false;
        uint64_t kth[2];
        ctx.fetch2(out_k.as<uint64_t>() + (num - 1), out_k.as<uint64_t>() + (num - 1), kth);
        if (kth[0] > thr_value) return false;
    }
    const uint64_t n_keep = (num != 0 && n_new > num) ? num : n_new;
    if (quirk && n_new >= num) {
        // lib.rs:206-208: once the sketch is full, re-occurrences of its largest element X are
        // ignored.  X's count = occurrences up to the moment T the last of the final elements
        // first appeared (elements already in the old state appeared "before" this batch).
        const uint64_t *x_ptr = out_k.as<uint64_t>() + (num - 1);
        set_u64(ctx.dsc(SC_TMAX), 0, st);
        set_u64(ctx.dsc(SC_CNT), 0, st);
        launch_first_new_max(ukeys, ufirst, nb, d_mins_.as<uint64_t>(), na, x_ptr, ctx.dsc(SC_TMAX), st);
        launch_count_key_upto(cand, cpos, nc, x_ptr, ctx.dsc(SC_TMAX), ctx.dsc(SC_CNT), st);
        launch_fix_max_abund(out_v.as<uint64_t>() + (num - 1), ukeys, ucnt, nb, x_ptr, ctx.dsc(SC_CNT), st);
        ctx.sync();
    }
    commit(out_k, out_v, n_keep, n_keep);
    return true;
}

// ---------------------------------------------------------------------------------------------
// add_sequence / add_sequences
// ---------------------------------------------------------------------------------------------
// ---- deferral of short sequences ---------------------------------------------------------------------------
// A caller of the unmodified reference ABI feeds reads one call at a time (150 bp per call in BASELINE cfg2,
// ffi.rs:55-70); going to the device per call costs 45 us whatever the length.  A short sequence that cannot raise
// an error -- only ACGT/acgt, or force == true (invalid windows are skipped, lib.rs:268-273) -- is therefore
// appended to a host-side stage and the call returns; the stage goes through add_sequences (which keeps
// per-sequence order semantics) when it reaches kDeferFlushBytes or when anything reads, combines or otherwise
// touches the sketch (flush_pending() is the gate).  A sequence that CAN raise InvalidDNA takes the synchronous
// path below -- after the deferred ones, in call order -- so the error, and the partial mutation before it,
// belong to the call that caused them.  Every staged sequence is known to be free of errors, so the stage is
// sketched with force = true whatever flags its calls carried.
//
// The stage starts as ordinary host memory and grows geometrically; a sketch that keeps streaming (past
// kStagePinAt bytes) moves to a page-locked buffer from a small process-wide pool, so that its flushes copy at
// PCIe rate, and gives it back when a read (not fullness) empties the stage.
bool g_defer_small_sequences = [] {
    const char *e = getenv("SMB200_DEFER_SEQ");
    return !(e && e[0] == '0');
}();
namespace {
const size_t kDeferMaxLen = size_t(1) << 16, kDeferFlushBytes = size_t(8) << 20;
const size_t kStageFull = kDeferFlushBytes + kDeferMaxLen;  // a stage never holds more than this
const size_t kStagePinAt = size_t(256) << 10;
const size_t kDeferTotalCap = size_t(1) << 30;  // see g_seq_pending_total
const size_t kAccountGranule = size_t(64) << 10;
const int kPinnedBuffersMax = 16;  // 16 x 8 MiB page-locked at most, whatever the number of sketches

std::mutex g_pin_mutex;
std::vector<uint8_t *> g_pin_free;
int g_pin_live = 0;
uint8_t *pinned_acquire() {
    {
        std::lock_guard<std::mutex> lk(g_pin_mutex);
        if (!g_pin_free.empty()) {
            uint8_t *p = g_pin_free.back();
            g_pin_free.pop_back();
            return p;
        }
        if (g_pin_live >= kPinnedBuffersMax) return nullptr;
        g_pin_live++;
    }
    void *p = nullptr;
    if (cudaMallocHost(&p, kStageFull) != cudaSuccess) {
        (void)cudaGetLastError();
        std::lock_guard<std::mutex> lk(g_pin_mutex);
        g_pin_live--;
        return nullptr;
    }
    return static_cast<uint8_t *>(p);
}
void pinned_release(uint8_t *p) {
    std::lock_guard<std::mutex> lk(g_pin_mutex);
    g_pin_free.push_back(p);
}

// every byte one of ACGTacgt?  (16 bytes per step: fold the case bit away, compare with the four letters)
bool all_acgt(const uint8_t *s, size_t n) {
    size_t i = 0;
#if defined(__SSE2__)
    const __m128i up = _mm_set1_epi8((char)0xDF), a = _mm_set1_epi8('A'), c = _mm_set1_epi8('C'), g = _mm_set1_epi8('G'),
                  t = _mm_set1_epi8('T');
    __m128i ok = _mm_set1_epi8((char)0xFF);
    for (; i + 16 <= n; i += 16) {
        const __m128i x = _mm_and_si128(_mm_loadu_si128(reinterpret_cast<const __m128i *>(s + i)), up);
        ok = _mm_and_si128(ok, _mm_or_si128(_mm_or_si128(_mm_cmpeq_epi8(x, a), _mm_cmpeq_epi8(x, c)),
                                            _mm_or_si128(_mm_cmpeq_epi8(x, g), _mm_cmpeq_epi8(x, t))));
    }
    if (_mm_movemask_epi8(ok) != 0xFFFF) return false;
#endif
    uint8_t all = 1;
    for (; i < n; i++) {
        const uint8_t x = s[i] & 0xDF;
        all &= (uint8_t)((x == 'A') | (x == 'C') | (x == 'G') | (x == 'T'));
    }
    return all != 0;
}
}  // namespace

SeqStage::~SeqStage() { drop(); }
void SeqStage::drop() {
    if (p) {
        if (pinned) pinned_release(p); else free(p);
    }
    if (accounted) g_seq_pending_total -= accounted;
    p = nullptr;
    n = cap = accounted = 0;
    pinned = false;
    offsets.assign(1, 0);
}
// room for `len` more bytes (len <= kDeferMaxLen, n < kDeferFlushBytes on entry)
void SeqStage::grow(size_t len) {
    const size_t need = n + len;
    if (need >= kStagePinAt && !pinned) {
        if (uint8_t *q = pinned_acquire()) {
            if (n) memcpy(q, p, n);
            free(p);
            p = q;
            cap = kStageFull;
            pinned = true;
            return;
        }
    }
    size_t want = cap ? cap * 2 : 4096;
    while (want < need) want *= 2;
    want = std::min(want, kStageFull);
    uint8_t *q = static_cast<uint8_t *>(realloc(p, want));
    if (!q) throw std::bad_alloc();
    p = q;
    cap = want;
}

void KmerMinHash::flush_sequences(bool stage_full) {
    SeqStage &sg = seq_stage_;
    if (sg.offsets.size() <= 1) return;
    // taken out first: add_sequences comes back here through flush_pending()
    std::vector<uint64_t> offs(1, 0);
    offs.swap(sg.offsets);
    const size_t n_bytes = sg.n;
    sg.n = 0;
    SeqBatch b;
    b.buf = sg.p;
    b.offsets = offs.data();
    b.n_seqs = offs.size() - 1;
    b.n_bytes = n_bytes;
    KmerMinHash *self = this;
    try {
        add_sequences(&self, 1, b, true);
    } catch (...) {
        sg.drop();
        throw;
    }
    if (sg.accounted) {
        g_seq_pending_total -= sg.accounted;
        sg.accounted = 0;
    }
    offs.assign(1, 0);      // keep the (already touched) storage for the next batch
    sg.offsets.swap(offs);
    if (!stage_full && sg.pinned) sg.drop();  // the caller went on to something else: page-locked memory goes back
}

void KmerMinHash::add_sequence(const uint8_t *seq, size_t len, bool force) {
    if (g_defer_small_sequences && !is_protein && ksize != 0 && len <= kDeferMaxLen && (force || all_acgt(seq, len))) {
        if (!Context::peek()) Context::get();  // no device: fail on this call, as the synchronous path would
        if (len < ksize) return;  // lib.rs:258: shorter than k adds nothing
        if (!pending_.empty()) flush_pending();  // add_hash events came first
        SeqStage &sg = seq_stage_;
        if (sg.n + len > sg.cap) sg.grow(len);
        memcpy(sg.p + sg.n, seq, len);
        sg.n += len;
        sg.offsets.push_back(sg.n);
        bool over_cap = false;
        if (sg.n > sg.accounted) {  // the process-wide total is kept in granules: one atomic per 64 KiB, not per call
            const size_t add = (sg.n - sg.accounted + kAccountGranule - 1) / kAccountGranule * kAccountGranule;
            sg.accounted += add;
            over_cap = (g_seq_pending_total += add) > kDeferTotalCap;
        }
        if (sg.n >= kDeferFlushBytes || over_cap) flush_sequences(true);
        return;
    }
    SeqBatch b;
    b.buf = seq;
    b.n_seqs = 1;
    b.n_bytes = len;
    KmerMinHash *self = this;
    add_sequences(&self, 1, b, force);
}

namespace {
struct PerSketch {
    uint64_t prev_cand = 0;
    uint64_t thr_fallback = U64_MAX;
    bool estimate = false;
    uint32_t tile_lo = 0;
    uint32_t tiles_total = 0;
    uint64_t first_bad = U64_MAX;
};
}  // namespace

void KmerMinHash::add_sequences(KmerMinHash *const *mhs, int n_mhs, const SeqBatch &batch, bool force) {
    if (n_mhs <= 0) return;
    if (n_mhs > 6) throw_internal("at most 6 sketches per batch call");
    // one sketch twice would share its candidate list, device scalars and tile counter between two passes
    for (int i = 0; i < n_mhs; i++)
        for (int j = 0; j < i; j++)
            if (mhs[i] == mhs[j]) throw_internal("a sketch appears more than once in one batch call");
    for (int i = 0; i < n_mhs; i++) {
        if (mhs[i]->ksize == 0) throw_internal("ksize 0");
        if (mhs[i]->is_protein && mhs[i]->ksize < 3)  // the reference reaches slice::windows(0), which panics
            throw SourmashError(ERR_PANIC, "sourmash panicked: size is zero");
    }
    for (int i = 0; i < n_mhs; i++) mhs[i]->flush_sequences();  // deferred add_sequence calls came first
    const uint64_t n = batch.n_bytes;
    if (n == 0) return;
    if (batch.offsets == nullptr && batch.read_len != 0 && n != batch.n_seqs * (uint64_t)batch.read_len)
        throw_internal("fixed-length batch: n_bytes != n_seqs * read_len");
    Context &ctx = Context::get();
    for (int i = 0; i < n_mhs; i++) ctx.adopt(mhs[i]->owner_);
    cudaStream_t st = ctx.stream;

    // ---- per-sketch preparation: order-dependent work first, thresholds, candidate space -------
    std::vector<PerSketch> ps(n_mhs);
    for (int i = 0; i < n_mhs; i++) {
        KmerMinHash &mh = *mhs[i];
        // hashes this call can produce at most: one per base (DNA) / per codon slot of the six frames
        const uint64_t windows_upper = mh.is_protein ? protein_slots(n, batch.n_seqs) : n;
        mh.flush_pending();
        if (mh.mode() != MODE_SCALED && mh.n_cand_) mh.ingest(ctx, false);
        mh.ensure_dev();
        mh.require_sorted("add_sequence");
        PerSketch &p = ps[i];
        p.prev_cand = mh.n_cand_;
        p.tiles_total = sketch_tile_count(n, n);
        double frac = 1.0;  // expected fraction of windows that survive the threshold
        if (mh.mode() == MODE_SCALED) {
            p.thr_fallback = mh.max_hash;
            frac = (double)mh.max_hash / 18446744073709551616.0;
        } else if (mh.mode() == MODE_NUM) {
            const double want = 8.0 * mh.num + 4096.0;
            if ((double)windows_upper > 4.0 * want) {
                frac = want / (double)windows_upper;
                p.thr_fallback = (uint64_t)(frac * 18446744073709551616.0);
                p.estimate = mh.n_mins_ < mh.num;  // a full sketch uses its own largest element instead
            }
        } else if (mh.max_hash) {
            p.thr_fallback = mh.max_hash;
            frac = (double)mh.max_hash / 18446744073709551616.0;
        }
        mh.reserve_candidates(ctx, mh.n_cand_ + (uint64_t)(frac * 1.25 * (double)windows_upper) + 4096);
        set_u64(mh.hs(0), mh.n_cand_, st);
        set_u64(mh.hs(2), U64_MAX, st);
        thr_from_state_kernel<<<1, 1, 0, st>>>(mh.hs(1), mh.d_mins_.as<uint64_t>(), mh.n_mins_,
                                               mh.mode() == MODE_NUM ? mh.num : 0, p.thr_fallback);
        SM_LAUNCHED();
    }

    // ---- bring the batch to the device (chunked, overlapped with the kernels) ------------------
    const uint8_t *d_buf = nullptr;
    const uint64_t *d_off = nullptr;
    const uint32_t bpr = (batch.read_len + 3) / 4;   // packed bytes per read
    if (batch.packed2 && (batch.offsets || batch.read_len == 0)) throw_internal("2-bit input needs fixed-length reads");
    if (batch.on_device && batch.packed2) {
        // packed reads already in HBM: expand them in one go, then as a device-resident ASCII batch
        ctx.ascii.reserve(((n + 15) & ~15ull) + 256);
        unpack_2bit_kernel<<<(unsigned)std::min<uint64_t>((n / 16 + 256) / 256, 148 * 16), 256, 0, st>>>(batch.packed2, ctx.ascii.as<uint8_t>(),
                                                                                                     0, batch.n_seqs, batch.read_len);
        SM_LAUNCHED();
        d_buf = ctx.ascii.as<uint8_t>();
    } else if (batch.on_device) {
        if ((reinterpret_cast<uintptr_t>(batch.buf) & 15) != 0) throw_internal("device sequence buffer must be 16-byte aligned");
        d_buf = batch.buf;
        d_off = batch.offsets;
    } else {
        if (batch.packed2) ctx.packed.reserve((size_t)batch.n_seqs * bpr + 256);
        ctx.ascii.reserve(((n + 15) & ~15ull) + 256);
        d_buf = ctx.ascii.as<uint8_t>();
        if (batch.offsets) {
            ctx.offsets.reserve((batch.n_seqs + 1) * 8);
            SM_CUDA(cudaMemcpyAsync(ctx.offsets.p, batch.offsets, (batch.n_seqs + 1) * 8, cudaMemcpyHostToDevice, st));
            d_off = ctx.offsets.as<uint64_t>();
        }
    }
    auto make_batch = [&](KmerMinHash &mh, uint64_t n_limit, uint32_t tile_lo) {
        SketchBatch sb;
        sb.buf = d_buf; sb.n = n; sb.n_limit = n_limit; sb.offsets = d_off; sb.n_seqs = batch.n_seqs;
        sb.read_len = batch.offsets ? 0 : batch.read_len; sb.tile_lo = tile_lo; sb.seed = mh.seed; sb.pos_base = 0;
        sb.first_bad = force ? nullptr : mh.hs(2);
        sb.tile_ctr = reinterpret_cast<uint32_t *>(mh.hs(3));  // this sketch's launches are stream-ordered
        return sb;
    };
    // protein sketches: translate / compact / hash over the whole device-resident batch (protein.cu)
    auto launch_protein = [&](KmerMinHash &mh) {
        const uint64_t total = protein_slots(n, batch.n_seqs);
        ctx.misc[0].reserve(total + 64);
        ctx.misc[1].reserve(total + 64);
        ctx.misc[2].reserve((total + 2) * 8);
        ctx.misc[3].reserve((total + 2) * 8);
        ctx.scan_tmp.reserve(scan_tmp_bytes(total + 1) + 256);
        ProteinBatch pb;
        pb.buf = d_buf; pb.n = n; pb.offsets = d_off; pb.n_seqs = batch.n_seqs;
        pb.read_len = batch.offsets ? 0 : batch.read_len; pb.ksize = mh.ksize; pb.seed = mh.seed;
        SketchOut o;
        o.thr = reinterpret_cast<const uint64_t *>(mh.hs(1));
        o.hash = mh.d_cand_hash_.as<uint64_t>();
        o.pos = mh.want_pos() ? mh.d_cand_pos_.as<uint64_t>() : nullptr;
        o.cap = mh.d_cand_hash_.cap / 8;
        o.counter = mh.hs(0);
        launch_protein_sketch(pb, o, ctx.misc[0].as<uint8_t>(), ctx.misc[1].as<uint8_t>(), ctx.misc[2].as<uint64_t>(),
                              ctx.misc[3].as<uint64_t>(), ctx.scan_tmp.p, st);
    };
    auto make_out = [&](KmerMinHash &mh) {
        SketchOut o;
        o.thr = reinterpret_cast<const uint64_t *>(mh.hs(1));
        o.hash = mh.d_cand_hash_.as<uint64_t>();
        o.pos = mh.want_pos() ? mh.d_cand_pos_.as<uint64_t>() : nullptr;
        o.cap = mh.d_cand_hash_.cap / 8;
        o.counter = mh.hs(0);
        return o;
    };
    // Copy chunks of a fixed 8 MiB (tapering off at the end of the batch).  The fused multi-k kernel
    // consumes bases at about the rate PCIe delivers them, so a chunk size that GROWS makes the kernels
    // of chunk c finish long before the (larger) chunk c+1 has landed -- the old 4 -> 32 MiB doubling
    // idled the GPU for ~0.5 ms per 300 MB batch.  With equal chunks only the first copy is exposed.
    uint64_t chunk = g_h2d_chunk_bytes;
    const uint64_t CHUNK_MAX = g_h2d_chunk_bytes;
    uint64_t copied = batch.on_device ? n : 0;
    if (!batch.on_device) SM_CUDA(cudaStreamSynchronize(st));  // scalars / offsets in place before the copy stream races ahead
    // every sketch's kernels go to its own stream, ordered after the preparation above and after
    // the chunk they read: the three k-sizes of a multi-k batch then overlap at their edges
    // (with per-kernel timing switched on they stay on one stream, so that each duration is the
    // kernel's own)
    const bool fan_out = !prof_enabled() && n_mhs > 1;
    auto kstream = [&](int i) { return fan_out ? ctx.k_streams[i] : st; };
    if (fan_out) {
        SM_CUDA(cudaEventRecord(ctx.prep_event, st));
        for (int i = 0; i < n_mhs; i++) SM_CUDA(cudaStreamWaitEvent(ctx.k_streams[i], ctx.prep_event, 0));
    }
    // DNA sketches with distinct fast-path k-sizes and one seed share a fused launch per chunk: the
    // tile is staged once and every k-size walks it (sketch.cu).  Member order = ascending k.
    std::vector<int> fused;
    if (g_fuse_multi_k) {
        for (int i = 0; i < n_mhs; i++) {
            const KmerMinHash &mh = *mhs[i];
            if (mh.is_protein || !sketch_has_fast_path(mh.ksize)) continue;
            bool ok = fused.empty() || mhs[fused[0]]->seed == mh.seed;
            for (int j : fused) ok = ok && mhs[j]->ksize != mh.ksize;
            if (ok && fused.size() < 3) fused.push_back(i);
        }
        std::sort(fused.begin(), fused.end(), [&](int a, int b) { return mhs[a]->ksize < mhs[b]->ksize; });
        if (fused.size() < 2) fused.clear();
    }
    auto in_fused = [&](int i) { return std::find(fused.begin(), fused.end(), i) != fused.end(); };
    size_t ev_i = 0;
    unsigned fused_turn = 0;
    do {
        if (!batch.on_device) {
            // ... and taper off again (half of what is left, not below 2 MiB): what remains after the
            // last copy has landed is the kernel of the last chunk only
            const uint64_t left = n - copied;
            uint64_t len = std::min<uint64_t>(chunk, left);
            if (left > (2ull << 20)) len = std::min<uint64_t>(len, std::max<uint64_t>((left / 2 + 4095) & ~4095ull, 2ull << 20));
            chunk = std::min<uint64_t>(chunk * 2, CHUNK_MAX);
            if (batch.packed2) {
                // whole reads per chunk: a quarter of the bytes cross PCIe, the copy stream expands them behind the copy
                const uint64_t r0 = copied / batch.read_len;
                const uint64_t r1 = std::min<uint64_t>(batch.n_seqs, std::max<uint64_t>(r0 + 1, (copied + len) / batch.read_len));
                SM_CUDA(cudaMemcpyAsync(ctx.packed.as<uint8_t>() + r0 * bpr, batch.packed2 + r0 * bpr, (r1 - r0) * bpr, cudaMemcpyHostToDevice,
                                        ctx.copy_stream));
                const uint64_t out_bytes = (r1 - r0) * batch.read_len;
                unpack_2bit_kernel<<<(unsigned)std::min<uint64_t>((out_bytes / 16 + 256) / 256, 148 * 8), 256, 0, ctx.copy_stream>>>(
                    ctx.packed.as<uint8_t>(), const_cast<uint8_t *>(d_buf), r0, r1, batch.read_len);
                SM_LAUNCHED();
                len = r1 * batch.read_len - copied;
            } else {
                SM_CUDA(cudaMemcpyAsync(const_cast<uint8_t *>(d_buf) + copied, batch.buf + copied, len, cudaMemcpyHostToDevice,
                                        ctx.copy_stream));
            }
            copied += len;
            if (ev_i >= ctx.chunk_events.size()) {
                cudaEvent_t e;
                SM_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                ctx.chunk_events.push_back(e);
            }
            SM_CUDA(cudaEventRecord(ctx.chunk_events[ev_i], ctx.copy_stream));
            if (fan_out) {
                for (int i = 0; i < n_mhs; i++) SM_CUDA(cudaStreamWaitEvent(ctx.k_streams[i], ctx.chunk_events[ev_i], 0));
            } else {
                SM_CUDA(cudaStreamWaitEvent(st, ctx.chunk_events[ev_i], 0));
            }
            ev_i++;
        }
        if (!fused.empty()) {
            const int lead = fused[0];
            PerSketch &p = ps[lead];
            const uint32_t kmax = mhs[fused.back()]->ksize;  // the widest halo decides which tiles are complete
            const uint32_t hi = (copied >= n) ? p.tiles_total : std::min(p.tiles_total, sketch_tiles_ready(kmax, copied));
            if (hi > p.tile_lo) {
                uint32_t ks[3];
                SketchOuts outs;
                for (size_t j = 0; j < 3; j++) {
                    KmerMinHash &m = *mhs[fused[std::min(j, fused.size() - 1)]];
                    outs.o[j] = make_out(m);
                    outs.first_bad[j] = force ? nullptr : m.hs(2);
                    if (j < fused.size()) ks[j] = m.ksize;
                }
                // consecutive chunks go to two streams in turn (each with its own tile counter: the group's
                // first two members lend theirs), so that the tail of one launch -- CTAs finishing their
                // last tile -- is filled by the next launch instead of idling the SMs
                const int turn = fused[fused_turn & 1];
                fused_turn++;
                SketchBatch sbm = make_batch(*mhs[lead], n, p.tile_lo);
                sbm.tile_ctr = reinterpret_cast<uint32_t *>(mhs[turn]->hs(3));
                launch_sketch_multi(ks, (int)fused.size(), sbm, outs, hi, ctx.sm_count, kstream(turn));
                for (int j : fused) ps[j].tile_lo = hi;
            }
        }
        for (int i = 0; i < n_mhs; i++) {
            KmerMinHash &mh = *mhs[i];
            PerSketch &p = ps[i];
            if (mh.is_protein || in_fused(i)) continue;  // protein: after the whole batch has arrived
            uint32_t hi = (copied >= n) ? p.tiles_total : std::min(p.tiles_total, sketch_tiles_ready(mh.ksize, copied));
            if (hi <= p.tile_lo) continue;
            launch_sketch(mh.ksize, make_batch(mh, n, p.tile_lo), make_out(mh), hi, ctx.sm_count, kstream(i));
            p.tile_lo = hi;
        }
    } while (copied < n);
    for (int i = 0; fan_out && i < n_mhs; i++) {  // back onto the library's stream
        SM_CUDA(cudaEventRecord(ctx.k_events[i], ctx.k_streams[i]));
        SM_CUDA(cudaStreamWaitEvent(st, ctx.k_events[i], 0));
    }
    for (int i = 0; i < n_mhs; i++)
        if (mhs[i]->is_protein) launch_protein(*mhs[i]);

    // ---- results: overflow / first failing k-mer / estimate too tight -> re-run from the device copy
    std::string error_kmer;
    int error_sketch = -1;
    for (int i = 0; i < n_mhs; i++) {
        KmerMinHash &mh = *mhs[i];
        PerSketch &p = ps[i];
        uint64_t n_limit = n;
        for (int attempt = 0;; attempt++) {
            SM_CUDA(cudaMemcpyAsync(ctx.h_scalars + SC_CAND0, mh.hs(0), 24, cudaMemcpyDeviceToHost, st));
            ctx.sync();
            const uint64_t count = ctx.h_scalars[SC_CAND0];
            const uint64_t fb = ctx.h_scalars[SC_CAND0 + 2];
            bool rerun = false;
            if (!force && fb != U64_MAX && n_limit == n) {  // stop where the reference stops (lib.rs:268-273)
                p.first_bad = fb;
                n_limit = fb;
                rerun = true;
            }
            if (count > mh.d_cand_hash_.cap / 8) {
                mh.n_cand_ = p.prev_cand;
                mh.reserve_candidates(ctx, count + 4096);
                rerun = true;
            }
            if (!rerun) {
                mh.n_cand_ = count;
                mh.host_valid_ = mh.host_valid_ && count == p.prev_cand;
                if (mh.mode() == MODE_SCALED) {
                    if (mh.n_cand_ > LAZY_CANDIDATES) mh.ingest(ctx, false);
                    break;
                }
                if (mh.mode() == MODE_REPLAY) {
                    // events in stream order: sort (pos, hash) by pos, replay
                    const uint64_t ne = mh.n_cand_;
                    mh.n_cand_ = 0;
                    if (ne) {
                        ctx.sort_tmp_k.reserve((ne + 1) * 8);
                        ctx.sort_tmp_v.reserve((ne + 1) * 8);
                        ctx.scan_tmp.reserve(radix_sort_scan_bytes(ne) + 256);
                        radix_sort_pairs(mh.d_cand_pos_.as<uint64_t>(), mh.d_cand_hash_.as<uint64_t>(), ne,
                                         ctx.sort_tmp_k.as<uint64_t>(), ctx.sort_tmp_v.as<uint64_t>(),
                                         bit_length(mh.is_protein ? protein_slots(n, batch.n_seqs) : n),  // positions: residue slots
                                         ctx.scan_tmp.p, ctx.scan_tmp.cap, st);
                        mh.replay(ctx, mh.d_cand_hash_.as<uint64_t>(), ne);
                    }
                    break;
                }
                // MODE_NUM
                if (mh.ingest(ctx, p.estimate, p.thr_fallback)) break;
                // estimate kept too few distinct hashes: widen and go again
                p.thr_fallback = (p.thr_fallback > (U64_MAX >> 6)) ? U64_MAX : (p.thr_fallback << 6);
                if (p.thr_fallback == U64_MAX) p.estimate = false;
                mh.reserve_candidates(ctx, (uint64_t)((double)p.thr_fallback / 18446744073709551616.0 * 1.25 *
                                                      (double)(mh.is_protein ? protein_slots(n, batch.n_seqs) : n)) + 4096);
            }
            if (attempt > 40) throw_internal("sketch re-run loop did not converge");
            // re-run over the device-resident batch
            set_u64(mh.hs(0), p.prev_cand, st);
            set_u64(mh.hs(2), U64_MAX, st);
            thr_from_state_kernel<<<1, 1, 0, st>>>(mh.hs(1), mh.d_mins_.as<uint64_t>(), mh.n_mins_,
                                                   mh.mode() == MODE_NUM ? mh.num : 0, p.thr_fallback);
            SM_LAUNCHED();
            if (mh.is_protein) {
                launch_protein(mh);
            } else {
                SketchBatch sb = make_batch(mh, n_limit, 0);
                sb.first_bad = nullptr;
                launch_sketch(mh.ksize, sb, make_out(mh), sketch_tile_count(n, n_limit), ctx.sm_count, st);
            }
        }
        if (p.first_bad != U64_MAX && error_sketch < 0) {
            error_sketch = i;
            std::vector<uint8_t> kmer(mh.ksize);
            SM_CUDA(cudaMemcpyAsync(kmer.data(), d_buf + p.first_bad, mh.ksize, cudaMemcpyDeviceToHost, st));
            ctx.sync();
            for (auto &c : kmer) if (c >= 'a' && c <= 'z') c = (uint8_t)(c - 32);  // lib.rs:253-256
            error_kmer.assign(kmer.begin(), kmer.end());
        }
    }
    if (error_sketch >= 0)
        throw SourmashError(ERR_INVALID_DNA, "invalid DNA character in input k-mer: " + error_kmer);
}

// ---------------------------------------------------------------------------------------------
// merge / compare
// ---------------------------------------------------------------------------------------------
// merge when an abundance vector is NOT as long as its mins.  That state is the reference's own doing: merge
// truncates mins to num and leaves the abundances as they are (lib.rs:395-400 "TODO: reduce this one too"), and
// the next merge then walks two iterators of different length (lib.rs:316-389).  What comes out depends on the
// order of the walk -- an abundance is taken when, and only when, the walk asks that side's iterator for one -- so
// this (rare) case is replayed by ONE device thread, step by step as the reference takes them:
//   other-only element: other's next abundance, if it has one left;
//   common element: other's next, and if there was one, self's next, and if there was one too, their sum;
//   self-only element: self's next, if there is one;
//   other runs out first: everything self's abundance iterator still holds; leftover of other: all it still holds.
__global__ void merge_out_of_step_kernel(const uint64_t *a, uint64_t na, const uint64_t *sa, uint64_t nsa, bool has_sa,
                                         const uint64_t *b, uint64_t nb, const uint64_t *sb, uint64_t nsb, bool has_sb,
                                         uint64_t *out, uint64_t *out_ab, unsigned long long *n_out, unsigned long long *n_out_ab) {
    uint64_t i = 0, j = 0, ia = 0, ib = 0, m = 0, ma = 0;
    bool broke = false;
    while (i < na) {
        if (j >= nb) {  // other exhausted: the rest of self, and ALL that is left of self's abundances
            while (i < na) out[m++] = a[i++];
            if (has_sa) while (ia < nsa) out_ab[ma++] = sa[ia++];
            broke = true;
            break;
        }
        const uint64_t x = b[j], v = a[i];
        if (x < v) {
            out[m++] = x; j++;
            if (has_sb && ib < nsb) out_ab[ma++] = sb[ib++];
        } else if (x == v) {
            out[m++] = x; j++; i++;
            if (has_sb && ib < nsb) {
                const uint64_t vb = sb[ib++];
                if (has_sa && ia < nsa) out_ab[ma++] = vb + sa[ia++];
            }
        } else {
            out[m++] = v; i++;
            if (has_sa && ia < nsa) out_ab[ma++] = sa[ia++];
        }
    }
    (void)broke;
    while (j < nb) out[m++] = b[j++];
    if (has_sb) while (ib < nsb) out_ab[ma++] = sb[ib++];
    *n_out = m;
    *n_out_ab = ma;
}

void KmerMinHash::merge(KmerMinHash &other) {
    check_compatible(other);
    flush(); other.flush();
    ensure_dev(); other.ensure_dev();
    require_sorted("merge"); other.require_sorted("merge");
    Context &ctx = home();
    cudaStream_t st = ctx.stream;
    const uint64_t na = n_mins_, nb = other.n_mins_;
    const bool sa = has_abunds_, ob = other.has_abunds_;
    if ((sa && n_abunds_ != na) || (ob && other.n_abunds_ != nb)) {
        const uint64_t nsa = sa ? n_abunds_ : 0, nsb = ob ? other.n_abunds_ : 0;
        d_mins_alt_.reserve((na + nb + 1) * 8);
        d_abunds_alt_.reserve((nsa + nsb + 1) * 8);
        merge_out_of_step_kernel<<<1, 1, 0, st>>>(d_mins_.as<uint64_t>(), na, d_abunds_.as<uint64_t>(), nsa, sa, other.d_mins_.as<uint64_t>(), nb,
                                                  other.d_abunds_.as<uint64_t>(), nsb, ob, d_mins_alt_.as<uint64_t>(),
                                                  d_abunds_alt_.as<uint64_t>(), ctx.dsc(SC_NUNIQ), ctx.dsc(SC_CNT));
        SM_LAUNCHED();
        ctx.read_scalars();
        const uint64_t n_union = ctx.h_scalars[SC_NUNIQ], n_ab = ctx.h_scalars[SC_CNT];
        has_abunds_ = true;  // lib.rs:393,400
        commit(d_mins_alt_, d_abunds_alt_, (num != 0 && n_union >= num) ? num : n_union, n_ab);
        return;
    }
    const bool both = sa && ob;
    const uint64_t n_cat = na + nb;
    ctx.sort_tmp_k.reserve((n_cat + 1) * 8);
    ctx.sort_tmp_v.reserve((n_cat + 1) * 8);
    ctx.scan_tmp.reserve(std::max(radix_sort_scan_bytes(n_cat), scan_tmp_bytes(n_cat)) + 256);
    for (int i = 0; i < 4; i++) ctx.misc[i].reserve((n_cat + 1) * 8);
    uint64_t *cat_k = ctx.misc[0].as<uint64_t>(), *cat_v = ctx.misc[1].as<uint64_t>(), *idx = ctx.misc[2].as<uint64_t>();
    if (na) SM_CUDA(cudaMemcpyAsync(cat_k, d_mins_.p, na * 8, cudaMemcpyDeviceToDevice, st));
    if (nb) SM_CUDA(cudaMemcpyAsync(cat_k + na, other.d_mins_.p, nb * 8, cudaMemcpyDeviceToDevice, st));
    if (both) {
        if (na) SM_CUDA(cudaMemcpyAsync(cat_v, d_abunds_.p, na * 8, cudaMemcpyDeviceToDevice, st));
        if (nb) SM_CUDA(cudaMemcpyAsync(cat_v + na, other.d_abunds_.p, nb * 8, cudaMemcpyDeviceToDevice, st));
    }
    radix_sort_pairs(cat_k, both ? cat_v : nullptr, n_cat, ctx.sort_tmp_k.as<uint64_t>(), ctx.sort_tmp_v.as<uint64_t>(),
                     64, ctx.scan_tmp.p, ctx.scan_tmp.cap, st);
    DevBuf &out_k = d_mins_alt_, &out_v = d_abunds_alt_;
    out_k.reserve((n_cat + 1) * 8);
    out_v.reserve((n_cat + 1) * 8);
    // the reference sums abundances where both sides track them (lib.rs:354-367)
    uint64_t *sums = both ? out_v.as<uint64_t>() : ctx.misc[3].as<uint64_t>();
    reduce_by_key(cat_k, both ? cat_v : nullptr, n_cat, out_k.as<uint64_t>(), sums, ctx.dsc(SC_NUNIQ), idx, ctx.scan_tmp.p, st);
    ctx.read_scalars();
    const uint64_t n_union = ctx.h_scalars[SC_NUNIQ];
    const uint64_t common = n_cat - n_union;
    uint64_t n_ab = 0;
    if (both) {
        n_ab = n_union;  // NOT truncated with mins (lib.rs:395-400 TODO)
    } else if (sa) {
        // only self tracks.  The reference advances self's abundance iterator when it emits a
        // self-only element and NOT on a common one (lib.rs:354-367: the inner `if let` chain
        // starts from other's iterator, which is None), so the values it emits are simply the
        // leading entries of self.abunds: one per self-only element, plus -- when other runs out
        // first and the `None` arm fires (lib.rs:336-343) -- everything that is left.
        uint64_t last_a = 0, last_b = 0;
        if (na) SM_CUDA(cudaMemcpyAsync(&last_a, d_mins_.as<uint64_t>() + (na - 1), 8, cudaMemcpyDeviceToHost, st));
        if (nb) SM_CUDA(cudaMemcpyAsync(&last_b, other.d_mins_.as<uint64_t>() + (nb - 1), 8, cudaMemcpyDeviceToHost, st));
        ctx.sync();
        const bool none_arm = na > 0 && (nb == 0 || last_a > last_b);
        n_ab = none_arm ? na : na - common;
        if (n_ab) SM_CUDA(cudaMemcpyAsync(out_v.p, d_abunds_.p, n_ab * 8, cudaMemcpyDeviceToDevice, st));
        ctx.sync();
    } else if (ob) {
        // only other tracks: its iterator stays in step (advanced on common elements too), so the
        // reference emits the abundances of the elements only other holds (lib.rs:344-352,384-388)
        uint64_t *flags = ctx.misc[0].as<uint64_t>(), *pre = ctx.misc[1].as<uint64_t>();
        launch_mark_common(other.d_mins_.as<uint64_t>(), nb, d_mins_.as<uint64_t>(), na, flags, st);
        scan_exclusive_u64(flags, pre, nb, ctx.scan_tmp.p, st);
        launch_compact_unflagged(other.d_abunds_.as<uint64_t>(), flags, pre, nb, out_v.as<uint64_t>(), st);
        ctx.sync();
        n_ab = nb - common;
    }
    const uint64_t n_keep = (num != 0 && n_union >= num) ? num : n_union;
    has_abunds_ = true;  // lib.rs:393,400: abunds becomes Some(..) unconditionally
    commit(out_k, out_v, n_keep, n_ab);
}

static void pair_stats(KmerMinHash &a, KmerMinHash &b, uint32_t num, uint64_t out[3]) {
    size_t na, nb;
    const uint64_t *da = a.device_mins(&na);
    const uint64_t *db = b.device_mins(&nb);
    Context &ctx = Context::get();  // both sketches were re-homed to this thread by device_mins()
    launch_pair_stats(da, na, db, nb, num, ctx.dsc(SC_PAIR0), ctx.stream);
    ctx.read_scalars();
    out[0] = ctx.h_scalars[SC_PAIR0];
    out[1] = ctx.h_scalars[SC_PAIR1];
    out[2] = ctx.h_scalars[SC_PAIR2];
}

uint64_t KmerMinHash::count_common(KmerMinHash &other) {
    check_compatible(other);
    flush(); other.flush();
    require_sorted("count_common"); other.require_sorted("count_common");
    uint64_t o[3];
    pair_stats(*this, other, 0, o);
    return o[0];
}

std::pair<uint64_t, uint64_t> KmerMinHash::intersection_size(KmerMinHash &other) {
    check_compatible(other);
    flush(); other.flush();
    require_sorted("intersection"); other.require_sorted("intersection");
    uint64_t o[3];
    pair_stats(*this, other, num, o);  // uses self.num (lib.rs:473-480)
    return {o[1], o[2]};
}

// lib.rs:438-468: the hashes of A n B that are also in combined = bottom_num(A u B), and |combined|.  A common
// element's rank in the union grows with its position, so those are simply the FIRST `common` elements of A n B,
// with `common` and |combined| as intersection_size gives them.
std::pair<std::vector<uint64_t>, uint64_t> KmerMinHash::intersection(KmerMinHash &other) {
    const std::pair<uint64_t, uint64_t> cs = intersection_size(other);
    std::vector<uint64_t> out(cs.first);
    if (cs.first) {
        size_t na, nb;
        const uint64_t *da = device_mins(&na);
        const uint64_t *db = other.device_mins(&nb);
        Context &ctx = Context::get();
        cudaStream_t st = ctx.stream;
        ctx.misc[0].reserve((na + 1) * 8);
        ctx.misc[1].reserve((na + 1) * 8);
        ctx.misc[2].reserve((cs.first + 1) * 8);
        ctx.scan_tmp.reserve(scan_tmp_bytes(na) + 256);
        uint64_t *flags = ctx.misc[0].as<uint64_t>(), *pre = ctx.misc[1].as<uint64_t>(), *kept = ctx.misc[2].as<uint64_t>();
        launch_mark_common(da, na, db, nb, flags, st);
        scan_exclusive_u64(flags, pre, na, ctx.scan_tmp.p, st);
        launch_compact_flagged(da, flags, pre, na, cs.first, kept, st);
        SM_CUDA(cudaMemcpyAsync(out.data(), kept, cs.first * 8, cudaMemcpyDeviceToHost, st));
        ctx.sync();
    }
    return {std::move(out), cs.second};
}

double KmerMinHash::compare(KmerMinHash &other) {
    const std::pair<uint64_t, uint64_t> cs = intersection_size(other);
    return (double)cs.first / (double)std::max<uint64_t>(1, cs.second);  // lib.rs:504
}

double KmerMinHash::containment(KmerMinHash &other) {
    const uint64_t common = count_common(other);
    return (double)common / (double)size();  // index.rs:152-154 (0/0 -> NaN)
}

}  // namespace smb200
